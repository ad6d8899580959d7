"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Golden scores AT THE BENCHMARKED CONFIGURATION (BASELINE config 5 shapes): 17 videos x 2 000 steps x 1 024-d features that
were rounded to bfloat16 (what the sweep stores), through the UNMODIFIED reference VASNet and DSN modules in float32 on
the CPU.  17 videos = 34 000 rows: more than one 32 768-row chunk of the packed scorer, so the GPU test runs the
chunked, two-stream path with the fused exp / head epilogues — exactly what bench.py times.  The features are
regenerated from seeds by the tests; only the outputs are stored.

    python -m oracle.gen_golden_sweep          (needs SMZ_REFERENCE_ROOT, see oracle/ref_import.py)
"""
import os

import numpy as np
import torch

from oracle.gen_golden_models import build_dsn, build_vasnet, checksums

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "sweep_golden.npz")
N_VIDEOS, T, VAS_SEED, DSN_SEED, SHARPEN = 17, 2000, 31, 32, 6.0


def sweep_features(video):
    """(T, 1024) bfloat16: non-negative L2-normalised rows (pool5-like), rounded to the sweep's storage type."""
    g = torch.Generator().manual_seed(70_000 + video)
    x = torch.randn(T, 1024, generator=g).abs()
    return (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)


def main():
    from oracle import ref_import
    ns = ref_import.load()
    torch.set_num_threads(os.cpu_count() or 1)
    vas = build_vasnet(ns.vasnet.VASNet, VAS_SEED, {}, SHARPEN)
    dsn = build_dsn(ns.dsn.DSN, DSN_SEED)
    out = {"vas/checksum": checksums(vas), "dsn/checksum": checksums(dsn)}
    ys_v, ys_d = [], []
    with torch.no_grad():
        for v in range(N_VIDEOS):
            x = sweep_features(v).float().unsqueeze(1)              # (T, 1, 1024) float32 holding bf16 values
            ys_v.append(vas(x.clone()).reshape(-1).numpy())
            ys_d.append(dsn(x).reshape(-1).numpy())
    out["vas/y"] = np.stack(ys_v).astype(np.float32)
    out["dsn/y"] = np.stack(ys_d).astype(np.float32)
    np.savez_compressed(GOLDEN, **out)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes; VASNet scores in", out["vas/y"].min(), out["vas/y"].max(),
          "DSN in", out["dsn/y"].min(), out["dsn/y"].max())


if __name__ == "__main__":
    main()
