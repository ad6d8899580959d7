"""SumGAN-att selector inference timings on the GPU (CUDA events), in one run:
  - Transformer.score_packed of models/sumgan_att.py (sm_100a kernels; 2 layers, 4 heads of 256) at a sweep shape
    (256 videos x T=2000, bf16 features) and at the synthetic TVSum shape (50 videos, float32 features);
  - the selector's torch modules on the same GPU: float32, eval(), one video per call (the reference's loop), and bf16
    with 16 videos per call;
  - the fused attention kernel alone (smz_mha_forward) at the sweep shape, 4 heads of 256 next to 8 heads of 128 (the
    same 4 T^2 D flops per video);
  - the native scores against the torch float32 scores on the same seeded inputs.
Algorithmic work per video: L (12 T D^2 + 4 T^2 D) + 2 T D flops.  Prints the card name and power limit; writes one JSON
line per measurement (stdout, and --out FILE when given)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from summarizer_b200 import _native as N
from summarizer_b200 import synthetic
from summarizer_b200.models.sumgan_att import Transformer

D, L, HEADS = 1024, 2, 4


def flops(lengths):
    return sum(L * (12 * T * D * D + 4 * T * T * D) + 2 * T * D for T in lengths)


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / iters


def torch_forward(sel, x):
    """The selector's torch modules (eval: dropout inactive), whatever path Transformer.forward would take."""
    return sel.out(sel.transformer_encoder(x))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sweep-videos", type=int, default=256)
    ap.add_argument("--torch-fp32-videos", type=int, default=32, help="videos of the sweep shape the fp32 loop times")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sumgan_att_perf.py measures on a CUDA device; none found")
    rows = []

    def emit(d):
        rows.append(d)
        print(json.dumps(d), flush=True)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    emit({"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else None})

    torch.manual_seed(0)
    m = Transformer(encoder_layers=L, attention_heads=HEADS).cuda().eval()
    mb = Transformer(encoder_layers=L, attention_heads=HEADS).cuda().eval()
    mb.load_state_dict(m.state_dict())
    mb = mb.to(torch.bfloat16)

    rng = np.random.default_rng(0)
    shapes = {
        "sweep": ([2000] * args.sweep_videos, torch.bfloat16),
        "tvsum": ([int(synthetic.make_video("tvsum", i, with_features=False)["n_steps"]) for i in range(50)], torch.float32),
    }
    for name, (lengths, dtype) in shapes.items():
        x = torch.from_numpy(np.abs(rng.standard_normal((sum(lengths), D), dtype=np.float32))).cuda().to(dtype)
        fl = flops(lengths)
        with torch.no_grad():
            s = timed(lambda: m.score_packed(x, lengths), 3)
            emit({"shape": name, "path": "score_packed", "features": str(dtype).split(".")[-1], "videos": len(lengths),
                  "frames": sum(lengths), "s": round(s, 5), "videos_per_s": round(len(lengths) / s, 1),
                  "tflops": round(fl / s / 1e12, 1)})
            native = m.score_packed(x, lengths)
            nv32 = min(len(lengths), args.torch_fp32_videos)
            cu = np.concatenate([[0], np.cumsum(lengths)])
            xs32 = [x[cu[i]:cu[i + 1]].float().unsqueeze(1).contiguous() for i in range(nv32)]
            s32 = timed(lambda: [torch_forward(m, xi) for xi in xs32], 1)
            emit({"shape": name, "path": "torch_fp32_one_video_per_call", "videos": nv32, "s": round(s32, 5),
                  "videos_per_s": round(nv32 / s32, 1), "tflops": round(flops(lengths[:nv32]) / s32 / 1e12, 1)})
            out32 = torch.cat([torch_forward(m, xi).reshape(-1) for xi in xs32])
            rel = ((native[:cu[nv32]] - out32).abs() / out32.abs().clamp_min(1e-6))
            emit({"shape": name, "compare": "score_packed vs torch fp32", "videos": nv32,
                  "max_rel": float(rel.max()), "p95_rel": float(rel.quantile(0.95)) if rel.numel() < 1 << 24 else None})
            # stock torch, bf16, 16 equal-length videos per call (ragged sets are grouped by length)
            groups = {}
            for i, T in enumerate(lengths):
                groups.setdefault(T, []).append(i)
            batches = []
            for T, idx in groups.items():
                for k in range(0, len(idx), 16):
                    sel = idx[k:k + 16]
                    batches.append(torch.stack([x[cu[i]:cu[i + 1]] for i in sel], 1).to(torch.bfloat16).contiguous())
            sb = timed(lambda: [torch_forward(mb, b) for b in batches], 1)
            emit({"shape": name, "path": "torch_bf16_16_videos_per_call", "videos": len(lengths), "s": round(sb, 5),
                  "videos_per_s": round(len(lengths) / sb, 1), "tflops": round(fl / sb / 1e12, 1)})
        del x

    # attention kernel alone at the sweep shape: 4 heads of 256 and 8 heads of 128 on the same qkv rows
    lengths = [2000] * args.sweep_videos
    qkv = torch.randn(sum(lengths), 3 * D, device="cuda").to(torch.bfloat16)
    out = torch.empty(sum(lengths), D, device="cuda", dtype=torch.bfloat16)
    cu = np.zeros(len(lengths) + 1, dtype=np.int32)
    np.cumsum(lengths, out=cu[1:])
    nb = C.c_int64(0)
    N.check(N.lib().smz_mha_workspace_bytes(len(lengths), C.byref(nb)))
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    af = sum(4 * T * T * D for T in lengths)
    for heads, width in ((4, 256), (8, 128)):
        def att():
            N.check(N.lib().smz_mha_forward(N.ptr(qkv), 3 * D, cu.ctypes.data_as(C.c_void_p), len(lengths), heads, width,
                                            N.ptr(out), D, N.ptr(ws), ws.numel(), N.current_stream()))
        s = timed(att, 10)
        emit({"shape": "sweep", "path": "smz_mha_forward", "heads": heads, "head_dim": width, "videos": len(lengths),
              "s": round(s, 6), "tflops": round(af / s / 1e12, 1)})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
