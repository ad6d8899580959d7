"""GPU: the scorers AT THE BENCHMARKED CONFIGURATION against goldens of the unmodified reference modules
(tests/golden/sweep_golden.npz, oracle/gen_golden_sweep.py): 17 videos x 2 000 steps, bfloat16 features, through
``score_packed`` — for VASNet that is two row chunks (16 videos, then 1) on the two internal streams, one attention
sub-chunk each (test_vasnet_plan_gpu.py asserts this plan) with the fused exp epilogue (no max subtraction), the fused
head epilogue, i.e. the very path bench.py times, checked against the reference's float32 forward and not against itself."""
import numpy as np
import pytest
import torch

from oracle import gen_golden_sweep as S
from oracle.gen_golden_models import build_dsn, build_vasnet, checksums
from summarizer_b200.models.dsn import DSN
from summarizer_b200.models.vasnet import VASNet

pytestmark = pytest.mark.gpu
GOLDEN = np.load(S.GOLDEN)


def packed_features():
    return torch.cat([S.sweep_features(v) for v in range(S.N_VIDEOS)]).cuda()


def rel_err(got, want):
    return ((got - want).abs() / want.abs().clamp_min(1e-6)).flatten()


def test_vasnet_t2000_bf16_packed_matches_reference():
    m = build_vasnet(VASNet, S.VAS_SEED, {}, S.SHARPEN)
    np.testing.assert_allclose(checksums(m), GOLDEN["vas/checksum"], rtol=1e-12)
    m = m.cuda()
    x = packed_features()
    with torch.no_grad():
        y = m.score_packed(x, [S.T] * S.N_VIDEOS).reshape(S.N_VIDEOS, S.T)
    want = torch.from_numpy(GOLDEN["vas/y"]).cuda()
    rel = rel_err(y, want)
    # north_star's 1e-2 on EVERY one of the 34 000 frames (bf16 features and Q | K | V, float16 attention output / y /
    # their weights, fp32 accumulation)
    frac_over = (rel > 1e-2).float().mean().item()
    print(f"vasnet T=2000 bf16: rel err median {rel.median().item():.2e} p99 {torch.quantile(rel[:1_000_000], 0.99).item():.2e} "
          f"max {rel.max().item():.2e}; frames over 1e-2: {frac_over:.2e}")
    assert rel.max().item() < 1e-2
    # per-video MSE loss against a ramp target: 1e-2 relative
    target = torch.linspace(0, 1, S.T, device="cuda")
    l_got, l_want = ((y - target) ** 2).mean(1), ((want - target) ** 2).mean(1)
    assert ((l_got - l_want).abs() / l_want).max().item() < 1e-2
    # a video scored alone gives the same result as inside the packed, chunked batch (same kernels, other tiling)
    with torch.no_grad():
        alone = m.score_packed(x[: S.T], [S.T])
    assert rel_err(alone, want[0]).max().item() < 1e-2


def test_dsn_t2000_bf16_packed_matches_reference():
    m = build_dsn(DSN, S.DSN_SEED)
    np.testing.assert_allclose(checksums(m), GOLDEN["dsn/checksum"], rtol=1e-12)
    m = m.cuda()
    x = packed_features()
    with torch.no_grad():
        y = m.score_packed(x, [S.T] * S.N_VIDEOS).reshape(S.N_VIDEOS, S.T)
    want = torch.from_numpy(GOLDEN["dsn/y"]).cuda()
    rel = rel_err(y, want)
    print(f"dsn T=2000 bf16: rel err median {rel.median().item():.2e} max {rel.max().item():.2e}")
    assert rel.max().item() < 1e-3
