"""Transformer inference (``smz_mha_forward``; ``score_packed`` -> ``smz_transformer_forward``) across its launch plan,
against a float64 reference.

The encoder runs a packed batch in row chunks of whole videos, up to 32 768 rows each (a longer video is a chunk of its
own); chunk k > 0 reads its input at row ``row0``, writes its attention table at byte ``v0 * 16`` of the table region
and its scores at ``scores + row0``.  The attention kernel is persistent: one work unit is a 128-row query tile of one
(video, head), units are numbered longest video first and CTA b of min(units, SMs) runs units b, b + grid, ...  State
carried from one unit to the next inside a CTA (the Q reload, the S double buffer and the K/V ring position, the
``o_done`` parity, the O accumulator reset, the epilogue pad inside P, the cursor moving across videos) only runs when
a CTA takes more than one unit.  A table of more than 224 videos (3 584 bytes) is uploaded by cudaMemcpyAsync instead
of a by-value kernel argument.

CPU part: oracle/transformer_plan.py restates the chunking, the work-buffer size and the attention schedule; it is
pinned against the library's ``smz_transformer_workspace_bytes`` / ``smz_mha_workspace_bytes``, and every batch below
is asserted to reach the structure it is meant to cover (chunks, units per CTA, video and nk-parity changes between
consecutive units of a CTA, table size), so a change of those constants fails here instead of quietly covering less.
oracle/transformer_ref.py, the float64 reference of the GPU part, is pinned against torch's own module in float64.

GPU part, against oracle/transformer_ref.py in float64 on the device.  Bars as in test_transformer_gpu.py: attention,
worst element within 1e-2 of the head's largest |reference| output; scores, worst-frame relative error 1e-2.
Measured on one NVIDIA B200 (1000 W power limit); attention error per element (|got - ref| / max |ref| of the head)
and score error per frame (relative), median / p95 / max:

  attention   mixed (9 videos, 432 units)                  2.4e-5  9.7e-5  1.1e-3
              wide_table (300 videos, 4 168 units)         5.0e-5  1.8e-4  2.7e-3
              n_heads = 1                                  2.9e-5  1.2e-4  6.9e-4
              n_heads = 2                                  3.3e-5  1.4e-4  9.1e-4
              n_heads = 16                                 3.4e-5  1.4e-4  1.3e-3
              online softmax, 1 000 keys                   2.0e-4  7.1e-4  4.3e-3
  scores      chunk_boundary, 2 layers, bf16 features      6.5e-4  2.0e-3  5.4e-3
                                        float32 features   6.5e-4  2.1e-3  5.6e-3
              chunk_boundary, more_residuals, bf16         5.8e-4  1.8e-3  4.7e-3
                                              float32      5.7e-4  1.8e-3  4.7e-3
              long_video (33 000 keys), 1 layer, bf16      5.2e-4  1.7e-3  4.8e-3
                                                 float32   5.1e-4  1.7e-3  4.1e-3

Neither the chunk boundary nor 33 000 keys moves the worst frame out of the 3e-3 .. 6.5e-3 range measured for short
videos in test_transformer_gpu.py.  The float64 reference takes 0.1 s for chunk_boundary (37 131 rows, 2 layers) and
0.3 s for long_video on the B200, with at most 3.6 GiB allocated on the device (the library's work buffer included).
"""
import time

import ctypes as C
import numpy as np
import pytest
import torch

from oracle import transformer_plan as TP
from oracle import transformer_ref as TR
from summarizer_b200 import _native as N
from summarizer_b200.models.transformer import Transformer
from test_transformer_gpu import (CONFIGS, assert_attention, cu_of, features, make_model, mha, packed_scores,
                                  reference_scores)

gpu = pytest.mark.gpu
SM_COUNT = 148              # B200; the GPU tests take the device's own count
SMALL_UPLOAD = 3584         # upload_small: larger tables go through cudaMemcpyAsync


def wide_lengths():
    return [int(t) for t in np.random.default_rng(11).integers(1, 301, 300)]


# direct smz_mha_forward calls, 8 heads
ATTN = {
    # 504 units, up to 4 per CTA; nk = 63 is odd, so consecutive units start on the other S buffer and ring stage.
    # Run by test_mha_single_video_matches_float64 (test_transformer_gpu.py).
    "many_units": [8000],
    # 432 units; consecutive units of a CTA change video and nk parity
    "mixed": [2001, 1500, 1100, 1000, 257, 256, 129, 128, 1],
    # a 4 800-byte table (cudaMemcpyAsync upload), about 29 units per CTA
    "wide_table": wide_lengths(),
}
# score_packed batches: (lengths, chunks (v0, v1, row0, rows), smz_transformer_workspace_bytes)
MODEL = {
    # two chunks, the second starting at the odd row 32 701
    "chunk_boundary": ([4000] * 8 + [700, 1, 4097, 333], [(0, 10, 0, 32701), (10, 12, 32701, 4430)], 605940736),
    # three chunks, the middle one a single video longer than a chunk
    "long_video": ([3, 33000, 5], [(0, 1, 0, 3), (1, 2, 3, 33000), (2, 3, 33003, 5)], 611425280),
}
# plan only: two chunks of one video each
PLAN_ONLY = {"two_long": ([20000, 20000], [(0, 1, 0, 20000), (1, 2, 20000, 20000)], 370561024)}
# score_packed cases: batch, model configuration
SCORE_CASES = {
    "chunk_boundary_L2": ("chunk_boundary", dict(encoder_layers=2)),
    "chunk_boundary_L2_more_residuals": ("chunk_boundary", dict(encoder_layers=2, more_residuals=True)),
    "long_video_L1": ("long_video", dict(encoder_layers=1)),
}
DTYPES = (torch.bfloat16, torch.float32)


# ---- plan (CPU) ---------------------------------------------------------------------------------------------------
def lib_workspace(lengths):
    cu = cu_of(lengths)
    b = C.c_int64(0)
    N.check(N.lib().smz_transformer_workspace_bytes(cu.ctypes.data_as(C.c_void_p), len(lengths), 0, C.byref(b)))
    return b.value


def lib_table(n_videos):
    b = C.c_int64(0)
    N.check(N.lib().smz_mha_workspace_bytes(n_videos, C.byref(b)))
    return b.value


def random_batches():
    rng = np.random.default_rng(8)
    out = []
    for _ in range(200):
        hi = int(rng.choice([16, 300, 3000, 20000, 40000]))
        out.append([int(t) for t in rng.integers(1, hi + 1, int(rng.integers(1, 400 if hi <= 300 else 50)))])
    return out


def test_plan_restatement_matches_library():
    """Work-buffer size (largest chunk's buffers + the whole batch's table) and table size agree with the restatement
    on the named batches and 200 random ones."""
    named = list(ATTN.values()) + [c[0] for c in MODEL.values()] + [c[0] for c in PLAN_ONLY.values()]
    for lengths in named + random_batches():
        assert lib_workspace(lengths) == TP.workspace_bytes(lengths), lengths
        assert lib_table(len(lengths)) == TP.table_bytes(len(lengths)), len(lengths)


@pytest.mark.parametrize("case", list(MODEL) + list(PLAN_ONLY))
def test_batch_reaches_its_plan(case):
    lengths, want, nbytes = (MODEL[case] if case in MODEL else PLAN_ONLY[case])
    got = [tuple(c) for c in TP.chunks(lengths)]
    assert got == want, f"{case}: chunks {got}, meant to reach {want}"
    assert lib_workspace(lengths) == TP.workspace_bytes(lengths) == nbytes
    if case == "chunk_boundary":
        assert got[1][2] % 2 == 1 and got[1][1] - got[1][0] > 1, "chunk 1 starts at an odd row and holds several videos"
    if case == "long_video":
        assert got[1][1] - got[1][0] == 1 and got[1][3] > TP.ROW_CHUNK, "a video longer than a chunk, alone"


def assert_schedule(case, sm_count):
    """The structure each attention batch is there to cover, on a device of sm_count SMs."""
    lengths = ATTN[case]
    sched = TP.mha_schedule(lengths, 8, sm_count)
    units = [u for cta in sched for u in cta]
    assert len(units) == len(set(units)) == 8 * sum((T + 127) // 128 for T in lengths)
    assert min(len(cta) for cta in sched) >= 2, f"{case}: some CTA runs a single unit"
    pairs = [(a, b) for cta in sched for a, b in zip(cta, cta[1:])]
    odd_start = sum(sum(u.nk for u in cta[:i]) % 2 for cta in sched for i in range(len(cta)))
    parity = sum(a.nk % 2 != b.nk % 2 for a, b in pairs)
    video = sum(a.video != b.video for a, b in pairs)
    if case == "many_units":
        assert odd_start > 0, "no unit starts on S buffer 1"
    else:
        assert parity > 0 and video > 0, f"{case}: {parity} nk-parity and {video} video changes between units"
    if case == "wide_table":
        assert len(lengths) * TP.TABLE_ENTRY > SMALL_UPLOAD
    return len(units), max(len(cta) for cta in sched), parity, video


@pytest.mark.parametrize("case", list(ATTN))
def test_attention_batch_reaches_its_schedule(case):
    units, per_cta, parity, video = assert_schedule(case, SM_COUNT)
    if case == "many_units":
        assert (units, per_cta) == (504, 4)
    if case == "mixed":
        assert (units, parity, video) == (432, 116, 284)
    if case == "wide_table":
        assert per_cta >= 28


def test_attention_reference_blocks_match_whole_softmax(monkeypatch):
    """TR.attention in small query blocks, 1 / 2 / 16 heads with a wider row stride, equals the softmax over whole
    logit matrices."""
    monkeypatch.setattr(TR, "BLOCK_BYTES", 4096)
    lengths = [3, 40, 1, 17]
    g = torch.Generator().manual_seed(3)
    for nh in (1, 2, 16):
        qkv = torch.randn(sum(lengths), 3 * nh * 128 + 64, generator=g, dtype=torch.float64)
        want = torch.empty(sum(lengths), nh * 128, dtype=torch.float64)
        for (r0, r1) in zip(cu_of(lengths)[:-1], cu_of(lengths)[1:]):
            for h in range(nh):
                q, k, v = (qkv[r0:r1, (i * nh + h) * 128:(i * nh + h + 1) * 128] for i in range(3))
                want[r0:r1, h * 128:(h + 1) * 128] = torch.softmax(q @ k.t() / np.sqrt(128.0), dim=1) @ v
        assert (TR.attention(qkv, lengths, nh) - want).abs().max().item() < 1e-13


def embedded(m, x, lengths):
    """x plus the module's positional embedding of each video (what forward adds before the encoder)."""
    if not m.max_length:
        return x
    parts = []
    for xv in torch.split(x, list(lengths)):
        T = xv.shape[0]
        pe = m.pos_embed(torch.arange(T)) if m.pos_embed_type == "simple" else m.pos_embed[:T]
        parts.append(xv.double() + pe.detach().double())
    return torch.cat(parts)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_reference_matches_torch_module(cfg):
    """The float64 restatement equals copy.deepcopy(m).double().eval() (torch's TransformerEncoder) on a ragged batch."""
    m = make_model(cfg)
    lengths = [5, 1, 37, 130]
    x = features(lengths, 9, torch.float32)
    want = reference_scores(m, x, lengths)
    with torch.no_grad():
        got = TR.scores(m, embedded(m, x, lengths), lengths)
    assert (got - want).abs().max().item() < 1e-12


# ---- GPU: attention -----------------------------------------------------------------------------------------------
def stats(err):
    s = err.flatten().sort().values
    return s[len(s) // 2].item(), s[int(0.95 * (len(s) - 1))].item(), s[-1].item()


def random_qkv(lengths, seed, width=3072, scale=1.0):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return (torch.randn(sum(lengths), width, generator=g, device="cuda") * scale).bfloat16()


def bf16_bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int16), b.view(torch.int16))


def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


@gpu
@pytest.mark.parametrize("case", list(ATTN))
def test_attention_batch_reaches_its_schedule_on_this_device(case):
    print(f"{case}: {sm_count()} SMs: units, most per CTA, parity / video changes {assert_schedule(case, sm_count())}")


@gpu
@pytest.mark.parametrize("case", ["mixed", "wide_table"])
def test_attention_batch_matches_float64(case):
    lengths = ATTN[case]
    _, err = assert_attention(random_qkv(lengths, 20), lengths)
    print(f"{case}: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
@pytest.mark.parametrize("case", ["mixed", "wide_table"])
def test_attention_invariance(case):
    """Bit equality, per video: (1) two calls; (2) the batch in another video order (other rows; for the wide table,
    whose lengths repeat, other CTAs and other positions in a CTA's sequence of units); (3) every other video's rows
    replaced by different finite values scaled by 50.  Any state leaking from one unit to the next, or any key of
    another video reaching a softmax, changes some bits."""
    lengths = ATTN[case]
    cu = cu_of(lengths)
    qkv = random_qkv(lengths, 21)
    rc, out = mha(qkv, lengths)
    assert rc == 0, N.lib().smz_last_error()
    assert bf16_bits_equal(mha(qkv, lengths)[1], out), "a repeated call differs"
    perm = [int(v) for v in np.random.default_rng(5).permutation(len(lengths))]
    plen = [lengths[v] for v in perm]
    if case == "wide_table":
        where = {(u.video, u.head, u.qt): (b, i) for b, cta in enumerate(TP.mha_schedule(lengths, 8, sm_count()))
                 for i, u in enumerate(cta)}
        moved = sum(where[(perm[u.video], u.head, u.qt)] != (b, i)
                    for b, cta in enumerate(TP.mha_schedule(plen, 8, sm_count())) for i, u in enumerate(cta))
        assert moved > len(where) // 10, f"only {moved} of {len(where)} units change CTA or position"
    rc, pout = mha(torch.cat([qkv[cu[v]:cu[v + 1]] for v in perm]), plen)
    assert rc == 0, N.lib().smz_last_error()
    pcu = cu_of(plen)
    for i, v in enumerate(perm):
        assert bf16_bits_equal(pout[pcu[i]:pcu[i + 1]], out[cu[v]:cu[v + 1]]), \
            f"video {v} ({lengths[v]} frames) differs in the permuted batch"
    other = random_qkv(lengths, 22, scale=50.0)
    assert torch.isfinite(other.float()).all()
    for v in range(len(lengths)):
        x = other.clone()
        x[cu[v]:cu[v + 1]] = qkv[cu[v]:cu[v + 1]]
        rc, iso = mha(x, lengths)
        assert rc == 0, N.lib().smz_last_error()
        assert bf16_bits_equal(iso[cu[v]:cu[v + 1]], out[cu[v]:cu[v + 1]]), \
            f"video {v} ({lengths[v]} frames) changes when the other videos' rows change"


@gpu
@pytest.mark.parametrize("n_heads", [1, 2, 16])
def test_attention_head_count_and_strides(n_heads):
    """Any head count with ld = 3 * n_heads * 128 + 64 (the 64 extra input columns are NaN and never read) and
    ldo = n_heads * 128 + 24: the 24 extra output columns keep their NaN sentinel; every head matches float64."""
    lengths = [300, 1, 129, 1000, 77, 256]
    w = n_heads * 128
    qkv = random_qkv(lengths, 23 + n_heads, width=3 * w + 64)
    qkv[:, 3 * w:] = float("nan")
    out, err = assert_attention(qkv, lengths, n_heads, ldo=w + 24)
    assert torch.isnan(out[:, w:].float()).all(), "columns past n_heads * 128 were written"
    print(f"n_heads={n_heads}: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
def test_online_softmax_rescales_per_warp():
    """One 1000-key video (8 key tiles).  Q and K of every head are built along one direction so that, in query tile 0,
    the row maximum rises in every key tile for rows 0-63 (softmax warps 0 and 1 rescale O after each tile, with a
    different alpha per row) and only in the first tile for rows 64-127 (warps 2 and 3 never rescale)."""
    T, nh = 1000, 8
    g = torch.Generator(device="cuda")
    g.manual_seed(24)
    qkv = torch.randn(T, 3 * nh * 128, generator=g, device="cuda") * 0.5
    trend = torch.arange(T, device="cuda") * (4.0 / T)
    sign = torch.where(torch.arange(128, device="cuda") < 64, 1.0, -1.0)
    c = sign * (20.0 + 10.0 * (torch.arange(128, device="cuda") % 64) / 64)
    for h in range(nh):
        qkv[:128, h * 128] = c
        qkv[:, (nh + h) * 128] = trend
    qkv = qkv.bfloat16()
    q64 = qkv.double()
    for h in range(nh):
        s = q64[:128, h * 128:(h + 1) * 128] @ q64[:, (nh + h) * 128:(nh + h + 1) * 128].t()
        tile_max = torch.stack([s[:, j:j + 128].amax(dim=1) for j in range(0, T, 128)], 1)     # [128, 8]
        run = tile_max.cummax(dim=1).values
        assert (tile_max[:64, 1:] > run[:64, :-1]).all(), "rows 0-63: the maximum must rise in every key tile"
        assert (tile_max[64:, 1:] < tile_max[64:, :1]).all(), "rows 64-127: the maximum must stay in the first tile"
    _, err = assert_attention(qkv, [T])
    print("online softmax: attention error median %.2e p95 %.2e max %.2e" % stats(err))


# ---- GPU: scores of the whole model -------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("case", list(SCORE_CASES))
def test_packed_scores_across_chunks(case, dtype):
    """score_packed against the float64 reference, every video bit-equal to itself scored alone and in the reversed
    batch (other chunks, other row offsets)."""
    batch, cfg = SCORE_CASES[case]
    lengths = MODEL[batch][0]
    torch.manual_seed(30)
    m = Transformer(**cfg).eval().cuda()
    g = torch.Generator(device="cuda")
    g.manual_seed(31)
    x = torch.randn(sum(lengths), 1024, generator=g, device="cuda").abs().to(dtype)     # non-negative, as pool5
    got = packed_scores(m, x, lengths)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    with torch.no_grad():
        want = TR.scores(m, x, lengths)
    torch.cuda.synchronize()
    rel = (got.double() - want).abs() / want.abs().clamp_min(1e-6)
    med, p95, mx = stats(rel)
    print(f"{case} {dtype}: worst-frame rel err median {med:.2e} p95 {p95:.2e} max {mx:.2e}; "
          f"float64 reference {time.perf_counter() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    assert mx <= 1e-2, mx
