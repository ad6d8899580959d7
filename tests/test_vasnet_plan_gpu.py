"""VASNet inference (``score_packed`` -> smz_vasnet_forward) across its launch plan, against a float64 reference.

The packed forward splits a batch into row chunks of up to 32 768 rows, each chunk into attention sub-chunks of up to
68 Mi logits, and runs consecutive chunks on two internal streams ("lanes"), each with its own copy of the chunk
buffers: chunk k uses lane k & 1, so chunk 2 reuses chunk 0's buffers.  The row-sum slots of the fused softmax are
indexed by the chunk-local row and zeroed first when some video of the chunk writes fewer of them ("ragged").

CPU part: oracle/vasnet_plan.py restates the plan; it is pinned against the library's own launch count and work-buffer
size, and every batch below is asserted to reach the plan structure it is meant to cover, so a change of the chunk or
budget constants fails here instead of silently shrinking what the GPU tests cover.

GPU part: each batch, with bfloat16 and with float32 features, on the fast path and on the exact path, against the
reference forward (oracle/models_torch.py) run in float64 on the device through torch, fed with the module's float32
parameters: the folded weights and every fused epilogue are checked against the unfolded reference.  Bars per frame
are set from B200 measurements (NVIDIA B200, 1000 W power limit); relative error per frame, median / p95 / max:

  case               fast, bf16 features   fast, fp32 features   exact, bf16 features  exact, fp32 features
  multi_sub          8.8e-4 2.4e-3 6.3e-3  1.2e-4 4.8e-4 1.9e-3  1.2e-3 5.0e-3 1.6e-2  1.2e-3 5.0e-3 1.7e-2
  lane_reuse         3.9e-4 1.6e-3 5.3e-3  2.1e-4 7.7e-4 3.0e-3  9.1e-4 4.2e-3 1.6e-2  9.1e-4 4.2e-3 1.7e-2
  lane_reuse_ragged  1.7e-3 3.9e-3 8.0e-3  8.3e-4 1.7e-3 3.3e-3  5.2e-3 1.3e-2 2.6e-2  5.2e-3 1.3e-2 2.8e-2
  unaligned          2.6e-3 4.8e-3 8.9e-3  2.9e-4 9.3e-4 3.4e-3  5.0e-3 1.3e-2 2.7e-2  5.0e-3 1.3e-2 2.9e-2
  tile_edges         1.4e-4 6.7e-4 2.3e-3  3.0e-5 1.9e-4 1.4e-3  3.5e-4 1.9e-3 6.8e-3  3.6e-4 2.0e-3 8.1e-3

The fast path with float32 features meets the bf16 bars of test_vasnet_gpu.py (worst frame 1e-2, p95 3e-3, absolute
2e-3).  With bf16 features its worst frame stays under 1e-2, but p95 reaches 4.8e-3 and the absolute error 2.5e-3 on
the long rows: the features are then the bf16 logit operands (float32 features go through float16).  The exact path
(the fallback when a range check trips) does not reach 1e-2 at these lengths: worst frame 2.9e-2, p95 1.3e-2.  Most
of that sits after the attention: with Wv scaled by 1e-5, so that attention adds almost nothing to y, the exact path
still reaches 2.2e-2 (bf16 LayerNorm output and W1 in the literal chain, where the fast path uses float16).
"""
import os
import subprocess
import sys

import ctypes as C
import numpy as np
import pytest
import torch

from oracle import models_torch as MT
from oracle import vasnet_plan as VP
from oracle.gen_golden_models import build_vasnet
from summarizer_b200 import _native as N
from summarizer_b200.models.vasnet import VASNet, _cu_seqlens, _Workspace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# (worst frame, p95, absolute) per frame, see the module docstring; the exact path's are those of test_vasnet_gpu.py
BARS = {("fast", "fp32"): (1e-2, 3e-3, 2e-3), ("fast", "bf16"): (1e-2, 6e-3, 3e-3),
        ("exact", "fp32"): (4e-2, 2e-2, 1.2e-2), ("exact", "bf16"): (4e-2, 2e-2, 1.2e-2)}

TILE_EDGES = [1, 2, 7, 8, 9, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513]
# name -> (lengths, videos per sub-chunk of each chunk, ragged per chunk, weight seed, sharpen)
CASES = {
    # chunk 0: two 6000-frame videos are 72.2 M logits > 71.3 M, one sub-chunk per video; chunk 1 ragged
    "multi_sub": ([6000] * 6 + [1234, 777, 1], [[1, 1, 1, 1, 1], [4]], [False, True], 51, 6.0),
    # three chunks: chunk 2 reuses lane 0's buffers
    "lane_reuse": ([2000] * 40, [[16], [16], [8]], [False, False, False], 52, 5.0),
    # the same, and chunk 2 is ragged while chunk 0, whose slots it reuses, wrote all of them
    "lane_reuse_ragged": ([2000] * 32 + [2000, 700, 1999, 129, 2000, 1], [[16], [16], [6]], [False, False, True], 53, 4.0),
    # odd row offsets across the chunk boundary; 12 345 and 9 999 frames are each over the budget (admitted alone)
    "unaligned": ([4097, 8191, 1, 12345, 7, 9999, 2049, 255, 257], [[1, 2, 1, 1], [1, 3]], [True, True], 54, 6.0),
    # GEMM M / N tails, the 64-column exp padding, videos with fewer row-sum slots than the sub-chunk
    "tile_edges": (TILE_EDGES, [[20]], [True], 55, 5.0),
}
# batches whose plan is documented elsewhere: the sweep golden (test_sweep_golden_gpu.py) crosses one chunk boundary
PLAN_ONLY = {"sweep_golden": ([2000] * 17, [[16], [1]], [False, False])}
DTYPES = ("bf16", "fp32")
gpu = pytest.mark.gpu


# ---- plan (CPU) ---------------------------------------------------------------------------------------------------
def lib_launches(lengths, mode, x_bf16):
    """smz_vasnet_launch_count (mode 0: fast inference path, 2: exact inference path)."""
    cu = _cu_seqlens(lengths)
    n = C.c_int64(0)
    N.check(N.lib().smz_vasnet_launch_count(cu.ctypes.data_as(C.c_void_p), len(lengths), mode, x_bf16, C.byref(n)))
    return n.value


def lib_plan(lengths):
    """(chunks, sub-chunks) of the library's plan.  A chunk of the fast path issues cvt + 3 + 2 * subs launches, cvt = 1
    for float32 features (their float16 copy) and 0 for bf16 ones."""
    n_f32, n_bf16 = lib_launches(lengths, 0, 0), lib_launches(lengths, 0, 1)
    chunks = n_f32 - n_bf16
    assert (n_bf16 - 3 * chunks) % 2 == 0
    return chunks, (n_bf16 - 3 * chunks) // 2


def lib_workspace(lengths, x_bf16):
    cu = _cu_seqlens(lengths)
    b = C.c_int64(0)
    N.check(N.lib().smz_vasnet_workspace_bytes(cu.ctypes.data_as(C.c_void_p), len(lengths), 0, x_bf16, C.byref(b)))
    return b.value


def random_batches():
    rng = np.random.default_rng(7)
    out = []
    for _ in range(200):
        hi = int(rng.choice([16, 300, 3000, 9000, 40000]))
        out.append([int(t) for t in rng.integers(1, hi + 1, int(rng.integers(1, 50)))])
    return out


def test_plan_restatement_matches_library():
    """Chunks and sub-chunks from the launch counts, the exact path's launch count and the work-buffer size (which holds
    one copy of the chunk buffers per lane) agree with the restatement on the named and 200 random batches."""
    named = [c[0] for c in CASES.values()] + [c[0] for c in PLAN_ONLY.values()]
    for lengths in named + random_batches():
        chunks = VP.plan(lengths)
        assert lib_plan(lengths) == (len(chunks), sum(len(c.subs) for c in chunks)), lengths
        for x_bf16 in (0, 1):
            assert lib_launches(lengths, 2, x_bf16) == VP.launch_count(chunks, x_bf16, exact=True), lengths
            assert lib_workspace(lengths, x_bf16) == VP.workspace_bytes(lengths, x_bf16), lengths


@pytest.mark.parametrize("case", list(CASES) + list(PLAN_ONLY))
def test_batch_reaches_its_plan(case):
    lengths, subs, ragged = (CASES[case] if case in CASES else PLAN_ONLY[case])[:3]
    chunks = VP.plan(lengths)
    assert lib_plan(lengths) == (len(chunks), sum(len(c.subs) for c in chunks))
    assert len(chunks) == len(subs), f"{case}: {len(chunks)} chunks, meant to reach {len(subs)}"
    got = [[s.v1 - s.v0 for s in c.subs] for c in chunks]
    assert got == subs, f"{case}: videos per sub-chunk {got}, meant to reach {subs}"
    assert [c.ragged for c in chunks] == ragged, f"{case}: ragged chunks {[c.ragged for c in chunks]}, meant {ragged}"
    if case == "unaligned":
        over = [s for c in chunks for s in c.subs if s.rows * s.ld > VP.LOGIT_BUDGET]
        assert [s.v1 - s.v0 for s in over] == [1, 1], "one video over the logits budget in each chunk, admitted alone"
        assert sum(lengths[:chunks[1].v0]) % 2 == 1, "chunk 1 starts at an odd row"
        assert VP.workspace_bytes(lengths, 0) > 2.5 * 2 ** 30, "two lanes of buffers for a 152 M-logit sub-chunk"


# ---- GPU: reference and helpers -----------------------------------------------------------------------------------
def features(lengths, seed, dtype):
    """Non-negative, L2-normalised rows (pool5-like, as oracle.gen_golden_models.make_input), drawn on the device."""
    g = torch.Generator(device="cuda")
    g.manual_seed(1000 + seed)
    x = torch.randn(sum(lengths), 1024, generator=g, device="cuda").abs()
    x = x / x.norm(dim=1, keepdim=True)
    return x.bfloat16() if dtype == "bf16" else x


def setup(case, dtype):
    lengths, _, _, seed, sharpen = CASES[case]
    return build_vasnet(VASNet, seed, {}, sharpen).cuda(), features(lengths, seed, dtype), lengths


def reference(m, x, lengths):
    """The reference forward in float64 on the device, one video at a time; bf16 features are widened as they are."""
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    with torch.no_grad():
        return MT.vasnet_forward_packed(sd, x.double(), lengths, scale=m.scale, eps=m.epsilon, aperture=m.aperture,
                                        ignore_self=m.ignore_self)


_REF = {}


def cached_reference(key, m, x, lengths):
    if key not in _REF:
        _REF[key] = reference(m, x, lengths)
    return _REF[key]


def check_close(label, got, want, bars):
    """NaN exactly where the reference is NaN; elsewhere the per-frame bars (worst frame, p95, absolute)."""
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), \
        f"{label}: NaN at frames {torch.nonzero(torch.isnan(got) != nan).flatten()[:16].tolist()} (reference disagrees)"
    if bool(nan.all()):
        print(f"{label}: all {nan.numel()} frames NaN, as the reference")
        return
    err = (got[~nan].double() - want[~nan]).abs()
    rel = err / want[~nan].abs().clamp_min(1e-6)
    med, p95, mx, ab = rel.median().item(), torch.quantile(rel, 0.95).item(), rel.max().item(), err.max().item()
    print(f"{label}: rel err median {med:.2e} p95 {p95:.2e} max {mx:.2e}; abs max {ab:.2e}"
          + (f"; {int(nan.sum())} NaN frames as the reference" if bool(nan.any()) else ""))
    assert mx < bars[0] and p95 < bars[1] and ab < bars[2], \
        f"{label}: relative error max {mx:.3e} p95 {p95:.3e}, absolute {ab:.3e}"


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def fast_scores(m, x, lengths):
    """The fast path without its fallback: the test fails if the range guard fired (then the fast path was not what
    got measured)."""
    y = m.score_packed(x, lengths, check=False)
    assert m._shadow["fast_ok"] and m.check_status(), "the fast path left its checked value range"
    return y


# ---- GPU: each batch against the reference --------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(CASES))
def test_fast_path_matches_float64_reference(case, dtype):
    m, x, lengths = setup(case, dtype)
    check_close(f"{case} {dtype} fast", fast_scores(m, x, lengths), cached_reference((case, dtype), m, x, lengths),
                BARS["fast", dtype])


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(CASES))
def test_exact_path_matches_float64_reference(case, dtype):
    m, x, lengths = setup(case, dtype)
    check_close(f"{case} {dtype} exact", m.score_packed(x, lengths, exact=True),
                cached_reference((case, dtype), m, x, lengths), BARS["exact", dtype])


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", ["multi_sub", "lane_reuse_ragged"])
def test_weights_outside_the_fast_range_take_the_exact_path(case, dtype):
    """Wo.Wv under the 1e-3 floor: fast_ok is False, so the call runs without a status word (exact chain, fused head)."""
    m, x, lengths = setup(case, dtype)
    with torch.no_grad():
        m.V.weight.mul_(1e-5)
    y = m.score_packed(x, lengths)
    assert not m._shadow["fast_ok"]
    assert same_bits(y, m.score_packed(x, lengths, exact=True))
    check_close(f"{case} {dtype} small Wv", y, reference(m, x, lengths), BARS["exact", dtype])


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(CASES))
def test_packed_rows_equal_each_video_alone(case, dtype):
    """Inference reads V in place (no leading pad columns at any row offset), so a video's rows inside the packed,
    chunked batch are bit-identical to the video scored alone, on both paths."""
    m, x, lengths = setup(case, dtype)
    for exact in (False, True):
        packed = m.score_packed(x, lengths, check=False, exact=exact)
        bad, o = [], 0
        for T in lengths:
            alone = m.score_packed(x[o:o + T], [T], check=False, exact=exact)
            if not same_bits(packed[o:o + T], alone):
                bad.append((o, T, (packed[o:o + T] - alone).abs().max().item()))
            o += T
        assert m.check_status()
        assert not bad, f"exact={exact}: (row0, T, max diff) of videos that differ from their own call: {bad[:8]}"


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(CASES))
def test_poisoned_work_buffer_changes_nothing(case, dtype):
    """0xFF bytes read as NaN in float32, bf16 and float16: a slot, padding column or lane copy read before it is
    written turns the repeat into NaN instead of passing on whatever the allocator handed out."""
    m, x, lengths = setup(case, dtype)
    for exact in (False, True):
        first = m.score_packed(x, lengths, check=False, exact=exact)
        m._ws.buf.fill_(0xFF)
        again = m.score_packed(x, lengths, check=False, exact=exact)
        assert m.check_status() and torch.isfinite(first).all()
        assert same_bits(first, again), \
            f"exact={exact}: {int(torch.isnan(again).sum())} NaN frames, {int((first != again).sum())} differ after poisoning"


# ---- GPU: attention options ---------------------------------------------------------------------------------------
OPTIONS = {"aperture300": (300, False), "ignore_self": (None, True), "aperture300_ignore_self": (300, True)}


@gpu
@pytest.mark.parametrize("opt", list(OPTIONS))
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", ["multi_sub", "tile_edges"])
def test_attention_options_across_sub_chunks(case, dtype, opt):
    """A 300-frame aperture crosses the 256-column tiles; ignore_self masks the diagonal.  Both batches hold a T = 1
    video, whose row ignore_self masks completely: NaN there as in the reference, and the NaN sum of squares raises the
    float16-range bit, so the fast result is checked unchecked (check=False)."""
    m, x, lengths = setup(case, dtype)
    m.aperture, m.ignore_self = OPTIONS[opt]
    want = reference(m, x, lengths)
    y = m.score_packed(x, lengths, check=False)
    assert m.check_status() == (not bool(torch.isnan(want).any()))
    check_close(f"{case} {dtype} {opt} fast", y, want, BARS["fast", dtype])
    check_close(f"{case} {dtype} {opt} exact", m.score_packed(x, lengths, exact=True), want, BARS["exact", dtype])


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("lengths, aperture", [(TILE_EDGES, 0), ([1], None), ([300, 1, 257, 1, 64], None)],
                         ids=["aperture0_tile_edges", "t1_alone", "t1_among_others"])
def test_fully_masked_rows_are_nan_where_the_reference_is(lengths, aperture, dtype):
    """ignore_self with aperture 0 masks every row, ignore_self on a T = 1 video its only row: softmax of all -inf is
    NaN, and the score too (the k1 ReLU epilogue once turned the NaN into 0 and gave such rows a finite score).  The
    NaN trips the float16-range guard, so score_packed(check=True) repeats the call on the exact path."""
    m = build_vasnet(VASNet, 56, {"ignore_self": True, "attention_aperture": aperture}, 5.0).cuda()
    x = features(lengths, 56, dtype)
    want = reference(m, x, lengths)
    assert torch.isnan(want).any()
    unchecked = m.score_packed(x, lengths, check=False)
    assert not m.check_status(), "a NaN row must raise the status word"
    exact = m.score_packed(x, lengths, exact=True)
    check_close(f"{len(lengths)} videos aperture={aperture} {dtype} fast", unchecked, want, BARS["fast", dtype])
    check_close(f"{len(lengths)} videos aperture={aperture} {dtype} exact", exact, want, BARS["exact", dtype])
    assert same_bits(m.score_packed(x, lengths), exact)


# ---- GPU: range guard, ordering, work buffer, sub-chunk budget ----------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_range_guard_tripped_by_the_last_chunk_only(dtype):
    """Features of one video in chunk 2 scaled until its logits leave [-80, 80]: the whole call is void and repeated
    on the exact path, while the rows of the untouched chunks were computed exactly as in a clean call."""
    m, x32, lengths = setup("lane_reuse", "fp32")
    last = VP.plan(lengths)[-1]
    row0 = sum(lengths[:last.v0])
    v = last.v0 + 3
    o, T = sum(lengths[:v]), lengths[v]
    with torch.no_grad():
        xv = x32[o:o + T]
        amax = ((xv @ m.Q.weight.t()) @ (xv @ m.K.weight.t()).t() * m.scale).abs().max().item()
    hot = x32.clone()
    hot[o:o + T] *= (200.0 / amax) ** 0.5         # logits scale with the square: the largest becomes ~200
    clean_x, hot_x = (t.bfloat16() if dtype == "bf16" else t for t in (x32, hot))
    clean = fast_scores(m, clean_x, lengths)
    unchecked = m.score_packed(hot_x, lengths, check=False)
    status = int(m._status.item())
    assert status & 1, f"status {status}: the logit-range bit did not fire"
    assert not m.check_status() and m.check_status(), "check_status() reports the violation once, then clears it"
    assert same_bits(unchecked[:row0], clean[:row0]), "rows of chunks 0 and 1 changed"
    assert same_bits(m.score_packed(hot_x, lengths), m.score_packed(hot_x, lengths, exact=True))


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_calls_are_ordered_on_the_callers_stream(dtype):
    """The lanes fork from and join back into the caller's stream: a repeat gives the same bits, and a call issued and
    consumed on a non-default stream equals the default-stream result."""
    m, x, lengths = setup("lane_reuse_ragged", dtype)
    fast, exact = fast_scores(m, x, lengths), m.score_packed(x, lengths, exact=True)
    assert same_bits(fast, fast_scores(m, x, lengths))
    assert same_bits(exact, m.score_packed(x, lengths, exact=True))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ok_fast = same_bits(m.score_packed(x, lengths, check=False), fast)     # compared on `side`, before any join
        ok_exact = same_bits(m.score_packed(x, lengths, exact=True), exact)
    torch.cuda.current_stream().wait_stream(side)
    assert m.check_status() and ok_fast and ok_exact


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_back_to_back_calls_that_grow_the_work_buffer(dtype):
    """A second, larger call grows the work buffer while the first may still be running; no synchronisation between
    them.  Both equal the same calls made one at a time."""
    (small, *_), (big, *_) = CASES["lane_reuse"], CASES["unaligned"]
    assert VP.workspace_bytes(big, dtype == "bf16") > VP.workspace_bytes(small, dtype == "bf16")
    m = build_vasnet(VASNet, 57, {}, 5.0).cuda()
    xs, xb = features(small, 57, dtype), features(big, 58, dtype)
    for exact in (False, True):
        m._ws = _Workspace()
        torch.cuda.synchronize()
        a = m.score_packed(xs, small, check=False, exact=exact)
        b = m.score_packed(xb, big, check=False, exact=exact)
        torch.cuda.synchronize()
        m._ws = _Workspace()
        a1 = m.score_packed(xs, small, check=False, exact=exact)
        torch.cuda.synchronize()
        b1 = m.score_packed(xb, big, check=False, exact=exact)
        torch.cuda.synchronize()
        assert m.check_status()
        assert same_bits(a, a1) and same_bits(b, b1), f"exact={exact}"


KNOB_LENGTHS = [2000] * 20 + [3000, 1500, 777, 6000]


def _knob_scores(out_path):
    """Scores of the budget-knob batch on both paths and for both feature types (run in a child process)."""
    m = build_vasnet(VASNet, 59, {}, 5.0).cuda()
    out = {"plan": lib_plan(KNOB_LENGTHS)}
    for dtype in DTYPES:
        x = features(KNOB_LENGTHS, 59, dtype)
        out[f"{dtype} fast"] = fast_scores(m, x, KNOB_LENGTHS).cpu()
        out[f"{dtype} exact"] = m.score_packed(x, KNOB_LENGTHS, exact=True).cpu()
    torch.save(out, out_path)


@gpu
def test_logit_budget_knob_changes_only_the_grouping(tmp_path):
    """SMZ_VASNET_LOGIT_MELEMS=1 (read once per process) puts every video in a sub-chunk of its own; only the
    grouping of the per-video problems changes, so the scores are bit-identical to the default plan's."""
    default = VP.plan(KNOB_LENGTHS)
    one = VP.plan(KNOB_LENGTHS, budget=1 << 20)
    assert sum(len(c.subs) for c in default) < len(KNOB_LENGTHS) == sum(len(c.subs) for c in one)
    out = tmp_path / "knob.pt"
    env = dict(os.environ, SMZ_VASNET_LOGIT_MELEMS="1")
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]; "
            f"import test_vasnet_plan_gpu as t; t._knob_scores({str(out)!r})")
    r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    child = torch.load(out)
    assert child["plan"] == (len(one), len(KNOB_LENGTHS)), f"child plan {child['plan']}"
    m = build_vasnet(VASNet, 59, {}, 5.0).cuda()
    for dtype in DTYPES:
        x = features(KNOB_LENGTHS, 59, dtype)
        assert same_bits(fast_scores(m, x, KNOB_LENGTHS).cpu(), child[f"{dtype} fast"]), f"{dtype} fast path"
        assert same_bits(m.score_packed(x, KNOB_LENGTHS, exact=True).cpu(), child[f"{dtype} exact"]), f"{dtype} exact path"
