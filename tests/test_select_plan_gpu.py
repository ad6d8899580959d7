"""Shot selection and evaluation (smz_select_shots, smz_eval_batch, smz_knapsack, smz_fscore) across the whole launch
plan of smz_select.cu, bit-exact against the C oracle (oracle/smz_oracle.c).

The plan is picked from the batch maxima: dp_kernel<K> for K in {2, 5, 9, 18, 27, 36, 54}, the 16-bit dp16_kernel<KW, MK>
in front of it (13 instantiations, handing videos back to dp_kernel through a fallback list), select_generic_kernel with
its take bits in shared memory or in the work buffer, four pooling routes (fused into dp16_kernel, pool_regular_kernel,
pool_smem_kernel, pool_kernel), the summary / F-score tail fused into the DP kernels or run stand-alone, and persistent
grids that shrink to whole rounds.  Each batch below holds one video that sets the plan and a few that ride along (an
all-zero-score video for the OR-tools item-0 quirk, a tie-heavy one, summaries longer and shorter than n_frames).

CPU part: oracle/select_plan.py restates the plan; every named batch is asserted to reach the structure it exists for at
148 SMs and 232 448 B of shared memory, and the batches together reach all 7 dp_kernel and all 13 dp16_kernel
instantiations.

GPU part, per batch: the work-buffer size equals the restatement (for one video, where occupancy drops out, and for the
batch); the kernels each call launches, with their grids and dynamic shared memory, are recorded with torch.profiler and
equal the restated list; and every output (seg_mean, values, picked, summary, mask, msum, overlap, gsum, f, avg_f,
max_f) equals the C oracle bit for bit, with status 0.  Outputs are filled with sentinels before every call and each
batch runs with two sets of scores, through select() and evaluate() (annotator rows as floats and as bits, the latter
with write_summary=False: the summary must keep its sentinel) for knapsack, and select() + fscore() for rank.

On an NVIDIA B200 (1000 W power limit) the GPU part runs in about 80 s, most of it in the host oracle: 28 s for the
benchmark's 10 000 videos, 16 s for the 70 000-video batch.  Before the stride-1 fix in pool_regular_video, every
segment mean of a stride-1 video that fits the staged scores read scores[0] (worst error 0.106, picks wrong); the
12 500-frame one beyond them took the cursor walk and was already right.
"""
import concurrent.futures as cf
import ctypes as C
import json
import os
import re
import tempfile
import threading

import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import select_plan as SP

gpu = pytest.mark.gpu
PROPORTION = 0.15
SWEEP_VIDEOS = 10000             # bench.py's --videos default; make_sweep_batch(seed=5000) as bench.py builds it
MANY_VIDEOS = 70000              # more than 65 535: the pooling and F-score kernels slice their grids


def capacity_of(n):
    return int(np.floor(n * PROPORTION))


# ---- batches (host only) ---------------------------------------------------------------------------------------------
def video(n_frames, seg=60, segs=None, stride=15, picks=None, n_users=2, nfps_delta=0, n_scores=None, kind="random",
          seed=0):
    """One video: segments of `seg` frames (or the given lengths), picks every `stride` frames (or the given ones),
    random 0/1 annotator rows.  kind: scores 'random', 'zero' (all-zero) or 'ties' (values in {0, 0.5, 1})."""
    rng = np.random.default_rng(seed)
    if segs is None:
        segs = [seg] * (n_frames // seg) + ([n_frames % seg] if n_frames % seg else [])
    segs = np.asarray(segs, np.int64)
    assert segs.sum() == n_frames
    ends = np.cumsum(segs)
    cps = np.stack([ends - segs, ends - 1], 1).astype(np.int32)
    nfps = segs.astype(np.int32)
    nfps[-1] += nfps_delta
    if picks is None:
        picks = np.arange(0, n_frames, stride)
    v = dict(n_frames=n_frames, picks=np.asarray(picks, np.int32), change_points=cps, n_frame_per_seg=nfps,
             user_summary=(rng.random((n_users, n_frames)) < 0.15).astype(np.float32), kind=kind)
    if n_scores is not None:
        v["n_scores"] = n_scores
    return v


def riders(seed):
    """Short videos that ride along with a batch's plan-setting video without changing its plan."""
    return [video(1000, kind="zero", seed=seed + 1),
            video(2000, seg=40, kind="ties", nfps_delta=-9, seed=seed + 2),
            video(1500, seg=50, nfps_delta=13, n_users=3, seed=seed + 3)]


def jittered_picks(n_frames, seed, last_at_end):
    rng = np.random.default_rng(seed)
    p = np.unique(np.clip(np.arange(0, n_frames, 15) + rng.integers(0, 9, (n_frames + 14) // 15), 0, n_frames - 1))
    p[0] = 0
    if last_at_end:
        p = np.append(p, n_frames)
    return p


# K edges: the largest n_frames with floor(0.15 n) + 1 <= K * 256
K_EDGE = {2: 3413, 5: 8533, 9: 15359, 18: 30719, 27: 46079, 36: 61439, 54: 92159}


def select_cases():
    """name -> (videos, expected structure).  Structure keys: k, dp16 (pair or None), bits_in_smem, pool (knapsack
    route), pool_rank, fused_tail."""
    c = {}
    c["k2_dp16_1_1"] = ([video(K_EDGE[2], seed=10), video(1500, stride=1, seed=11)] + riders(12)[:2],
                        dict(k=2, dp16=(1, 1), pool="fused", fused_tail=True))
    for K, n in K_EDGE.items():
        if K == 2:
            continue
        kw = (K + 1) // 2
        if K == 54:    # 300-frame segments leave room for ~11 000 staged scores: stride-1 videos inside and beyond
            main = [video(n, seg=300, seed=K), video(10000, stride=1, seed=K + 1), video(12500, stride=1, seed=K + 2)]
        else:
            main = [video(n, seed=K)]
        c[f"k{K}_dp16_{kw}_2"] = (main + riders(100 + K), dict(k=K, dp16=(kw, 2), pool="fused", fused_tail=True))
        long_seg = [600] + [60] * ((n - 600) // 60) + ([(n - 600) % 60] if (n - 600) % 60 else [])
        c[f"k{K}_dp16_{kw}_{kw}"] = ([video(n, segs=long_seg, seed=200 + K)] + riders(300 + K)[1:],
                                     dict(k=K, dp16=(kw, kw), pool="fused", fused_tail=True))
    c["segment_count_sets_k"] = ([video(3000, seg=2, seed=20), video(900, seg=3, kind="zero", seed=21)],
                                 dict(k=9, dp16=(5, 2), pool="regular", fused_tail=True))
    c["generic_bits_in_smem"] = ([video(100000, seg=2500, seed=30), video(5000, seg=125, kind="ties", seed=31),
                                  video(3000, kind="zero", nfps_delta=-9, seed=32)],
                                 dict(k=0, bits_in_smem=True))
    c["generic_bits_in_work_buffer"] = ([video(100000, seed=40), video(4000, kind="zero", nfps_delta=13, seed=41)],
                                        dict(k=0, bits_in_smem=False))
    heavy = [14000] + [60] * 1266 + [40]
    c["dp54_too_large_generic"] = ([video(90000, segs=heavy, seed=50), video(2000, kind="ties", seed=51)],
                                   dict(k=0, bits_in_smem=False, over_dp54=True))
    c["irregular_picks"] = ([video(K_EDGE[18], seed=60),
                             video(20000, picks=jittered_picks(20000, 61, False), seed=61),
                             video(12000, picks=jittered_picks(12000, 62, True), seed=62),
                             video(5000, n_scores=(5000 + 14) // 15 - 1, seed=63)],
                            dict(k=18, dp16=(9, 2), pool="fused", fused_tail=True))
    c["pool_smem"] = ([video(20000, seg=8, seed=70), video(3000, kind="ties", seed=71)],
                      dict(k=18, dp16=(9, 2), pool="smem", fused_tail=True))
    cursor = [23] * 2000 + [24] * 1000
    c["pool_cursor"] = ([video(70000, segs=cursor, seed=80), video(2500, kind="zero", seed=81)],
                        dict(k=54, dp16=(27, 2), pool="cursor", fused_tail=True))
    # 65 videos whose segment counts cover all 64 cost buckets of the dp queue's longest-first order
    c["order_buckets"] = ([video(5 * s, seg=5, n_users=1, seed=90 + s) for s in
                           sorted({max(1, -(-b * 641 // 64)) for b in range(64)} | {640})],
                          dict(k=5, dp16=(3, 2), pool="fused", fused_tail=True))
    return c


def maxima(videos):
    n_segs = [len(v["n_frame_per_seg"]) for v in videos]
    return dict(n_videos=len(videos), max_n_segs=max(n_segs), max_capacity=max(capacity_of(v["n_frames"]) for v in videos),
                max_n_frames=max(int(v["n_frames"]) for v in videos),
                max_seg_frames=max(int(np.max(v["n_frame_per_seg"])) for v in videos))


def restate(m, **kw):
    return SP.plan(m["n_videos"], m["max_n_segs"], m["max_capacity"], m["max_n_frames"], m["max_seg_frames"], **kw)


# knapsack over explicit values (smz_knapsack): per dp16 pair, the 16-bit pass and every condition of its hand-over
K_OF_KW = {1: 2, 3: 5, 5: 9, 9: 18, 14: 27, 18: 36, 27: 54}


def handover_items(kind, cap, wmax, rng):
    """(values, weights) of one video.  plain: the 16-bit DP runs to the end; overflow: a few light items worth 30 000
    make the top cell outgrow 16 bits part-way (the heavy zero-value items keep the 'hopeless' guess off); hopeless:
    the value density guess sends it to the 32-bit kernel up front; big: values above 32 767; negative values."""
    if kind == "overflow":
        light = 12
        m = -(-2 * 30000 * light * cap // (45000 * 250))
        w = np.concatenate([rng.integers(1, 4, light), rng.integers(200, 251, m)])
        p = np.concatenate([np.full(light, 30000), rng.integers(0, 6, m)])
        o = rng.permutation(len(w))
        return p[o], w[o]
    n = 150
    w = rng.integers(1, wmax + 1, n)
    if kind == "hopeless":
        return np.full(n, 30000), rng.integers(50, 251, n)
    p = rng.integers(0, 1001, n)
    if kind == "big":
        p[rng.integers(0, n, 5)] = 40000
    if kind == "negative":
        p = rng.integers(-500, 1001, n)
    return p, w


def handover_cases(seed=0):
    out = {}
    for kw, mk in SP.DP16_PAIRS:
        K = K_OF_KW[kw]
        cap = K * 256 - 8
        wmax = min(cap, kw * 256) if mk == kw and kw > 1 else (512 if kw > 1 else 256)
        rng = np.random.default_rng(1000 * kw + mk + seed)
        vids = [handover_items(kind, cap - 3 * i, wmax, rng) + (cap - 3 * i,)
                for i, kind in enumerate(("plain", "overflow", "hopeless", "big", "negative"))]
        if mk == kw and kw > 1:           # the MK = KW variant needs an item heavier than 512 (and not heavier than cap)
            p, w, cp = vids[0]
            w[0] = 600
            vids[0] = (p, w, cp)
        out[f"handover_{kw}_{mk}"] = vids
    return out


def knapsack_maxima(cases):
    return dict(n_videos=len(cases), max_n_segs=max(len(w) for _, w, _ in cases), max_capacity=max(c for _, _, c in cases),
                max_n_frames=0, max_seg_frames=max(int(np.max(w)) for _, w, _ in cases))


FALLBACK_VIDEOS = 2000


def fallback_cases(seed=0):
    rng = np.random.default_rng(77 + seed)
    return [handover_items("overflow", 4600, 250, rng) + (4600,) for _ in range(FALLBACK_VIDEOS)]


def sweep_maxima():
    """Batch maxima of make_sweep_batch(SWEEP_VIDEOS, seed=5000), from its host-side segment draw."""
    from summarizer_b200 import synthetic
    segs = [synthetic._segments(np.random.default_rng(5000 + i), 30000, 60 if i % 16 == 15 else None)[1]
            for i in range(SWEEP_VIDEOS)]
    return dict(n_videos=SWEEP_VIDEOS, max_n_segs=max(len(s) for s in segs), max_capacity=capacity_of(30000),
                max_n_frames=30000, max_seg_frames=max(int(s.max()) for s in segs))


def many_videos(n=MANY_VIDEOS):
    return [video(40, seg=20, n_users=1, seed=i % 7) for i in range(n)]


# ---- plan structure (CPU) --------------------------------------------------------------------------------------------
def test_k_edges_follow_capacity():
    for K, n in K_EDGE.items():
        assert SP.k_of_capacity(capacity_of(n)) == K and SP.k_of_capacity(capacity_of(n + 1)) != K, (K, n)
    assert SP.k_of_capacity(capacity_of(3414)) == 5
    assert SP.k_of_capacity(450, 1500) == 9


def check_structure(name, m, want, **kw):
    p = restate(m, **kw)
    assert p.k == want["k"], (name, p)
    if p.k == 0:
        assert p.bits_in_smem == want["bits_in_smem"], (name, p)
        if want.get("over_dp54"):      # K = 54 would cover the capacity, but its rows do not fit shared memory
            assert SP.k_of_capacity(m["max_capacity"], m["max_n_segs"]) == 54
            assert SP.dp_layout_total(54, m["max_n_segs"], p.pad_weight, 0) * 4 > kw.get("optin", SP.B200_OPTIN)
        return p
    assert (p.kw16, p.mk16) == want["dp16"], (name, p)
    assert (p.front_words > 0) == want["fused_tail"], (name, p)
    route, mi = SP.pooling(p, m["n_videos"], m["max_n_segs"], m["max_n_frames"], "knapsack", kw.get("optin", SP.B200_OPTIN))
    assert route == want["pool"], (name, route)
    if name == "segment_count_sets_k":     # too many segment lists for the fused route's staged scores: mi < 64
        wp = SP.dp16_layout(p.kw16, p.mk16, m["max_n_segs"], p.front_words)[0]
        assert wp - 4 * m["max_n_segs"] < 64
    return p


def test_cases_reach_their_structure_on_a_b200():
    ks, pairs = set(), set()
    for name, (vids, want) in select_cases().items():
        m = maxima(vids)
        p = check_structure(name, m, want)
        ks.add(p.k)
        if p.kw16:
            pairs.add((p.kw16, p.mk16))
        if name == "k54_dp16_27_2":    # stride-1 videos: one inside the staged scores, one beyond them
            mi = SP.pooling(p, m["n_videos"], m["max_n_segs"], m["max_n_frames"], "knapsack")[1]
            assert vids[1]["n_frames"] <= mi < vids[2]["n_frames"]
            assert SP.pooling(p, m["n_videos"], m["max_n_segs"], m["max_n_frames"], "rank")[0] == "regular"
        if name == "k2_dp16_1_1":
            mi = SP.pooling(p, m["n_videos"], m["max_n_segs"], m["max_n_frames"], "knapsack")[1]
            assert vids[1]["n_frames"] <= mi
        if name == "irregular_picks":
            assert vids[2]["picks"][-1] == vids[2]["n_frames"] and vids[1]["picks"][-1] < vids[1]["n_frames"]
            assert vids[3]["n_scores"] < len(vids[3]["picks"])
        if name == "order_buckets":
            M = m["max_n_segs"]
            buckets = {63 - min(max(len(v["n_frame_per_seg"]) * 64 // (M + 1), 0), 63) for v in vids}
            assert buckets == set(range(64))
    for name, cases in handover_cases().items():
        p = restate(knapsack_maxima(cases))
        assert name == f"handover_{p.kw16}_{p.mk16}" and p.k == K_OF_KW[p.kw16], (name, p)
        ks.add(p.k)
        pairs.add((p.kw16, p.mk16))
    assert ks == set(SP.DP_K) | {0}
    assert pairs == set(SP.DP16_PAIRS)
    # fallback list longer than the dp_kernel grid
    p = restate(knapsack_maxima(fallback_cases()))
    assert p.kw16 == 9 and p.grid < FALLBACK_VIDEOS
    # more than 65 535 videos: rank pools in two slices of pool_regular_kernel, fscore() slices fscore_kernel
    m = maxima(many_videos(4)) | dict(n_videos=MANY_VIDEOS)
    p = restate(m)
    names = [x.name for x in SP.launches(p, "select", MANY_VIDEOS, m["max_n_segs"], m["max_n_frames"], "rank")]
    assert names.count("pool_regular_kernel") == 2
    assert [x.name for x in SP.launches(p, "fscore", MANY_VIDEOS, 2, 40)].count("fscore_kernel") == 2


def test_bench_scale_plan_shrinks_the_dp16_grid():
    m = sweep_maxima()
    p = restate(m)
    assert p.k == 18 and (p.kw16, p.mk16) == (9, 2) and p.front_words > 0
    g16 = SP.B200_SMS * SP.occupancy_estimate("dp16_kernel<9,2>", p.smem16_bytes)
    assert p.grid16 < g16 < SWEEP_VIDEOS and -(-SWEEP_VIDEOS // p.grid16) > 1


# ---- device helpers --------------------------------------------------------------------------------------------------
def lib_workspace(m):
    from summarizer_b200 import _native as N
    b = C.c_int64(0)
    N.check(N.lib().smz_select_workspace_bytes(m["n_videos"], m["max_n_segs"], m["max_capacity"], m["max_n_frames"],
                                               m["max_seg_frames"], C.byref(b)))
    return b.value


def device_limits():
    pr = torch.cuda.get_device_properties(torch.cuda.current_device())
    return dict(optin=pr.shared_memory_per_block_optin, sm_count=pr.multi_processor_count)


_NAME = re.compile(r"(\w+)(<[^()]*>)?\(")


def kernel_name(s):
    m = _NAME.search(s)
    base = (m.group(1) + (m.group(2) or "")) if m else s.split("::")[-1]
    return base.replace(" ", "")


def record(fn):
    """Kernels launched by fn(): [(name, grid, shared memory)] in stream order.  Names from the profiler's events,
    grids and shared memory (static + dynamic) from its exported trace."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA
                 and not e.name.startswith(("Memset", "Memcpy", "[memset", "[memcpy"))), key=lambda e: e.time_range.start)
    names = [kernel_name(e.name) for e in ev]
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    ker = sorted((e for e in trace["traceEvents"] if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    assert names, "the profiler recorded no kernel events"
    assert [kernel_name(e["name"]) for e in ker] == names
    return [(n, tuple(e["args"]["grid"]), e["args"]["shared memory"]) for n, e in zip(names, ker)]


def check_launches(got, want, what):
    assert [g[0] for g in got] == [w.name for w in want], what
    for g, w in zip(got, want):
        assert g[1] == w.grid, (what, g, w)
        if w.smem is not None:                # reported: dynamic + static (a few hundred bytes at most)
            assert w.smem <= g[2] <= w.smem + 2048, (what, g, w)


def occupancy_from(got, m, sm_count, occ=None):
    """Resident CTAs per SM of the DP kernels as the recorded grids imply (only needed once a grid has more videos
    than resident CTAs): dp_kernel's grid is sm_count * per_sm; dp16_kernel's is the shrunk grid of some per_sm.
    occ: what earlier calls on the same batch implied (updated)."""
    n = m["n_videos"]
    occ = {} if occ is None else occ
    for name, grid, _ in got:
        if name.startswith("dp_kernel") and grid[0] < n:
            assert grid[0] % sm_count == 0, (name, grid)
            occ[name] = grid[0] // sm_count
        if name.startswith("dp16_kernel") and grid[0] < n:
            cands = [p for p in range(1, 33) if SP.shrink_grid(n, sm_count * p) == grid[0]]
            assert cands, (name, grid)
            occ[name] = cands[0]
    return lambda name, smem: occ.get(name, 1)


SENTINEL = dict(seg_mean=float("nan"), values=-123456, picked=0xAB, summary=-777.0, mask=0x5A5A5A5A, msum=-5, overlap=-5,
                gsum=-5, f=-5.0, avg_f=-5.0, max_f=-5.0, status=7)


def fill_sentinels(b):
    for k, x in SENTINEL.items():
        getattr(b, k).fill_(x)


def host_inputs(b):
    return dict(picks=b.d_picks.cpu().numpy(), cps=b.d_cps.cpu().numpy().reshape(-1, 2), nfps=b.d_nfps.cpu().numpy())


def users_chunk(b, v0, v1):
    """Annotator rows of videos [v0, v1) as host arrays, copied in one slice."""
    d = b.h_desc
    lo = int(d[v0]["user_off"])
    hi = int(d[v1 - 1]["user_off"]) + int(d[v1 - 1]["n_users"]) * int(d[v1 - 1]["user_ld"])
    h = b.d_users[lo:hi].cpu().numpy()
    out = []
    for v in range(v0, v1):
        o, nu, ld, nf = int(d[v]["user_off"]) - lo, int(d[v]["n_users"]), int(d[v]["user_ld"]), int(d[v]["n_frames"])
        out.append(h[o:o + nu * ld].reshape(nu, ld)[:, :nf] if nu else None)
    return out


def oracle_video(sc, picks, cps, nfps, n_frames, users, method):
    ref_sum, parts = c_oracle.generate_summary(sc, cps, n_frames, nfps, picks, PROPORTION, method)
    m = np.zeros((n_frames + 31) // 32 * 32, np.uint8)
    lim = min(n_frames, len(ref_sum))
    m[:lim] = ref_sum[:lim] > 0
    r = dict(seg_mean=parts["seg_score"], values=parts["values"].astype(np.int32), picks=parts["picks"],
             summary=ref_sum, mask=np.packbits(m, bitorder="little").view(np.uint32), msum=int(m.sum()))
    if users is not None:
        r["ev"] = c_oracle.evaluate_summary(ref_sum, users)
    return r


def compare(b, h, scores, method, fields, pool, memo, chunk=128):
    """Device outputs of b against the oracle, every video, bit for bit.  fields: which outputs the call wrote;
    'summary_sentinel' = the summary must still hold its sentinel.  memo: oracle results of these scores, by
    (method, video)."""
    d = b.h_desc
    out = {k: getattr(b, k).cpu().numpy() for k in ("seg_mean", "values", "picked", "summary", "mask", "msum", "overlap",
                                                    "gsum", "f", "avg_f", "max_f", "status")}
    assert not out["status"][: b.n_videos].any(), np.nonzero(out["status"][: b.n_videos])[0][:8]
    mask_u = out["mask"].view(np.uint32)
    for v0 in range(0, b.n_videos, chunk):
        v1 = min(v0 + chunk, b.n_videos)
        todo = [v for v in range(v0, v1) if (method, v) not in memo]
        users = users_chunk(b, v0, v1) if b.has_users and todo else [None] * (v1 - v0)

        def one(v):
            if (method, v) in memo:
                return memo[method, v]
            x = d[v]
            so, po, sg, ns = int(x["score_off"]), int(x["picks_off"]), int(x["seg_off"]), int(x["n_segs"])
            return oracle_video(scores[so:so + int(x["n_scores"])], h["picks"][po:po + int(x["n_picks"])],
                                h["cps"][sg:sg + ns], h["nfps"][sg:sg + ns], int(x["n_frames"]), users[v - v0], method)
        for v, r in zip(range(v0, v1), pool.map(one, range(v0, v1))):
            memo[method, v] = r
            x = d[v]
            sg, ns = int(x["seg_off"]), int(x["n_segs"])
            assert out["seg_mean"][sg:sg + ns].tobytes() == r["seg_mean"].tobytes(), (v, "seg_mean")
            assert np.array_equal(out["values"][sg:sg + ns], r["values"]), (v, "values")
            assert np.nonzero(out["picked"][sg:sg + ns])[0].tolist() == r["picks"], (v, "picked")
            assert not np.any(out["picked"][sg:sg + ns] > 1), (v, "picked")
            so, sl = int(x["summ_off"]), int(x["summ_len"])
            if "summary_sentinel" in fields:
                assert np.all(out["summary"][so:so + sl] == SENTINEL["summary"]), (v, "summary written")
            else:
                assert out["summary"][so:so + sl].tobytes() == r["summary"].tobytes(), (v, "summary")
            mo = int(x["mask_off"])
            assert np.array_equal(mask_u[mo:mo + len(r["mask"])], r["mask"]), (v, "mask")
            assert out["msum"][v] == r["msum"], (v, "msum")
            if "f" in fields:
                e, uo, nu = r["ev"], int(x["ucount_off"]), int(x["n_users"])
                assert np.array_equal(out["overlap"][uo:uo + nu], e["overlap"]), (v, "overlap")
                assert np.array_equal(out["gsum"][uo:uo + nu], e["gsum"]), (v, "gsum")
                assert out["f"][uo:uo + nu].tobytes() == e["f"].tobytes(), (v, "f")
                assert out["avg_f"][v] == e["avg_f"] and out["max_f"][v] == e["max_f"], (v, "avg_f / max_f")


def case_scores(vids, run):
    out = []
    for i, v in enumerate(vids):
        rng = np.random.default_rng(1000 * run + i)
        n = int(v.get("n_scores", len(v["picks"])))
        kind = v.get("kind", "random")
        s = np.zeros(n) if kind == "zero" else (rng.integers(0, 3, n) / 2.0 if kind == "ties" else rng.random(n))
        out.append(s.astype(np.float32))
    return np.concatenate(out)


@pytest.fixture(scope="module")
def pool():
    with cf.ThreadPoolExecutor(max_workers=min(os.cpu_count() or 1, 32)) as ex:
        yield ex


def run_batch(b, m, scores_fn, runs, pool, apis=("select", "evaluate", "evaluate_bits", "rank"), lim=None,
              occupancy=None):
    """Every API on batch b, `runs` times with different scores: launches against the restated plan on the first run,
    outputs against the oracle on every run."""
    lim = lim or device_limits()
    h = host_inputs(b)
    h_bits = b.pack_user_summary_host(b.d_users.cpu(), n_threads=8).cuda() if "evaluate_bits" in apis else None
    p = None
    occ = {}
    for run in range(runs):
        sc = scores_fn(run)
        d_sc = torch.from_numpy(sc).cuda() if isinstance(sc, np.ndarray) else sc
        h_sc = sc if isinstance(sc, np.ndarray) else sc.cpu().numpy()
        memo = {}
        for api in apis:
            method = "rank" if api == "rank" else "knapsack"
            fill_sentinels(b)
            if api == "select":
                call, fields = (lambda: b.select(d_sc)), ()
            elif api == "evaluate":
                call, fields = (lambda: b.evaluate(d_sc)), ("f",)
            elif api == "evaluate_bits":
                call, fields = (lambda: b.evaluate(d_sc, write_summary=False, d_bits=h_bits)), ("f", "summary_sentinel")
            else:
                call, fields = (lambda: (b.select(d_sc, method="rank"), b.fscore())), ("f",)
            if run == 0:
                got = record(call)
                p = restate(m, occupancy=occupancy or occupancy_from(got, m, lim["sm_count"], occ), **lim)
                assert lib_workspace(m) == p.workspace_bytes
                assert lib_workspace(dict(m, n_videos=1)) == restate(dict(m, n_videos=1), **lim).workspace_bytes
                want = SP.launches(p, "select" if api != "evaluate_bits" and api != "evaluate" else "evaluate",
                                   m["n_videos"], m["max_n_segs"], m["max_n_frames"], method,
                                   user_bits=api == "evaluate_bits", **lim)
                if api == "rank":
                    want += SP.launches(p, "fscore", m["n_videos"], m["max_n_segs"], m["max_n_frames"],
                                        sm_count=lim["sm_count"])
                check_launches(got, want, api)
            else:
                call()
            torch.cuda.synchronize()
            compare(b, h, h_sc, method, fields, pool, memo)
    return p


# ---- plan + results (GPU) --------------------------------------------------------------------------------------------
SELECT_CASES = select_cases()


@gpu
@pytest.mark.parametrize("name", list(SELECT_CASES))
def test_select_and_evaluate_match_oracle(name, pool):
    from summarizer_b200.batch import VideoBatch
    vids, want = SELECT_CASES[name]
    lim = device_limits()
    m = maxima(vids)
    check_structure(name, m, want, **lim)
    b = VideoBatch(vids, proportion=PROPORTION)
    run_batch(b, m, lambda run: case_scores(vids, run), 2, pool, lim=lim)


def knapsack_batch(cases):
    from summarizer_b200 import _native as N
    from summarizer_b200.batch import VideoBatch
    desc = np.zeros(len(cases), dtype=N.VIDEO_DESC)
    so = 0
    for i, (vals, w, cap) in enumerate(cases):
        desc[i]["seg_off"], desc[i]["n_segs"], desc[i]["capacity"], desc[i]["mask_off"] = so, len(w), cap, 0
        so += len(w)
    nfps = np.concatenate([np.asarray(c[1], np.int32) for c in cases])
    b = VideoBatch.from_packed(desc, np.zeros(1, np.int32), np.zeros(2, np.int32), nfps, None, PROPORTION)
    vals = torch.from_numpy(np.concatenate([np.asarray(c[0], np.int32) for c in cases])).cuda()
    return b, vals


def check_knapsack(cases, pool, lim, occupancy=None):
    b, vals = knapsack_batch(cases)
    m = knapsack_maxima(cases)
    b.picked.fill_(0xAB); b.status.fill_(7)
    got = record(lambda: b.knapsack(vals))
    occ = occupancy or occupancy_from(got, m, lim["sm_count"])
    p = restate(m, occupancy=occ, **lim)
    assert lib_workspace(m) == p.workspace_bytes
    check_launches(got, SP.launches(p, "knapsack", m["n_videos"], m["max_n_segs"], 0, **lim), "knapsack")
    picked, st = b.picked.cpu().numpy(), b.status.cpu().numpy()
    assert not st[: len(cases)].any()
    refs = list(pool.map(lambda c: c_oracle.knapsack(*c), cases))
    so = 0
    for i, ((vals_i, w, cap), ref) in enumerate(zip(cases, refs)):
        assert np.nonzero(picked[so:so + len(w)])[0].tolist() == ref, i
        so += len(w)
    return p, got


@gpu
@pytest.mark.parametrize("pair", SP.DP16_PAIRS, ids=[f"{a}_{b}" for a, b in SP.DP16_PAIRS])
def test_dp16_hand_over_every_instantiation(pair, pool):
    lim = device_limits()
    for seed in (0, 1):
        cases = handover_cases(seed)[f"handover_{pair[0]}_{pair[1]}"]
        p, _ = check_knapsack(cases, pool, lim)
        assert (p.kw16, p.mk16) == pair


@gpu
def test_fallback_list_longer_than_the_dp_kernel_grid(pool):
    lim = device_limits()
    p, got = check_knapsack(fallback_cases(), pool, lim)
    assert p.kw16 == 9 and p.grid < FALLBACK_VIDEOS and [g for g in got if g[0] == "dp_kernel<18>"][0][1][0] == p.grid


@gpu
def test_more_than_65535_videos(pool):
    from summarizer_b200.batch import VideoBatch
    vids = many_videos()
    lim = device_limits()
    m = maxima(vids)
    b = VideoBatch(vids, proportion=PROPORTION)
    p = run_batch(b, m, lambda run: case_scores(vids, run), 1, pool, apis=("evaluate", "rank"), lim=lim)
    assert p.kw16 and SP.pooling(p, MANY_VIDEOS, m["max_n_segs"], m["max_n_frames"], "rank")[0] == "regular"


@gpu
def test_bench_scale_evaluate(pool):
    """evaluate() on the benchmark's batch (make_sweep_batch(10 000, seed=5000)): a shrunk multi-round dp16 grid,
    annotator rows at offsets above 2^31 elements, every video against the oracle."""
    from summarizer_b200 import synthetic
    lim = device_limits()
    b = synthetic.make_sweep_batch(SWEEP_VIDEOS, "cuda", seed=5000)
    try:
        assert int(b.h_desc[-1]["user_off"]) > 2 ** 31
        m = dict(n_videos=b.n_videos, max_n_segs=b.max_n_segs, max_capacity=b.max_capacity, max_n_frames=b.max_n_frames,
                 max_seg_frames=b.max_seg_frames)

        def scores(run):
            g = torch.Generator(device="cuda")
            g.manual_seed(run)
            return torch.rand(b.total_scores, generator=g, device="cuda")
        p = run_batch(b, m, scores, 1, pool, apis=("evaluate",), lim=lim)
        g16 = p.grid16
        per_sm16 = occupancy_from([(p.dp16_name(), (g16, 1, 1), 0)], m, lim["sm_count"])(p.dp16_name(), 0)
        assert p.kw16 and -(-SWEEP_VIDEOS // g16) > 1             # several rounds per CTA
        assert g16 < lim["sm_count"] * per_sm16                     # shrunk to whole rounds
    finally:
        del b
        torch.cuda.empty_cache()


@gpu
def test_select_from_four_threads_equals_one_thread():
    """One run of select() from 4 host threads on their own streams, batches with different maxima (so different
    plans and shared-memory sizes are planned at the same time), against the same calls made one after another."""
    from summarizer_b200.batch import VideoBatch
    names = ["k2_dp16_1_1", "k18_dp16_9_9", "generic_bits_in_smem", "pool_smem"]
    batches = [VideoBatch(SELECT_CASES[n][0], proportion=PROPORTION) for n in names]
    scores = [torch.from_numpy(case_scores(SELECT_CASES[n][0], 0)).cuda() for n in names]
    keys = ("seg_mean", "values", "picked", "summary", "mask", "msum")
    start = threading.Barrier(len(names))
    errors = []

    def work(i):
        try:
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                start.wait()
                batches[i].select(scores[i])
            s.synchronize()
        except Exception as e:          # noqa: BLE001 — reported below
            errors.append(e)
    for b in batches:
        fill_sentinels(b)
    torch.cuda.synchronize()
    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(names))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    got = [{k: getattr(b, k).cpu().numpy().tobytes() for k in keys} for b in batches]
    for b, sc, g in zip(batches, scores, got):
        fill_sentinels(b)
        b.select(sc)
        torch.cuda.synchronize()
        assert not b.status[: b.n_videos].any()
        for k in keys:
            assert getattr(b, k).cpu().numpy().tobytes() == g[k], k
