"""CPU tests of the oracle itself: it must agree with numpy, with the golden vectors generated
from the unmodified reference, with the reference imported live (given a checkout, see oracle/ref_import.py) and, for
the restated OR-tools solver, with brute force."""
import itertools
import os

import numpy as np
import pytest

from oracle import c_oracle, eval_np as E

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "eval_golden.npz")


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def test_pairwise_mean_matches_numpy_bitwise():
    rng = np.random.default_rng(1)
    for n in list(range(1, 200)) + [255, 256, 257, 300, 511, 1000, 1025, 4097, 30000]:
        a = rng.random(n).astype(np.float32)
        assert E.mean_f32(a).tobytes() == a.mean().tobytes(), n
        assert c_oracle.mean_f32(a).tobytes() == a.mean().tobytes(), n


def test_pairwise_mean_piecewise_constant():
    rng = np.random.default_rng(2)
    for _ in range(100):
        n = int(rng.integers(30, 301))
        a = np.repeat(rng.random(n // 15 + 2).astype(np.float32), 15)[int(rng.integers(0, 15)):][:n]
        assert E.mean_f32(a).tobytes() == a.mean().tobytes()


def test_oracle_matches_golden(golden):
    for name in golden["names"]:
        g = lambda k: golden[f"{name}/{k}"]
        nf = int(g("n_frames"))
        assert np.array_equal(E.upsample(g("scores"), nf, g("picks")), g("frame_scores"))
        seg = E.segment_scores(g("frame_scores"), g("cps"))
        for method in ("knapsack", "rank"):
            if method == "rank" and len(np.unique(seg)) < len(seg):
                # np.argsort (unstable, SIMD-dispatched quicksort) decides ties in the reference:
                # machine dependent, therefore unpinned (DESIGN.md); exactness only without ties
                continue
            s = E.generate_summary(g("scores"), g("cps"), nf, g("nfps").tolist(), g("picks"), 0.15, method)
            assert np.array_equal(s.astype(np.uint8), g(f"summary_{method}")), (name, method)
            sc, _ = c_oracle.generate_summary(g("scores"), g("cps"), nf, g("nfps"), g("picks"), 0.15, method)
            assert np.array_equal(sc.astype(np.uint8), g(f"summary_{method}")), (name, method)
            f = E.evaluate_summary(s, g("user_summary").astype(np.float32))
            assert np.float64(f[0]) == g(f"f_{method}")[0] and np.float64(f[1]) == g(f"f_{method}")[1]
            fc = c_oracle.evaluate_summary(s, g("user_summary").astype(np.float32))
            assert np.float64(fc["avg_f"]) == g(f"f_{method}")[0] and np.float64(fc["max_f"]) == g(f"f_{method}")[1]
        s = g("summary_knapsack").astype(np.float32)
        us = g("user_summary").astype(np.float32)
        for tag, m in (("long", np.concatenate([s, np.ones(7, np.float32)])), ("short", s[: nf - 11])):
            f = E.evaluate_summary(m, us)
            assert np.float64(f[0]) == g(f"f_{tag}")[0] and np.float64(f[1]) == g(f"f_{tag}")[1], (name, tag)


def _brute(p, w, c):
    best = 0
    for r in range(len(p) + 1):
        for comb in itertools.combinations(range(len(p)), r):
            if sum(w[i] for i in comb) <= c:
                best = max(best, sum(p[i] for i in comb))
    return best


def test_knapsack_restatement_optimal_and_consistent():
    rng = np.random.default_rng(3)
    zero_profit_picks = 0
    for _ in range(400):
        n = int(rng.integers(1, 11))
        w = rng.integers(1, 25, n)
        p = rng.integers(0, 8, n)
        c = int(rng.integers(0, 70))
        a = E.knapsack_dp_ortools(p, w, c)
        b = E.knapsack_dp_takebits(p, w, c)
        cc = c_oracle.knapsack(p, w, c)
        assert a == b == cc
        if w.sum() > c:
            assert sum(w[i] for i in a) <= c
            assert sum(p[i] for i in a) == _brute(p.tolist(), w.tolist(), c)
            zero_profit_picks += any(p[i] == 0 for i in a)
    assert zero_profit_picks > 0          # the item-0 default-id quirk is observable


def test_knapsack_all_fit_shortcut():
    assert E.knapsack_dp_takebits([0, 0, 5], [3, 4, 5], 12) == [0, 1, 2]
    assert c_oracle.knapsack([0, 0, 5], [3, 4, 5], 12) == [0, 1, 2]


def test_fscore_counts_exact():
    rng = np.random.default_rng(4)
    us = (rng.random((5, 1000)) < 0.2).astype(np.float32)
    m = (rng.random(1000) < 0.15).astype(np.float32)
    ov, ms, gs = E.overlap_counts(m, us)
    r = c_oracle.evaluate_summary(m, us)
    assert np.array_equal(ov, r["overlap"]) and np.array_equal(gs, r["gsum"]) and ms == r["msum"]
    assert np.array_equal(E.fscores_from_counts(ov, ms, gs), r["f"])


@pytest.mark.reference
def test_oracle_matches_live_reference():
    from oracle import ref_import
    from summarizer_b200 import synthetic
    R = ref_import.load().eval
    rng = np.random.default_rng(5)
    for i in range(12):
        v = synthetic.make_video("tvsum", 200 + i, n_frames=int(rng.integers(900, 6000)), n_users=4,
                                 uniform_segments=60 if i % 2 else None, with_features=False)
        scores = rng.random(int(v["n_steps"])).astype(np.float32)
        args = (scores, v["change_points"], int(v["n_frames"]), v["n_frame_per_seg"].tolist(), v["picks"])
        for method in ("knapsack", "rank"):
            ref = R.generate_summary(*args, 0.15, method)
            assert np.array_equal(ref, E.generate_summary(*args, 0.15, method))
            fr = R.evaluate_summary(ref, v["user_summary"])
            fo = E.evaluate_summary(ref, v["user_summary"])
            assert np.float64(fr[0]) == np.float64(fo[0]) and np.float64(fr[1]) == np.float64(fo[1])
