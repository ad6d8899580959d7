"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Generates the committed golden fixtures under tests/golden/ by running the UNMODIFIED reference
(imported from $SMZ_REFERENCE_ROOT through oracle/ref_import.py) on seeded synthetic inputs.
With a reference checkout:   SMZ_REFERENCE_ROOT=<checkout> python -m oracle.gen_golden

  tests/golden/eval_golden.npz     inputs + reference outputs of generate_summary (knapsack via the
                                   restated OR-tools solver, and 'rank'), upsample, evaluate_summary
  tests/golden/models_golden.npz   VASNet / DSN reference forward outputs for seeded weights+inputs
                                   (weights are regenerated from the seed by the tests)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import  # noqa: E402
from summarizer_b200 import synthetic  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def eval_cases():
    """(name, video dict, scores) — small, ragged, tie-heavy and edge cases."""
    cases = []
    rng = np.random.default_rng(42)
    for i, (nf, uni) in enumerate([(950, None), (1499, None), (2100, 60), (4494, None), (3001, 45),
                                   (7777, None), (640, 30), (9721, 60)]):
        v = synthetic.make_video("summe", 100 + i, n_frames=nf, n_users=3 + i % 4, uniform_segments=uni,
                                 with_features=False)
        n_steps = int(v["n_steps"])
        if i % 3 == 0:
            scores = rng.random(n_steps).astype(np.float32)
        elif i % 3 == 1:   # quantised scores -> many equal segment values
            scores = (rng.integers(0, 4, n_steps) / 4.0).astype(np.float32)
        else:              # sigmoid-like, concentrated
            scores = (1 / (1 + np.exp(-rng.standard_normal(n_steps)))).astype(np.float32)
        cases.append((f"case{i}", v, scores))
    return cases


def gen_eval(ns):
    R = ns.eval
    out = {}
    names = []
    for name, v, scores in eval_cases():
        names.append(name)
        nf = int(v["n_frames"])
        args = (scores, v["change_points"], nf, v["n_frame_per_seg"].tolist(), v["picks"])
        out[f"{name}/scores"] = scores
        out[f"{name}/n_frames"] = np.int64(nf)
        out[f"{name}/picks"] = v["picks"]
        out[f"{name}/cps"] = v["change_points"]
        out[f"{name}/nfps"] = v["n_frame_per_seg"]
        out[f"{name}/user_summary"] = v["user_summary"].astype(np.uint8)
        out[f"{name}/frame_scores"] = R.upsample(scores, nf, v["picks"])
        for method in ("knapsack", "rank"):
            s = R.generate_summary(*args, 0.15, method)
            out[f"{name}/summary_{method}"] = s.astype(np.uint8)
            avg_f, max_f = R.evaluate_summary(s, v["user_summary"])
            out[f"{name}/f_{method}"] = np.asarray([avg_f, max_f], dtype=np.float64)
        # truncated / padded machine summaries (utils/eval.py:141-145)
        s = out[f"{name}/summary_knapsack"].astype(np.float32)
        for tag, m in (("long", np.concatenate([s, np.ones(7, np.float32)])), ("short", s[: nf - 11])):
            avg_f, max_f = R.evaluate_summary(m, v["user_summary"])
            out[f"{name}/f_{tag}"] = np.asarray([avg_f, max_f], dtype=np.float64)
    out["names"] = np.asarray(names)
    # correlation.ipynb cells 24-26 known answers
    x = np.array([0.9, 0.3, 0.7]); y = np.array([[0.4, 0.8, 1.0]])
    out["kat/spearman"] = np.float64(R.evaluate_scores(x, y, "spearmanr"))
    out["kat/kendall"] = np.float64(R.evaluate_scores(x, y, "kendalltau"))
    np.savez_compressed(os.path.join(GOLDEN, "eval_golden.npz"), **out)
    print("eval_golden.npz:", len(names), "cases; KAT", out["kat/spearman"], out["kat/kendall"])


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    ns = ref_import.load()
    gen_eval(ns)
    if "--models" in sys.argv or True:
        try:
            from oracle import gen_golden_models
            gen_golden_models.generate(ns, GOLDEN)
        except ImportError:
            pass


if __name__ == "__main__":
    main()
