"""CPU: host-side logic of the drop-in surface — configuration, CLI parsing, fold scheduling, the `summarizer`
alias package, split fixtures, state-dict compatibility with the reference modules."""
import json
import os

import numpy as np
import pytest
import torch

from summarizer_b200.main import parse_extra, plan_folds
from summarizer_b200.utils import Proportion, parse_splits_filename
from summarizer_b200.utils.config import HParameters

PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "summarizer_b200")


def make_hps(tmp_path, **kw):
    hps = HParameters()
    hps.log_root = str(tmp_path)
    hps.tensorboard = False
    hps.allow_cpu = True
    args = dict(model="vasnet", use_cuda="no", splits_files="summe", log_level="error", extra_params={})
    args.update(kw)
    hps.load_from_args(args)
    return hps


def test_hparameters_defaults_and_shorthands(tmp_path):
    hps = make_hps(tmp_path)
    assert (hps.lr, hps.weight_decay, hps.epochs, hps.test_every_epochs) == (5e-5, 1e-5, 10, 2)
    assert hps.summary_proportion == 0.15 and hps.selection_algorithm == "knapsack"
    (sf,) = hps.splits_files
    assert sf.endswith("splits/summe_splits.json") and hps.dataset_name_of_file[sf] == "summe"
    assert "summe" in hps.dataset_of_file[sf] and len(hps.splits_of_file[sf]) == 5
    assert hps.weights_path[sf].endswith("summe_splits.json.pth") and hps.pred_path[sf].endswith("summe_splits.json_preds.h5")
    assert os.path.exists(os.path.join(hps.log_path, "train.log")) and os.path.exists(os.path.join(hps.log_path, "vasnet.py"))
    assert hps.model_class.__name__ == "VASNetTrainer"
    all_ = make_hps(tmp_path, splits_files="overfit")
    assert [os.path.basename(s) for s in all_.splits_files] == ["tvsum_splits_overfit.json", "summe_splits_overfit.json"]
    lst = make_hps(tmp_path, splits_files="splits/tvsum_splits.json,splits/summe_splits.json")   # documented superset
    assert len(lst.splits_files) == 2
    with pytest.raises(KeyError):
        make_hps(tmp_path, model="no_such_model")


def test_cli_extra_params_parsing():
    assert parse_extra(["--local", "12", "--ignore_self", "--scale", "0.06"]) == {"local": "12", "ignore_self": True, "scale": "0.06"}
    assert parse_extra([]) == {}
    assert 0.15 in Proportion() and 0 not in Proportion() and 1.5 not in Proportion()


def test_fold_scheduler_is_balanced_and_complete():
    costs = [(f, c) for f, c in enumerate([40, 10, 35, 12, 30, 11, 9, 41, 8, 10])]   # SumMe+TVSum-like: 10 jobs
    for world in (1, 2, 4, 8):
        plan = plan_folds(costs, world)
        assert sorted(j for r in plan for j in r) == list(range(10))
        loads = [sum(dict(costs)[j] for j in r) for r in plan]
        assert max(loads) <= sum(dict(costs).values()) / world + max(c for _, c in costs)
    assert plan_folds(costs, 3) == plan_folds(costs, 3)


def test_split_fixtures_shape():
    for name, n_train, n_test in (("summe", 20, 5), ("tvsum", 40, 10)):
        ds, splits = parse_splits_filename(os.path.join(PKG, "splits", f"{name}_splits.json"))
        assert ds == name and len(splits) == 5
        for s in splits:
            assert len(s["train_keys"]) == n_train and len(s["test_keys"]) == n_test
            assert not set(s["train_keys"]) & set(s["test_keys"])
        _, over = parse_splits_filename(os.path.join(PKG, "splits", f"{name}_splits_overfit.json"))
        assert len(over) == 1 and over[0]["train_keys"] == over[0]["test_keys"] and len(over[0]["train_keys"]) == 10


def test_summarizer_alias_package_serves_the_same_objects():
    import summarizer  # noqa: F401
    from summarizer.models.vasnet import VASNet as A
    from summarizer.utils.eval import generate_summary as g
    from summarizer_b200.models.vasnet import VASNet as B
    from summarizer_b200.utils.eval import generate_summary as h
    assert A is B and g is h
    from summarizer.main import train  # noqa: F401


def test_trainer_opens_synthetic_dataset_and_stages_keys(tmp_path):
    hps = make_hps(tmp_path, splits_files="summe")
    t = hps.model_class(hps, hps.splits_files[0])
    train_keys, test_keys = t._get_train_test_keys(0)
    assert len(train_keys) == 20 and len(test_keys) == 5
    d = t.dataset["video_1"]
    assert int(d["n_frames"][()]) == 4494 and d["features"][...].shape == (300, 1024)
    seq, target = t._video_tensors("video_1")
    assert seq.shape == (300, 1, 1024) and float(target.min()) == 0.0 and float(target.max()) == 1.0


def test_state_dict_matches_reference_modules():
    """The drop-in VASNet keeps the reference module's state-dict layout, so a reference .pth loads unchanged.  Against
    what the reference's own VASNet recorded: its key names and order and the initial values it drew at seeded entries
    of each tensor (the entries depend on the tensor's size; tests/golden/train_golden.npz), and the per-parameter
    checksums of the positional-embedding configurations (tests/golden/models_golden.npz).  With a reference checkout
    (oracle/ref_import.py) also live: key lists, shapes and loading a reference state dict."""
    from oracle import gen_golden_train as G
    from oracle import ref_import
    from oracle.gen_golden_models import VASNET_CASES, build_vasnet, checksums
    from summarizer_b200.models.vasnet import VASNet
    train = np.load(G.GOLDEN)
    prefix = "vasnet/w0/"
    names = [k[len(prefix):] for k in train.files if k.startswith(prefix)]      # stored in the reference's state_dict order
    torch.manual_seed(G.RUNS["vasnet"]["seed"])
    sampled = G.sampled_params(VASNet())
    assert list(sampled) == names
    for k in names:
        np.testing.assert_array_equal(sampled[k], train[prefix + k], err_msg=k)
    models = np.load(os.path.join(os.path.dirname(__file__), "golden", "models_golden.npz"))
    pos_cases = [c for c in VASNET_CASES if "pos_embed" in c[4]]
    assert pos_cases
    for name, seed, _, _, kw, sharpen in pos_cases:
        np.testing.assert_allclose(checksums(build_vasnet(VASNet, seed, kw, sharpen)), models[f"{name}/checksum"], rtol=1e-12)
    if not ref_import.available():
        return
    ref = ref_import.load()
    for kw in ({}, {"max_length": 32, "pos_embed": "simple"}):
        a, b = ref.vasnet.VASNet(**kw).state_dict(), VASNet(**kw).state_dict()
        assert list(a.keys()) == list(b.keys())
        assert all(a[k].shape == b[k].shape for k in a)
    m = VASNet()
    m.load_state_dict(ref.vasnet.VASNet().state_dict())   # a reference .pth loads unchanged


def test_host_pack_user_summary_matches_numpy():
    """smz_host_pack_user_summary (host threads, no GPU): bit j of word w of a row = (frame 32w+j > 0); NaN and
    negatives are 0; ragged row lengths and strides."""
    import ctypes
    from summarizer_b200 import _native as N
    shapes = [(100, 3), (4097, 2), (31, 1), (64, 4)]
    desc = np.zeros(len(shapes), dtype=N.VIDEO_DESC)
    rng = np.random.default_rng(0)
    rows, off = [], 0
    for i, (nf, nu) in enumerate(shapes):
        ld = (nf + 3) // 4 * 4
        desc[i]["n_frames"], desc[i]["n_users"], desc[i]["user_off"], desc[i]["user_ld"] = nf, nu, off, ld
        a = rng.standard_normal((nu, ld)).astype(np.float32)
        a[a < 0.3] = 0
        a[0, :5] = np.nan
        a[-1, -7:] = -1.0
        rows.append(a)
        off += nu * ld
    flat = np.concatenate([a.reshape(-1) for a in rows])
    words = ((desc["n_frames"].astype(np.int64) + 31) // 32) * desc["n_users"]
    boff = np.zeros(len(shapes), np.int64)
    boff[1:] = np.cumsum(words)[:-1]
    for n_threads in (1, 3, 16):
        out = np.full(int(words.sum()), 0xDEADBEEF, np.uint32)
        N.check(N.lib().smz_host_pack_user_summary(desc.ctypes.data_as(ctypes.c_void_p), len(shapes), flat.ctypes.data_as(ctypes.c_void_p),
                                                   boff.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p), n_threads))
        for i, a in enumerate(rows):
            nf = int(desc[i]["n_frames"]); W = (nf + 31) // 32
            for u in range(a.shape[0]):
                pad = np.zeros(W * 32, bool)
                with np.errstate(invalid="ignore"):
                    pad[:nf] = a[u, :nf] > 0
                ref = np.packbits(pad.reshape(W, 32), axis=1, bitorder="little").view(np.uint32).reshape(-1)
                assert (out[boff[i] + u * W: boff[i] + (u + 1) * W] == ref).all(), (n_threads, i, u)


def test_step_graphs_disabled_is_plain_eager():
    """StepGraphs with graphs off (CPU runs, --cuda_graphs no, data-parallel mode) just calls the step."""
    from summarizer_b200.models import StepGraphs
    calls = []
    g = StepGraphs(trainer=None, enabled=False)
    for key in ("a", "b", "a", "a"):
        assert g.run(key, lambda k: (calls.append(k) or (k,))) == (key,)
    assert calls == ["a", "b", "a", "a"] and g.graphs == {} and g.pool is None


def test_concurrent_fold_runner_schedules_reports_and_propagates_errors():
    """main._train_jobs_concurrently (--concurrent_folds K) with stand-in trainers on the CPU: every
    (split file, fold) job runs exactly once, heaviest first; the best fold per file is the highest correlation with the
    FIRST fold on ties (main.py:33-35) and carries a host copy of its weights; a failing fold surfaces as the caller's
    exception."""
    import logging
    import threading
    import time
    import types
    import torch
    from summarizer_b200 import main as M
    started, lock = [], threading.Lock()
    corr = {(0, 0): 0.2, (0, 1): 0.7, (0, 2): 0.7, (1, 0): 0.1, (1, 1): -0.3}

    class FakeTrainer:
        def __init__(self, hps, sf):
            self.sf, self.i = sf, hps.splits_files.index(sf)
            self.dataset = {f"v{k}": {"features": np.zeros((10 * (k + 1) * (self.i + 1), 4))} for k in range(3)}
            self.best_weights = None

        def reset(self):
            return self

        def train(self, fold):
            with lock:
                started.append((self.i, fold))
            if hps.fail_on == (self.i, fold):
                raise RuntimeError("fold blew up")
            time.sleep(0.01)
            self.best_weights = {"w": torch.full((2,), float(10 * self.i + fold))}
            return corr[(self.i, fold)], 0.5, 0.6

    hps = types.SimpleNamespace(splits_files=["a.json", "b.json"], epochs=2, use_cuda=False, fail_on=None,
                                logger=logging.getLogger("test"), model_class=FakeTrainer,
                                splits_of_file={"a.json": [{"train_keys": ["v0", "v1", "v2"]}, {"train_keys": ["v0"]}, {"train_keys": ["v1"]}],
                                                "b.json": [{"train_keys": ["v2"]}, {"train_keys": ["v0", "v2"]}]})
    models = {sf: FakeTrainer(hps, sf) for sf in hps.splits_files}
    jobs = [(0, 0), (0, 1), (0, 2), (1, 0), (1, 1)]
    res, best = M._train_jobs_concurrently(hps, models, jobs, 3, 0, 1)
    assert sorted(started) == jobs and set(res) == set(jobs)
    assert started[0] == (1, 1)                                   # heaviest job first: 2 epochs x (20 + 60) frames
    assert res[(0, 1)] == (0.7, 0.5, 0.6)
    assert best[0][:2] == (0.7, 1) and best[1][:2] == (0.1, 0)    # tie between folds 1 and 2 of file 0 -> the first
    assert torch.equal(best[0][2]["w"], torch.full((2,), 1.0)) and torch.equal(best[1][2]["w"], torch.full((2,), 10.0))
    hps.fail_on = (0, 2)
    with pytest.raises(RuntimeError, match="fold blew up"):
        M._train_jobs_concurrently(hps, models, jobs, 2, 0, 1)
