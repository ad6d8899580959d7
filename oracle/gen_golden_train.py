"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Golden TRAINING trajectories from the UNMODIFIED reference trainers (models/vasnet.py:171-238 VASNetTrainer.train,
models/dsn.py:60-183 DSNTrainer.train, models/sumgan.py:320-533 SumGANTrainer.pretrain / .train), run on the CPU in
float32 over a tiny synthetic dataset through the dict-backed h5py stand-in of oracle/ref_import.py.

Everything random the reference draws is pinned WITHOUT touching its code:
  * initial weights        torch.manual_seed(seed) right before Trainer.reset()
  * key order              random.seed(seed) right before Trainer.train()
  * VASNet dropout         the model's ``dropout`` attribute (an nn.Dropout INSTANCE) is replaced by a module that applies
                           keep-masks regenerated from seeds (``vasnet_keep_masks``), p = 0.5 scaling included
  * DSN episodes           ``Bernoulli`` in the dsn module's namespace is replaced by a subclass whose ``sample()`` thresholds
                           seeded uniforms; the sampled actions are STORED (the GPU run replays them: a probability that
                           differs in the 4th digit must not flip an episode)
  * SumGAN noise           ``torch.randn_like`` / ``torch.rand`` are wrapped for the duration of the run: draw number c comes
                           from ``noise_tensor(c, ...)``, a generator seeded with c, so the GPU test regenerates every tensor
What is stored (tests/golden/train_golden.npz): per-epoch training losses (per optimizer step when an epoch has one video),
the six SumGAN log terms, the VAE pre-training loss, DSN rewards, the (corr, avg F, max F) Trainer.test returns after
each epoch, train()'s return tuple, and initial / final values of sampled parameter entries (the Adam updates).

    python -m oracle.gen_golden_train          (needs SMZ_REFERENCE_ROOT, see oracle/ref_import.py)
"""
import contextlib
import logging
import os
import random
import re
import types

import numpy as np
import torch

from summarizer_b200 import synthetic

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "train_golden.npz")

# model -> tiny run.  frames: n_frames of video_1.. (n_steps = ceil(n_frames / 15)); the LAST video is the test key
RUNS = {
    "vasnet": dict(frames=[600, 750, 660], seed=11, epochs=3, lr=2e-4, extra={}),
    "dsn": dict(frames=[600, 750, 660], seed=12, epochs=3, lr=1e-3, extra={}),
    # one training video: every epoch is ONE optimizer step per phase, so the per-epoch log terms are per-step values;
    # epochs 0-1 add the discriminator noise (sumgan.py:465-468), epoch 2 does not; one VAE pre-training epoch
    "sumgan": dict(frames=[240, 300], seed=13, epochs=3, lr=1e-4, extra={"pretrain_vae": 1, "epoch_noise": 2}),
    "sumgan_sup": dict(frames=[240, 300], seed=14, epochs=1, lr=1e-4, extra={"pretrain_vae": 0, "epoch_noise": 0, "sup": True}),
}
WEIGHT_DECAY = 1e-5
MASK_SEED, NOISE_SEED, ACTION_SEED, SAMPLE_SEED = 51_000, 52_000, 53_000, 54_000
_RAND, _RANDN = torch.rand, torch.randn          # the real ones (seeded_noise() swaps the module attributes)


# ---- shared by the generator and the tests ---------------------------------------------------------------------------
def tiny_videos(frames):
    """{video_k: fields} — SumMe-shaped synthetic videos (summarizer_b200/synthetic.py), 3 annotators."""
    return {f"video_{i + 1}": synthetic.make_video("summe", 900 + i, n_frames=f, n_users=3) for i, f in enumerate(frames)}


def tiny_split(frames):
    keys = [f"video_{i + 1}" for i in range(len(frames))]
    return {"train_keys": keys[:-1], "test_keys": keys[-1:]}


def vasnet_keep_masks(step, T):
    """KEEP masks (uint8) of the three p=0.5 dropouts of optimizer step `step` (vasnet.py:130,136,142): attention
    (T, T), residual (T, 1024), hidden (T, 1024)."""
    g = torch.Generator().manual_seed(MASK_SEED + step)
    return tuple((_RAND(shape, generator=g) >= 0.5).to(torch.uint8) for shape in ((T, T), (T, 1024), (T, 1024)))


def noise_tensor(c, kind, shape):
    """Draw number `c` of a SumGAN run (kind "randn" or "rand")."""
    g = torch.Generator().manual_seed(NOISE_SEED + c)
    return _RANDN(shape, generator=g) if kind == "randn" else _RAND(shape, generator=g)


def sample_indices(name, numel, k=48):
    """Flat indices of the entries of parameter `name` whose initial / final values are stored."""
    rng = np.random.default_rng(SAMPLE_SEED + sum(name.encode()))
    return np.sort(rng.choice(numel, size=min(k, numel), replace=False))


def sampled_params(model):
    out = {}
    for name, p in model.state_dict().items():
        out[name] = p.detach().reshape(-1).cpu().numpy()[sample_indices(name, p.numel())].astype(np.float64)
    return out


# ---- reference-side plumbing ---------------------------------------------------------------------------------------------
class Recorder:
    """hps.writer stand-in: keeps every add_scalar (tag, value, step); histograms are dropped."""
    def __init__(self):
        self.scalars = {}

    def add_scalar(self, tag, value, step=None):
        self.scalars.setdefault(tag.split("/", 2)[-1], []).append(float(value))

    def add_histogram(self, *a, **k):
        pass


class LogCapture(logging.Handler):
    def __init__(self):
        super().__init__()
        self.lines = []

    def emit(self, record):
        self.lines.append(record.getMessage())


def reference_trainer(ns, cls, run, name):
    from oracle.ref_import import DictFile
    DictFile.registry[f"tiny_{name}"] = tiny_videos(run["frames"])
    log = logging.getLogger(f"golden_{name}")
    log.handlers, log.propagate = [], False
    cap = LogCapture()
    log.addHandler(cap)
    log.setLevel(logging.DEBUG)
    hps = types.SimpleNamespace(
        logger=log, dataset_of_file={"sf": f"tiny_{name}"}, dataset_name_of_file={"sf": "summe"},
        splits_of_file={"sf": [tiny_split(run["frames"])]}, use_cuda=False, cuda_device=0, lr=run["lr"],
        weight_decay=WEIGHT_DECAY, epochs=run["epochs"], test_every_epochs=1, extra_params=dict(run["extra"]),
        writer=Recorder(), summary_proportion=0.15, selection_algorithm="knapsack")
    torch.manual_seed(run["seed"])
    t = cls(hps, "sf").reset()
    return t, hps, cap


def pack(out, name, t, hps, ret, before):
    for tag, vals in hps.writer.scalars.items():
        out[f"{name}/{tag}"] = np.asarray(vals, dtype=np.float64)
    out[f"{name}/return"] = np.asarray(ret, dtype=np.float64)
    after = sampled_params(t.model)
    for k in before:
        out[f"{name}/w0/{k}"] = before[k]
        out[f"{name}/w1/{k}"] = after[k]


class MaskedDropout(torch.nn.Module):
    """Drop-in for the VASNet's nn.Dropout(0.5) instance: identical arithmetic (x * keep / (1 - p)), seeded keep-masks."""
    def __init__(self):
        super().__init__()
        self.step, self.site, self.masks = 0, 0, None

    def forward(self, x):
        if not self.training:
            return x
        if self.site == 0:
            self.masks = vasnet_keep_masks(self.step, x.shape[1])
        keep = self.masks[self.site].to(x.dtype).reshape(x.shape)
        self.site += 1
        if self.site == 3:
            self.site, self.step = 0, self.step + 1
        return x * keep * 2.0


def golden_vasnet(ns, out):
    run = RUNS["vasnet"]
    t, hps, _ = reference_trainer(ns, ns.vasnet.VASNetTrainer, run, "vasnet")
    t.model.dropout = MaskedDropout()
    before = sampled_params(t.model)
    random.seed(run["seed"])
    ret = t.train(0)
    pack(out, "vasnet", t, hps, ret, before)


def golden_dsn(ns, out):
    run = RUNS["dsn"]
    t, hps, _ = reference_trainer(ns, ns.dsn.DSNTrainer, run, "dsn")
    before = sampled_params(t.model)
    actions = []
    state = {"n": 0}
    real = ns.dsn.Bernoulli

    class SeededBernoulli(real):
        def sample(self, sample_shape=torch.Size()):
            g = torch.Generator().manual_seed(ACTION_SEED + state["n"])
            state["n"] += 1
            a = (_RAND(self.probs.shape, generator=g) < self.probs).to(self.probs.dtype)
            actions.append(a.reshape(-1).to(torch.uint8).numpy())
            return a

    ns.dsn.Bernoulli = SeededBernoulli
    try:
        random.seed(run["seed"])
        ret = t.train(0)
    finally:
        ns.dsn.Bernoulli = real
    pack(out, "dsn", t, hps, ret, before)
    out["dsn/actions"] = np.concatenate(actions)                 # episodes in call order, each n_steps of its video long
    out["dsn/action_lengths"] = np.asarray([len(a) for a in actions], dtype=np.int64)


@contextlib.contextmanager
def seeded_noise(counter):
    real_randn_like, real_rand = torch.randn_like, torch.rand

    def randn_like(x, **kw):
        c = counter["n"]
        counter["n"] += 1
        return noise_tensor(c, "randn", tuple(x.shape)).to(x.dtype)

    def rand(*shape, **kw):
        shape = tuple(shape[0]) if len(shape) == 1 and isinstance(shape[0], (tuple, list, torch.Size)) else tuple(shape)
        c = counter["n"]
        counter["n"] += 1
        return noise_tensor(c, "rand", shape)

    torch.randn_like, torch.rand = randn_like, rand
    try:
        yield
    finally:
        torch.randn_like, torch.rand = real_randn_like, real_rand


def golden_sumgan(ns, out, name):
    run = RUNS[name]
    t, hps, cap = reference_trainer(ns, ns.sumgan.SumGANTrainer, run, name)
    before = sampled_params(t.model)
    counter = {"n": 0}
    random.seed(run["seed"])
    with seeded_noise(counter):
        ret = t.train(0)
    pack(out, name, t, hps, ret, before)
    out[f"{name}/noise_draws"] = np.asarray([counter["n"]], dtype=np.int64)
    lvae = [float(m.group(1)) for line in cap.lines for m in [re.search(r"Lvae:\s*([-0-9.einfa]+)", line)] if m]
    out[f"{name}/Lvae"] = np.asarray(lvae, dtype=np.float64)     # logged with 5 decimals (sumgan.py:351)


def main(argv=None):
    """python -m oracle.gen_golden_train [model ...]: regenerates the named runs (default: all) and merges them into
    the existing file."""
    import sys
    from oracle import ref_import
    ns = ref_import.load()
    torch.set_num_threads(os.cpu_count() or 1)
    which = list(sys.argv[1:] if argv is None else argv) or list(RUNS)
    out = dict(np.load(GOLDEN)) if os.path.exists(GOLDEN) else {}
    for name in which:
        for k in [k for k in out if k.startswith(name + "/")]:
            del out[k]
        if name == "vasnet":
            golden_vasnet(ns, out)
        elif name == "dsn":
            golden_dsn(ns, out)
        else:
            golden_sumgan(ns, out, name)
        print(name, {k.split("/", 1)[1]: np.round(v, 5).tolist() for k, v in out.items()
                     if k.startswith(name + "/") and "/w" not in k and "actions" not in k})
    np.savez_compressed(GOLDEN, **out)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
