"""CPU: the torch restatement of the scorers (oracle/models_torch.py) reproduces the golden outputs of
the UNMODIFIED reference modules (tests/golden/models_golden.npz), and — when a checkout of the reference is
present (oracle/ref_import.py) — the live reference modules."""
import os

import numpy as np
import pytest
import torch

from oracle import models_torch as MT
from oracle.gen_golden_models import DSN_CASES, VASNET_CASES, build_dsn, build_vasnet, checksums, make_input
from summarizer_b200.models.vasnet import VASNet

GOLDEN = np.load(os.path.join(os.path.dirname(__file__), "golden", "models_golden.npz"))


@pytest.mark.parametrize("case", [c for c in VASNET_CASES if "max_length" not in c[4]], ids=lambda c: c[0])
def test_vasnet_restatement_matches_golden(case):
    name, seed, T, B, kw, sharpen = case
    m = build_vasnet(VASNet, seed, kw, sharpen)
    sd = m.state_dict()
    x = make_input(seed, T, B)
    with torch.no_grad():
        y = torch.stack([MT.vasnet_forward(sd, x[:, b], scale=m.scale, eps=m.epsilon, aperture=m.aperture,
                                           ignore_self=m.ignore_self) for b in range(B)], 1)
    np.testing.assert_allclose(y.numpy(), GOLDEN[f"{name}/y"][:, :, 0], rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize("case", DSN_CASES[:3], ids=lambda c: c[0])
def test_dsn_restatement_matches_golden(case):
    from summarizer_b200.models.dsn import DSN
    name, seed, T, B = case
    m = build_dsn(DSN, seed)
    # the drop-in module draws the reference's initial weights: the golden holds the reference's per-parameter checksums
    np.testing.assert_allclose(checksums(m), GOLDEN[f"{name}/checksum"], rtol=1e-12)
    sd = m.state_dict()
    x = make_input(seed, T, B)
    with torch.no_grad():
        y = torch.stack([MT.dsn_forward(sd, x[:, b]) for b in range(B)], 1)
    np.testing.assert_allclose(y.numpy(), GOLDEN[f"{name}/y"][:, :, 0], rtol=2e-5, atol=2e-6)


def test_dsn_reward_restatement_matches_live_reference():
    """oracle.models_torch.dsn_reward == the reference's DSNTrainer.compute_reward (dsn.py:185-236): over the episodes
    the reference trainer drew (stored actions), the per-epoch mean rewards it logged (tests/golden/train_golden.npz);
    with a reference checkout (oracle/ref_import.py) also live, on more lengths, far_sim and an empty selection."""
    import types
    from oracle import gen_golden_train as G
    from oracle import ref_import
    train = np.load(G.GOLDEN)
    videos = G.tiny_videos(G.RUNS["dsn"]["frames"]).values()
    feats = {int(v["n_steps"]): torch.from_numpy(np.asarray(v["features"], dtype=np.float32)) for v in videos}
    assert len(feats) == len(videos)                              # an episode's length names its video
    acts, lens = train["dsn/actions"], train["dsn/action_lengths"]
    offs = np.concatenate([[0], np.cumsum(lens)])
    got = [float(MT.dsn_reward(feats[int(n)], torch.from_numpy(acts[o:o + n].astype(np.float32)), far_sim=False,
                               temp_dist_thre=20)) for o, n in zip(offs, lens)]
    want = train["dsn/Train/Reward"]
    # every video runs the same number of episodes per epoch: the mean of the per-video means is the episodes' mean
    assert len(got) % len(want) == 0
    np.testing.assert_allclose(np.reshape(got, (len(want), -1)).mean(1), want, rtol=1e-5)
    if not ref_import.available():
        return
    ref = ref_import.load().dsn.DSNTrainer
    me = types.SimpleNamespace(hps=types.SimpleNamespace(use_cuda=False))
    g = torch.Generator().manual_seed(4)
    for T, p, far in [(60, 0.5, False), (200, 0.3, False), (150, 0.6, True), (80, 0.0, False)]:
        seq = make_input(70 + T, T, 1)
        actions = (torch.rand(T, 1, 1, generator=g) < p).float()
        want = float(ref.compute_reward(me, seq, actions, far_sim=far, temp_dist_thre=20))
        got = MT.dsn_reward(seq[:, 0], actions.reshape(-1), far_sim=far, temp_dist_thre=20)
        assert got == pytest.approx(want, rel=1e-5, abs=1e-7)
