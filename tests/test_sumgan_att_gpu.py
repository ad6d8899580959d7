"""SumGAN-att selector inference on the sm_100a kernels (``smz_mha_forward`` at head width 256;
``Transformer.score_packed`` -> ``smz_sumgan_att_selector_forward``) against a float64 reference.

The selector (models/sumgan_att.py ``Transformer``) is ``sigmoid(out(layer_norm(TransformerEncoder(x))))`` with post-norm
``nn.TransformerEncoderLayer(d_model=1024, nhead=4, dim_feedforward=1024)`` layers: four heads of 256.  At width 256 the
attention kernel takes key tiles of 64 keys (128 at width 128), so the number of key tiles of a unit, and with it the
S-buffer and ring parity a CTA's next unit starts on, is ceil(T / 64).

CPU part: the float64 selector reference below (built on oracle/transformer_ref.py's generic ``encoder_layer``) is
pinned against ``copy.deepcopy(sel).double().eval()``; every attention batch is asserted to reach its intended schedule
at width 256; the ctypes mirror of ``smz_sumgan_att_selector_params`` matches gcc; unsupported head counts and widths are
refused before any device work.

GPU part.  Bars as in test_transformer_gpu.py: attention, worst element within 1e-2 of the head's largest |reference|
output; scores, worst-frame relative error 1e-2.  Measured on one NVIDIA B200 (1000 W power limit); attention error per
element (|got - ref| / max |ref| of the head) and score error per frame (relative), median / p95 / max:

  attention (4 heads of 256)   one video, T = 2 .. 8000          2.2e-4  8.0e-4  3.0e-3 .. 2.6e-4  9.2e-4  3.5e-3
                               (T = 1: exact, the output is V)
                               ragged, unaligned starts          3.1e-5  1.3e-4  2.8e-3
                               logits of several hundred         0       3.5e-5  2.8e-3
                               mixed (12 videos, 452 units)      1.7e-5  6.3e-5  1.3e-3
                               wide_table (300 videos)           4.7e-5  1.7e-4  2.7e-3
                               long (11 950 keys)                2.4e-4  7.9e-4  3.2e-3
                               n_heads = 1, wide strides         3.2e-5  1.3e-4  8.1e-4
                               n_heads = 2, wide strides         2.9e-5  1.2e-4  7.8e-4
  selector scores, bf16 / float32 features (max)
                               2 layers, 4 heads (default)       2.7e-4  8.4e-4  1.6e-3 / 1.7e-3
                               1 layer, 4 heads                  1.9e-4  5.8e-4  1.4e-3 / 1.2e-3
                               4 layers, 4 heads                 4.2e-4  1.2e-3  2.7e-3 / 2.0e-3
                               1 layer, 8 heads (width 128)      1.9e-4  6.0e-4  1.2e-3 / 1.0e-3
                               2 layers, 4 heads, eps 1e-3       2.7e-4  8.3e-4  1.6e-3 / 1.7e-3
                               chunk_boundary (37 131 rows)      2.6e-4  8.2e-4  2.3e-3 / 2.2e-3
                               long_video (33 000 frames)        1.9e-4  6.1e-4  1.7e-3 / 1.6e-3
  trainer, native against the torch modules in float32 (worst frame)                 2.4e-3

Width 256 lands in the same error range as width 128 (test_transformer_gpu.py, test_transformer_plan_gpu.py): the
error comes from bf16 P and bf16 output, not from the head width.
"""
import copy
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle import transformer_plan as TP
from oracle import transformer_ref as TR
from summarizer_b200 import _native as N
from summarizer_b200.models.sumgan_att import SelectorParams, Transformer
from test_transformer_gpu import cu_of, mha, packed_scores
from test_transformer_plan_gpu import MODEL, SMALL_UPLOAD, SM_COUNT, bf16_bits_equal, random_qkv, sm_count, stats, wide_lengths

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HD = 256
BKV = 64            # keys per tile at head width 256
DTYPES = (torch.bfloat16, torch.float32)


# ---- float64 reference and schedule (CPU) -------------------------------------------------------------------------
def selector_scores(sel, x, lengths):
    """Scores of a sumgan_att.Transformer selector for packed rows x [sum T, 1024] -> float64 [sum T] on x's device:
    the encoder layers, the encoder's final norm (the selector's ``layer_norm``), out[0] and sigmoid."""
    h = x.to(torch.float64)
    for L in sel.transformer_encoder.layers:
        h = TR.encoder_layer(L, h, lengths, sel.attention_heads)
    lin = sel.out[0]
    h = TR._layer_norm(h, sel.layer_norm)
    return torch.sigmoid(h @ lin.weight.detach().to(h).t() + lin.bias.detach().to(h)).reshape(-1)


def mha256_schedule(lengths, n_heads, sm_count):
    """oracle/transformer_plan.mha_schedule with the key-tile count of width 256 (the unit order does not depend on the
    key tile: units are 128-row query tiles)."""
    return [[u._replace(nk=(lengths[u.video] + BKV - 1) // BKV) for u in cta]
            for cta in TP.mha_schedule(lengths, n_heads, sm_count)]


CONFIGS = {
    "L2_H4": dict(encoder_layers=2, attention_heads=4),       # SumGANAtt's selector default
    "L1_H4": dict(encoder_layers=1, attention_heads=4),
    "L4_H4": dict(encoder_layers=4, attention_heads=4),
    "L1_H8": dict(encoder_layers=1, attention_heads=8),       # heads 128 wide
    "L2_H4_eps": dict(encoder_layers=2, attention_heads=4, epsilon=1e-3),
}


def make_selector(cfg, seed=0):
    torch.manual_seed(seed)
    return Transformer(**CONFIGS[cfg]).eval()


def features(lengths, seed, dtype, device="cpu"):
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(sum(lengths), 1024, generator=g, device=device).abs()      # non-negative, as pool5 features
    return x.to(dtype)


def torch_selector(sel, x):
    """The selector's torch modules (what forward ran before the native path existed)."""
    return sel.out(sel.transformer_encoder(x))


@pytest.mark.parametrize("cfg", ["L2_H4", "L1_H8", "L2_H4_eps"])
def test_selector_reference_matches_torch_module(cfg):
    """The float64 restatement equals copy.deepcopy(sel).double().eval() (torch's TransformerEncoder), video by video."""
    sel = make_selector(cfg)
    lengths = [5, 1, 37, 130]
    x = features(lengths, 9, torch.float32)
    ref = copy.deepcopy(sel).double().eval()
    with torch.no_grad():
        want = torch.cat([torch_selector(ref, xv.double().unsqueeze(1)).reshape(-1) for xv in torch.split(x, lengths)])
        got = selector_scores(sel, x, lengths)
    assert (got - want).abs().max().item() < 1e-12


# direct smz_mha_forward calls at width 256, 4 heads
ATTN = {
    # 376 units, 2-3 per CTA; nk = 187 is odd, so consecutive units start on the other S buffer and ring stage
    "long": [11950],
    # 452 units, 3-4 per CTA; consecutive units of a CTA change video and nk parity
    "mixed": [3001, 2500, 2001, 1800, 1500, 1100, 1000, 257, 256, 129, 65, 1],
    # a 4 800-byte table (cudaMemcpyAsync upload)
    "wide_table": wide_lengths(),
}


def assert_schedule(case, sm):
    lengths = ATTN[case]
    sched = mha256_schedule(lengths, 4, sm)
    units = [u for cta in sched for u in cta]
    assert len(units) == len(set(units)) == 4 * sum((T + 127) // 128 for T in lengths)
    assert min(len(cta) for cta in sched) >= 2, f"{case}: some CTA runs a single unit"
    pairs = [(a, b) for cta in sched for a, b in zip(cta, cta[1:])]
    odd_start = sum(sum(u.nk for u in cta[:i]) % 2 for cta in sched for i in range(len(cta)))
    parity = sum(a.nk % 2 != b.nk % 2 for a, b in pairs)
    video = sum(a.video != b.video for a, b in pairs)
    if case == "long":
        assert odd_start > 0, "no unit starts on S buffer 1"
    else:
        assert parity > 0 and video > 0, f"{case}: {parity} nk-parity and {video} video changes between units"
    if case == "wide_table":
        assert len(lengths) * TP.TABLE_ENTRY > SMALL_UPLOAD
    return len(units), max(len(cta) for cta in sched), parity, video


@pytest.mark.parametrize("case", list(ATTN))
def test_attention256_batch_reaches_its_schedule(case):
    units, per_cta, parity, video = assert_schedule(case, SM_COUNT)
    if case == "long":
        assert (units, per_cta) == (376, 3)
    if case == "mixed":
        assert units == 452


def test_selector_params_size_matches_header():
    src = ('#include <stdio.h>\n#include "summarizer_b200.h"\n'
           'int main(){printf("%zu\\n", sizeof(smz_sumgan_att_selector_params));return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", os.path.join(d, "s")])
        size = int(subprocess.check_output([os.path.join(d, "s")]))
    assert size == C.sizeof(SelectorParams)


def test_unsupported_heads_and_widths_are_refused_without_gpu():
    """n_heads other than 4 / 8 for the selector, head_dim other than 128 / 256 for attention: SMZ_ERR_UNSUPPORTED
    before any device work."""
    cu = cu_of([4])
    one = C.c_void_p(256)
    for nh in (2, 16):
        p = SelectorParams(256, nh, 256, 256, 1e-5, 256, 256)
        rc = N.lib().smz_sumgan_att_selector_forward(one, 0, cu.ctypes.data_as(C.c_void_p), 1, C.byref(p), 1, one, one,
                                                     1 << 30, None)
        assert rc == -3 and b"n_heads" in N.lib().smz_last_error()
    for hd in (64, 512):
        rc = N.lib().smz_mha_forward(one, 3 * 4 * hd, cu.ctypes.data_as(C.c_void_p), 1, 4, hd, one, 4 * hd, one, 1024, None)
        assert rc == -3 and b"head_dim" in N.lib().smz_last_error()


# ---- GPU: attention at width 256 ----------------------------------------------------------------------------------
def assert_attention256(qkv, lengths, n_heads=4, ldo=None):
    """smz_mha_forward (head_dim 256) on bf16 qkv against float64: in every head, the worst element within 1e-2 of that
    head's largest |reference| output.  Returns the output and the per-element errors."""
    w = n_heads * HD
    rc, out = mha(qkv, lengths, n_heads, head_dim=HD, ldo=ldo or w)
    assert rc == 0, N.lib().smz_last_error()
    want = TR.attention(qkv.double(), lengths, n_heads, head_dim=HD).view(-1, n_heads, HD)
    got = out[:, :w].double().view(-1, n_heads, HD)
    assert torch.isfinite(got).all()
    rel = (got - want).abs() / want.abs().amax(dim=(0, 2), keepdim=True)
    err = rel.amax(dim=(0, 2))
    assert (err < 1e-2).all(), f"worst element / max |reference| per head: {err.tolist()}"
    return out, rel


@gpu
@pytest.mark.parametrize("T", [1, 2, 63, 64, 65, 127, 128, 129, 700, 2000, 8000])
def test_mha256_single_video_matches_float64(T):
    """One video, 4 heads of 256, N(0,1) bf16 inputs.  T = 63 / 64 / 65 straddle a key tile, 127 / 128 / 129 a query
    tile; T = 8000 is 252 units, more than one per CTA.  Measured worst element / max |reference|: 2.9e-3 to 3.5e-3
    for T >= 2 (T = 1 is exact)."""
    _, err = assert_attention256(random_qkv([T], T, width=3 * 4 * HD), [T])
    print(f"T={T}: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
def test_mha256_ragged_batch_with_unaligned_starts():
    """Video starts at rows 0, 5, 305, 306, 435, 1212: none tile-aligned past the first; rows of the next video inside a
    key tile are masked."""
    lengths = [5, 300, 1, 129, 777, 64]
    _, err = assert_attention256(random_qkv(lengths, 40, width=3 * 4 * HD), lengths)
    print("ragged: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
def test_mha256_logits_of_several_hundred():
    """q and k scaled by 20: logits reach several hundred, where exp without a running max overflows."""
    lengths = [300, 400]
    qkv = random_qkv(lengths, 41, width=3 * 4 * HD).float()
    qkv[:, :2 * 4 * HD] *= 20.0
    qkv = qkv.bfloat16()
    q, k = qkv[:300, :HD].double(), qkv[:300, 4 * HD:5 * HD].double()
    assert (q @ k.t() / 16.0).abs().max().item() > 300
    _, err = assert_attention256(qkv, lengths)
    print("logits: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
@pytest.mark.parametrize("case", list(ATTN))
def test_mha256_batch_matches_float64(case):
    print(f"{case}: {sm_count()} SMs: units, most per CTA, parity / video changes {assert_schedule(case, sm_count())}")
    lengths = ATTN[case]
    _, err = assert_attention256(random_qkv(lengths, 42, width=3 * 4 * HD), lengths)
    print(f"{case}: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
@pytest.mark.parametrize("n_heads", [1, 2])
def test_mha256_head_count_and_strides(n_heads):
    """ld = 3 * n_heads * 256 + 64 (the 64 extra input columns are NaN and never read) and ldo = n_heads * 256 + 24:
    the 24 extra output columns keep their NaN sentinel; every head matches float64."""
    lengths = [300, 1, 129, 1000, 77, 256]
    w = n_heads * HD
    qkv = random_qkv(lengths, 43 + n_heads, width=3 * w + 64)
    qkv[:, 3 * w:] = float("nan")
    out, err = assert_attention256(qkv, lengths, n_heads, ldo=w + 24)
    assert torch.isnan(out[:, w:].float()).all(), "columns past n_heads * 256 were written"
    print(f"n_heads={n_heads}: attention error median %.2e p95 %.2e max %.2e" % stats(err))


@gpu
@pytest.mark.parametrize("case", ["mixed", "wide_table"])
def test_mha256_invariance(case):
    """Bit equality, per video: two calls; the batch in another video order; every other video's rows replaced by
    different finite values scaled by 50."""
    lengths = ATTN[case]
    cu = cu_of(lengths)
    qkv = random_qkv(lengths, 44, width=3 * 4 * HD)
    rc, out = mha(qkv, lengths, 4, head_dim=HD, ldo=4 * HD)
    assert rc == 0, N.lib().smz_last_error()
    assert bf16_bits_equal(mha(qkv, lengths, 4, head_dim=HD, ldo=4 * HD)[1], out), "a repeated call differs"
    perm = [int(v) for v in np.random.default_rng(6).permutation(len(lengths))]
    plen = [lengths[v] for v in perm]
    rc, pout = mha(torch.cat([qkv[cu[v]:cu[v + 1]] for v in perm]), plen, 4, head_dim=HD, ldo=4 * HD)
    assert rc == 0, N.lib().smz_last_error()
    pcu = cu_of(plen)
    for i, v in enumerate(perm):
        assert bf16_bits_equal(pout[pcu[i]:pcu[i + 1]], out[cu[v]:cu[v + 1]]), f"video {v} differs in the permuted batch"
    other = random_qkv(lengths, 45, width=3 * 4 * HD, scale=50.0)
    for v in range(0, len(lengths), max(1, len(lengths) // 12)):
        x = other.clone()
        x[cu[v]:cu[v + 1]] = qkv[cu[v]:cu[v + 1]]
        rc, iso = mha(x, lengths, 4, head_dim=HD, ldo=4 * HD)
        assert rc == 0, N.lib().smz_last_error()
        assert bf16_bits_equal(iso[cu[v]:cu[v + 1]], out[cu[v]:cu[v + 1]]), \
            f"video {v} ({lengths[v]} frames) changes when the other videos' rows change"


# ---- GPU: selector scores -----------------------------------------------------------------------------------------
def check_scores(sel, x, lengths, label):
    got = packed_scores(sel, x, lengths)
    with torch.no_grad():
        want = selector_scores(sel, x, lengths)
    rel = (got.double() - want).abs() / want.abs().clamp_min(1e-6)
    med, p95, mx = stats(rel)
    print(f"{label}: worst-frame rel err median {med:.2e} p95 {p95:.2e} max {mx:.2e}")
    assert mx <= 1e-2, mx


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_selector_scores_match_float64(cfg, dtype):
    """score_packed on a ragged batch (1 .. 700 frames, unaligned starts) against float64; every video bit-equal to
    itself scored alone and in the reversed batch.  Measured worst frame 1.0e-3 to 2.7e-3 (module docstring)."""
    sel = make_selector(cfg).cuda()
    lengths = [1, 64, 65, 129, 700]
    check_scores(sel, features(lengths, 3, dtype, "cuda"), lengths, f"{cfg} {dtype}")


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("case", ["chunk_boundary", "long_video"])
def test_selector_scores_across_chunks(case, dtype):
    """Two chunks, the second starting at the odd row 32 701 (2 layers); a 33 000-frame video alone in its chunk
    (1 layer).  Measured worst frame 1.6e-3 to 2.3e-3."""
    lengths = MODEL[case][0]
    assert [tuple(c) for c in TP.chunks(lengths)] == MODEL[case][1]
    sel = make_selector("L2_H4" if case == "chunk_boundary" else "L1_H4").cuda()
    check_scores(sel, features(lengths, 31, dtype, "cuda"), lengths, f"{case} {dtype}")


# ---- GPU: behaviour and routing -----------------------------------------------------------------------------------
@gpu
def test_sumgan_att_forward_batch_equals_score_packed():
    from summarizer_b200.models.sumgan_att import SumGANAtt
    torch.manual_seed(0)
    m = SumGANAtt().cuda().eval()
    x = torch.rand(200, 3, 1024, device="cuda")
    with torch.no_grad():
        y = m(x)
        s = m.summarizer.selector.score_packed(x.permute(1, 0, 2).reshape(-1, 1024), [200] * 3)
    assert y.shape == (200, 3, 1)
    assert torch.equal(y.permute(1, 0, 2).reshape(-1), s)


@gpu
def test_training_and_graph_forwards_run_the_torch_modules():
    sel = make_selector("L2_H4").cuda().train()
    x = torch.rand(50, 2, 1024, device="cuda")
    torch.manual_seed(5)
    y = sel(x)
    torch.manual_seed(5)
    assert torch.equal(y, torch_selector(sel, x))
    y.sum().backward()
    assert all(p.grad is not None for p in sel.transformer_encoder.layers[0].parameters())
    sel.eval()                                # eval with grad enabled still builds a graph: torch modules too
    y = sel(x)
    assert y.requires_grad and torch.equal(y, torch_selector(sel, x))


@gpu
def test_uncovered_head_count_keeps_torch_output():
    torch.manual_seed(0)
    sel = Transformer(encoder_layers=2, attention_heads=2).cuda().eval()
    assert not sel.native_covered()
    x = torch.rand(64, 2, 1024, device="cuda")
    with torch.no_grad():
        assert torch.equal(sel(x), torch_selector(sel, x))


@gpu
def test_scores_follow_load_state_dict():
    sel, other = make_selector("L2_H4", seed=0).cuda(), make_selector("L2_H4", seed=1).cuda()
    x = features([400], 7, torch.float32, "cuda")
    with torch.no_grad():
        before = sel.score_packed(x, [400])
        sel.load_state_dict(other.state_dict())
        after = sel.score_packed(x, [400])
        want = other.score_packed(x, [400])
    assert not torch.equal(before, after)
    assert torch.equal(after, want)


def make_trainer(tmp_path, **kw):
    from summarizer_b200.utils.config import HParameters
    hps = HParameters()
    hps.log_root = str(tmp_path)
    hps.tensorboard = False
    args = dict(model="sumgan_att", use_cuda="yes", splits_files="summe", log_level="error",
                extra_params={"pretrain_ae": 0})
    args.update(kw)
    hps.load_from_args(args)
    return hps.model_class(hps, hps.splits_files[0]).reset()


def torch_path_scores(trainer, keys):
    sel = trainer.model.summarizer.selector
    out = []
    with torch.no_grad():
        for k in keys:
            seq, _ = trainer._video_tensors(k)
            out.append(torch_selector(sel, seq).reshape(-1).float())
    return out


def rel_err(a, b):
    return ((a - b).abs() / b.abs().clamp_min(1e-6)).max().item()


@gpu
def test_scores_follow_train_step(tmp_path):
    """One train_step (the library's Adam updates the selector in place): the next eval scores use the new weights.
    The discriminator is 1024 wide: the library's recurrence implements hidden sizes 1024 and 2048."""
    t = make_trainer(tmp_path, epochs=1, extra_params={"pretrain_ae": 0, "cLSTM_hidden_size": 1024})
    train_keys, test_keys = t._get_train_test_keys(0)
    keys = test_keys[:3]
    t.model.eval()
    before = torch.cat(t._score_keys(keys)).cpu()
    t._make_optimizers()                      # what train() sets up before its first train_step
    t.loss_BCE = torch.nn.BCELoss()
    t.model.train()
    x, y = t._video_tensors(train_keys[0])
    t.train_step(x, y, epoch=100)
    t.model.eval()
    after = torch.cat(t._score_keys(keys)).cpu()
    ref = torch.cat(torch_path_scores(t, keys)).cpu()
    assert not torch.equal(after, before)
    assert rel_err(after, ref) <= 1e-2


@gpu
def test_trainer_test_and_predict_dataset(tmp_path):
    """SumGANAttTrainer scores all test videos in one packed native call, within 1e-2 of the torch modules' (float32)
    scores (measured 2.4e-3); test() and predict_dataset() run on it."""
    t = make_trainer(tmp_path, epochs=1)
    _, keys = t._get_train_test_keys(0)
    t.model.eval()
    native = torch.cat(t._score_keys(keys)).cpu()
    ref = torch.cat(torch_path_scores(t, keys)).cpu()
    print(f"trainer: worst-frame rel err {rel_err(native, ref):.2e}")
    assert rel_err(native, ref) <= 1e-2
    t.test(0)
    t.best_weights = t.model.state_dict()
    t.predict_dataset(str(tmp_path / "preds.h5"))
    assert (tmp_path / "preds.h5").exists()
