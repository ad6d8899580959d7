"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Plain float32 PyTorch restatement of the reference scorers' forward passes, written against a state
dict with the reference's key names so it can be fed with the product modules' parameters:

  vasnet_forward   models/vasnet.py:92-148 (eval mode, or training mode with explicit keep-masks)
                   (vasnet_forward_packed: the same over a packed batch, video by video)
  dsn_forward      models/dsn.py:38-47     (nn.LSTM semantics restated step by step: gates i,f,g,o)

Pinned by tests/test_oracle_models.py against tests/golden/models_golden.npz, i.e. against outputs of the
UNMODIFIED reference modules.  Used by the GPU parity tests (gradients through autograd), by
__graft_entry__.smoke() and as bench.py's timed CPU baseline for the scoring stage.
"""
import math

import torch
import torch.nn.functional as F


def vasnet_forward(sd, x, scale=None, eps=1e-6, aperture=None, ignore_self=False, keep_att=None, keep_y=None,
                   keep_h=None):
    """x: (T, 1024) float32 of ONE video -> scores (T,).  keep_*: optional 0/1 masks of the three
    p=0.5 dropouts (vasnet.py:130,136,142): kept entries are scaled by 2."""
    T, D = x.shape
    scale = 1.0 / math.sqrt(D) if scale is None else scale
    K = x @ sd["K.weight"].t()                                   # vasnet.py:114
    Q = x @ sd["Q.weight"].t()                                   # :115
    V = x @ sd["V.weight"].t()                                   # :116
    e = (Q @ K.t()) * scale                                      # :118-119
    if ignore_self:                                              # :121-122
        e = e.masked_fill(torch.eye(T, dtype=torch.bool, device=x.device), float("-inf"))
    if aperture is not None:                                     # :124-127 (incl. the e*e == 0 quirk)
        scope = torch.tril(e, diagonal=aperture) * torch.triu(e, diagonal=-aperture)
        e = e.masked_fill(scope == 0, float("-inf"))
    alpha = torch.softmax(e, dim=1)                              # :129
    if keep_att is not None:
        alpha = alpha * keep_att * 2.0                           # :130
    c = (alpha @ V) @ sd["attention_head_projection.weight"].t()  # :131-132
    y = c + x                                                    # :135
    if keep_y is not None:
        y = y * keep_y * 2.0                                     # :136
    y = F.layer_norm(y, (D,), sd["layer_norm.weight"], sd["layer_norm.bias"], eps)       # :137
    y = torch.relu(y @ sd["k1.weight"].t() + sd["k1.bias"])      # :140-141
    if keep_h is not None:
        y = y * keep_h * 2.0                                     # :142
    y = F.layer_norm(y, (D,), sd["layer_norm.weight"], sd["layer_norm.bias"], eps)       # :143
    return torch.sigmoid(y @ sd["k2.weight"].t() + sd["k2.bias"]).reshape(T)             # :144-145


def vasnet_forward_packed(sd, x, lengths, **kw):
    """vasnet_forward over a packed batch x (sum T, 1024), one video at a time, in the dtype and on the device of x
    (float64 on the GPU for the parity tests of the packed scorer) -> scores (sum T,)."""
    sd = {k: v.to(x) for k, v in sd.items()}
    return torch.cat([vasnet_forward(sd, xv, **kw) for xv in torch.split(x, list(lengths))])


def lstm_direction(x, w_ih, w_hh, b_ih, b_hh, reverse=False):
    """One direction of torch.nn.LSTM (zero initial state): x (T, I) -> h (T, H).
    Gate order i, f, g, o; c_t = f*c + i*g; h_t = o*tanh(c_t)."""
    T = x.shape[0]
    H = w_hh.shape[1]
    pre = x @ w_ih.t() + b_ih + b_hh
    h = x.new_zeros(H)
    c = x.new_zeros(H)
    out = [None] * T
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        g = pre[t] + w_hh @ h
        i, f, gg, o = g[:H], g[H:2 * H], g[2 * H:3 * H], g[3 * H:]
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
        h = torch.sigmoid(o) * torch.tanh(c)
        out[t] = h
    return torch.stack(out, 0)


def dsn_forward(sd, x):
    """x: (T, 1024) of ONE video -> probs (T,)   (dsn.py:38-47: BiLSTM(1024->256) + Linear(512,1) + sigmoid)."""
    hf = lstm_direction(x, sd["rnn.weight_ih_l0"], sd["rnn.weight_hh_l0"], sd["rnn.bias_ih_l0"], sd["rnn.bias_hh_l0"])
    hb = lstm_direction(x, sd["rnn.weight_ih_l0_reverse"], sd["rnn.weight_hh_l0_reverse"],
                        sd["rnn.bias_ih_l0_reverse"], sd["rnn.bias_hh_l0_reverse"], reverse=True)
    h = torch.cat([hf, hb], 1)
    return torch.sigmoid(h @ sd["out.0.weight"].t() + sd["out.0.bias"]).reshape(-1)


def dsn_reward(seq, actions, far_sim=False, temp_dist_thre=20):
    """models/dsn.py:185-236 compute_reward for ONE episode: seq (T, 1024) float32, actions (T,) 0/1 ->
    0.5 * (R_div + R_rep) as a python float.  No frame picked -> 0 (dsn.py:199-203); a single picked frame:
    R_div = 0 (dsn.py:207-210) and R_rep over that one column (the reference raises on the 0-d index there)."""
    pick = torch.nonzero(actions.reshape(-1) > 0).reshape(-1)
    P = int(pick.numel())
    if P == 0:
        return 0.0
    T = seq.shape[0]
    if P == 1:
        reward_div = torch.tensor(0.)
    else:
        normed = seq / seq.norm(p=2, dim=1, keepdim=True)                      # :214
        dissim = 1. - normed @ normed.t()                                      # :215
        sub = dissim[pick][:, pick]                                            # :216
        if not far_sim:
            td = (pick[None, :] - pick[:, None]).abs()                         # :219-221
            sub = torch.where(td > temp_dist_thre, torch.ones_like(sub), sub)  # :222
        reward_div = sub.sum() / (P * (P - 1.))                                # :223
    sq = seq.pow(2).sum(dim=1, keepdim=True).expand(T, T)                      # :226
    dist = sq + sq.t() - 2 * (seq @ seq.t())                                   # :227-228
    reward_rep = torch.exp(-dist[:, pick].min(1)[0].mean())                    # :229-231
    return float((reward_div + reward_rep) * 0.5)


# ---- SumGAN (models/sumgan.py:23-258) -----------------------------------------------------------------------
def lstm_layer(x, w_ih, w_hh, b_ih, b_hh, h0=None, c0=None, reverse=False):
    """One direction of one torch.nn.LSTM layer with an initial state: x (T, I) -> (y (T, H), h_n (H), c_n (H))."""
    T, H = x.shape[0], w_hh.shape[1]
    pre = x @ w_ih.t() + b_ih + b_hh
    h = x.new_zeros(H) if h0 is None else h0
    c = x.new_zeros(H) if c0 is None else c0
    out = [None] * T
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        g = pre[t] + w_hh @ h
        i, f, gg, o = g[:H], g[H:2 * H], g[2 * H:3 * H], g[3 * H:]
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
        h = torch.sigmoid(o) * torch.tanh(c)
        out[t] = h
    return torch.stack(out, 0), h, c


def lstm_stack(sd, prefix, x, num_layers=2, bidirectional=False, h0=None, c0=None):
    """torch.nn.LSTM (batch 1) from the state-dict entries ``prefix + weight_ih_l0`` ...: x (T, I) ->
    (y (T, nd*H), h_n (L*nd, H), c_n (L*nd, H)) in nn.LSTM's layer-major, direction-minor order."""
    nd = 2 if bidirectional else 1
    hs, cs = [], []
    for layer in range(num_layers):
        ys = []
        for d in range(nd):
            sfx = f"_l{layer}" + ("_reverse" if d else "")
            k = layer * nd + d
            y, h, c = lstm_layer(x, sd[prefix + "weight_ih" + sfx], sd[prefix + "weight_hh" + sfx], sd[prefix + "bias_ih" + sfx],
                                 sd[prefix + "bias_hh" + sfx], None if h0 is None else h0[k], None if c0 is None else c0[k], bool(d))
            ys.append(y); hs.append(h); cs.append(c)
        x = torch.cat(ys, 1)
    return x, torch.stack(hs, 0), torch.stack(cs, 0)


def sumgan_slstm(sd, x, prefix="summarizer.s_lstm."):
    """sLSTM.forward (sumgan.py:36-46), batch 1: x (T, 1024) -> scores (T,)."""
    y, _, _ = lstm_stack(sd, prefix + "lstm.", x, 2, True)
    return torch.sigmoid(y @ sd[prefix + "out.weight"].t() + sd[prefix + "out.bias"]).reshape(-1)


def sumgan_elstm(sd, x, prefix="summarizer.vae.e_lstm."):
    """eLSTM.forward (sumgan.py:61-72), batch 1: -> (mu (2, H), logvar (2, H), c_last (2, H))."""
    _, h, c = lstm_stack(sd, prefix + "lstm.", x, 2, False)
    return h @ sd[prefix + "mu.weight"].t() + sd[prefix + "mu.bias"], h @ sd[prefix + "logvar.weight"].t() + sd[prefix + "logvar.bias"], c


def sumgan_dlstm(sd, T, h, c, prefix="summarizer.vae.d_lstm."):
    """dLSTM.forward (sumgan.py:98-115), batch 1: one-step 2-layer LSTM calls fed with their own output, the
    reconstruction of every step, time-reversed: -> x_hat (T, 1024)."""
    x = h.new_zeros(1, h.shape[1])
    outs = []
    for _ in range(T):
        x, h, c = lstm_stack(sd, prefix + "lstm.", x, 2, False, h, c)
        outs.append(x @ sd[prefix + "recons.weight"].t() + sd[prefix + "recons.bias"])
    return torch.flip(torch.cat(outs, 0), (0,))


def sumgan_clstm(sd, x, prefix="gan.c_lstm."):
    """cLSTM.forward (sumgan.py:199-210), batch 1: -> (prob scalar tensor (1,), h_last (H,))."""
    y, _, _ = lstm_stack(sd, prefix + "lstm.", x, 2, False)
    h_last = y[-1]
    return torch.sigmoid(h_last @ sd[prefix + "out.0.weight"].t() + sd[prefix + "out.0.bias"]), h_last


def sumgan_chain(sd, x, probes):
    """The deterministic chain the parity tests use (reparameterisation replaced by h = mu): scores -> eLSTM on the
    weighted features -> dLSTM -> cLSTM, and a scalar probe loss that reaches every parameter.
    probes: dict of fixed random tensors (x_hat, mu, logvar, h_last)."""
    scores = sumgan_slstm(sd, x)
    mu, logvar, c = sumgan_elstm(sd, x * scores[:, None])
    x_hat = sumgan_dlstm(sd, x.shape[0], mu, c)
    prob, h_last = sumgan_clstm(sd, x_hat)
    loss = (x_hat * probes["x_hat"]).sum() + (mu * probes["mu"]).sum() + (logvar * probes["logvar"]).sum() \
        + (h_last * probes["h_last"]).sum() + prob.sum() + (scores * probes["scores"]).sum()
    return dict(scores=scores, mu=mu, logvar=logvar, c=c, x_hat=x_hat, prob=prob, h_last=h_last, loss=loss)


def sumgan_probes(seed, T):
    g = torch.Generator().manual_seed(30_000 + seed)
    return dict(x_hat=torch.randn(T, 1024, generator=g), mu=torch.randn(2, 2048, generator=g),
                logvar=torch.randn(2, 2048, generator=g), h_last=torch.randn(1024, generator=g),
                scores=torch.randn(T, generator=g))
