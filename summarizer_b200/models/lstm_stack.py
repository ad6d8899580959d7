"""LSTM layers of the SumGAN family on the sm_100a recurrence kernels (csrc/smz_lstm.cu), with autograd.

What ``nn.LSTM`` hands to cuDNN in the reference (models/sumgan.py:43,69,95,207) is split the way the hardware
wants it: the input projections, dX and every weight gradient are whole-sequence tcgen05 GEMMs
(``summarizer_b200.dense.gemm``), the recurrence itself is one cooperative kernel per layer, and the dLSTM's
step-wise decode loop (sumgan.py:106-112: T separate one-step ``nn.LSTM`` calls, each re-reading its own output)
is ONE kernel.  The ``nn.LSTM`` modules only own the parameters (reference state-dict names and init stream);
they are never executed.  Batch 1 per call (the trainer's shape); callers loop over the batch dimension."""
import ctypes as C

import torch

from .. import _native as N
from ..dense import gemm
from ._packed import ShadowCache  # noqa: F401 (earlier import location)


class LstmSeq(C.Structure):
    """struct smz_lstm_seq (include/summarizer_b200.h)."""
    _fields_ = [(k, C.c_int32) for k in ("T", "H", "reverse", "ldpre", "ldy", "lddy", "ldg", "B")] + \
               [(k, C.c_void_p) for k in ("pre", "whh", "whh_t", "h0", "c0", "y", "gates", "cs", "h_last", "c_last",
                                          "dy", "dh_last", "dc_last", "dgates", "dh0", "dc0")]


class LstmDecode(C.Structure):
    """struct smz_lstm_decode (include/summarizer_b200.h)."""
    _fields_ = [("T", C.c_int32), ("H", C.c_int32), ("B", C.c_int32), ("reserved", C.c_int32)] + \
               [(k, C.c_void_p) for k in ("w_ih0", "w_hh0", "w_ih1", "w_hh1", "w_ih0_t", "w_hh0_t", "w_ih1_t", "w_hh1_t",
                                          "bias0", "bias1", "h_init", "c_init", "hs0", "hs1", "gates0", "gates1", "cs0", "cs1",
                                          "dy", "dgates0", "dgates1", "dh_init", "dc_init")]


def _off(t, elems):
    """device address of t.data_ptr() + elems elements (None stays None)."""
    return None if t is None else t.data_ptr() + elems * t.element_size()


def _sync_ws(device):
    return torch.empty(256, dtype=torch.uint8, device=device)


def _bf(t):
    return t.detach().to(torch.bfloat16).contiguous()


def layer_params(lstm, layer):
    """[(w_ih, w_hh, b_ih, b_hh)] per direction of ``lstm``'s layer."""
    out = []
    for sfx in ("", "_reverse")[: 2 if lstm.bidirectional else 1]:
        out.append(tuple(getattr(lstm, f"{n}_l{layer}{sfx}") for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")))
    return out


class _LayerShadow:
    def __init__(self, dirs):
        self.w_ih = _bf(torch.cat([d[0] for d in dirs], 0))                       # [nd*4H, in]
        self.bias = torch.cat([d[2] + d[3] for d in dirs]).detach().float().contiguous()
        self.whh = [_bf(d[1]) for d in dirs]                                      # [4H, H]
        self.whh_t = [_bf(d[1].t()) for d in dirs]                                # [H, 4H]


MAX_B = 4       # sequences of equal length per recurrence launch (csrc/smz_lstm.cu)


class _LstmLayerFn(torch.autograd.Function):
    """One (possibly bidirectional) LSTM layer over B <= 4 sequences of the same length that share the weights:
    (x [B,T,in], h0 [nd,B,H]|None, c0 [nd,B,H]|None) -> (y [B,T,nd*H], h_last [nd,B,H], c_last [nd,B,H]).  The per-step cost
    of the recurrence is the grid barrier and the weight stream, so the extra sequences are nearly free."""

    @staticmethod
    def forward(ctx, x, h0, c0, meta, *flat):
        N.require_device()
        cache, key, nd, H = meta
        dirs = [flat[4 * i: 4 * i + 4] for i in range(nd)]
        training = any(ctx.needs_input_grad)
        sh = cache.get(flat, lambda: _LayerShadow(dirs), key=key, fresh=training)
        B, T, dev = x.shape[0], x.shape[1], x.device
        xb = _bf(x).reshape(B * T, -1)
        pre = gemm(xb, sh.w_ih, bias=sh.bias)                                     # [B*T, nd*4H]
        f32 = dict(dtype=torch.float32, device=dev)
        y = torch.empty(B, T, nd * H, **f32)
        gates = torch.empty(B, T, nd * 4 * H, **f32) if training else None
        cs = torch.empty(nd, B, T, H, **f32) if training else None
        h_last, c_last = torch.empty(nd, B, H, **f32), torch.empty(nd, B, H, **f32)
        h0c = None if h0 is None else h0.detach().float().contiguous()
        c0c = None if c0 is None else c0.detach().float().contiguous()
        arr = (LstmSeq * nd)()
        for i in range(nd):
            a = arr[i]
            a.T, a.H, a.B, a.reverse, a.ldpre, a.ldy, a.ldg = T, H, B, i, nd * 4 * H, nd * H, nd * 4 * H
            a.pre, a.whh = _off(pre, i * 4 * H), sh.whh[i].data_ptr()
            a.h0, a.c0 = _off(h0c, i * B * H), _off(c0c, i * B * H)
            a.y, a.gates, a.cs = _off(y, i * H), _off(gates, i * 4 * H), _off(cs, i * B * T * H)
            a.h_last, a.c_last = _off(h_last, i * B * H), _off(c_last, i * B * H)
        N.check(N.lib().smz_lstm_seq_forward(arr, nd, N.ptr(_sync_ws(dev)), N.current_stream()))
        ctx.meta, ctx.sh, ctx.saved = meta, sh, (xb, y, gates, cs, h0c, c0c)
        ctx.set_materialize_grads(False)
        return y, h_last, c_last

    @staticmethod
    def backward(ctx, dy, dh_last, dc_last):
        cache, key, nd, H = ctx.meta
        sh = ctx.sh
        xb, y, gates, cs, h0c, c0c = ctx.saved
        B, T, dev = y.shape[0], y.shape[1], y.device
        f32 = dict(dtype=torch.float32, device=dev)
        dgates = torch.empty(B, T, nd * 4 * H, **f32)
        dh0, dc0 = torch.empty(nd, B, H, **f32), torch.empty(nd, B, H, **f32)
        dy = None if dy is None else dy.float().contiguous()
        dh_last = None if dh_last is None else dh_last.float().contiguous()
        dc_last = None if dc_last is None else dc_last.float().contiguous()
        arr = (LstmSeq * nd)()
        for i in range(nd):
            a = arr[i]
            a.T, a.H, a.B, a.reverse, a.lddy, a.ldg = T, H, B, i, nd * H, nd * 4 * H
            a.whh_t = sh.whh_t[i].data_ptr()
            a.c0 = _off(c0c, i * B * H)
            a.gates, a.cs = _off(gates, i * 4 * H), _off(cs, i * B * T * H)
            a.dy, a.dh_last, a.dc_last = _off(dy, i * H), _off(dh_last, i * B * H), _off(dc_last, i * B * H)
            a.dgates, a.dh0, a.dc0 = _off(dgates, i * 4 * H), _off(dh0, i * B * H), _off(dc0, i * B * H)
        N.check(N.lib().smz_lstm_seq_backward(arr, nd, N.ptr(_sync_ws(dev)), N.current_stream()))
        dgb = dgates.to(torch.bfloat16).reshape(B * T, nd * 4 * H)
        dx = gemm(dgb, sh.w_ih, b_mn=True).reshape(B, T, -1) if ctx.needs_input_grad[0] else None
        dw_ih = gemm(dgb, xb, a_mn=True, b_mn=True)                               # [nd*4H, in], summed over the B sequences
        db = dgates.sum((0, 1))
        grads = []
        for i in range(nd):
            h_first = (torch.zeros(B, H, **f32) if h0c is None else h0c[i]).unsqueeze(1)            # [B,1,H]
            yi = y[:, :, i * H:(i + 1) * H]
            hprev = torch.cat([h_first, yi[:, :-1]], 1) if i == 0 else torch.cat([yi[:, 1:], h_first], 1)
            dw_hh = gemm(dgb[:, i * 4 * H:(i + 1) * 4 * H], _bf(hprev).reshape(B * T, H), a_mn=True, b_mn=True)
            dbi = db[i * 4 * H:(i + 1) * 4 * H]
            grads += [dw_ih[i * 4 * H:(i + 1) * 4 * H], dw_hh, dbi, dbi]
        ctx.saved = None
        return (dx, dh0 if ctx.needs_input_grad[1] else None, dc0 if ctx.needs_input_grad[2] else None, None, *grads)


def _batched(x):
    return (x.unsqueeze(0), True) if x.dim() == 2 else (x, False)


def lstm_layer(cache, lstm, layer, x, h0=None, c0=None):
    """One layer of ``lstm`` over x [B,T,in] (float32 cuda, B <= 4) -> (y [B,T,nd*H], h_last [nd,B,H], c_last [nd,B,H])."""
    dirs = layer_params(lstm, layer)
    flat = [p for d in dirs for p in d]
    meta = (cache, (id(lstm), layer), len(dirs), lstm.hidden_size)
    return _LstmLayerFn.apply(x.float(), h0, c0, meta, *flat)


def lstm_stack(cache, lstm, x, h0=None, c0=None):
    """All layers of ``lstm`` (nn.LSTM semantics) over sequences of equal length: x [B,T,in] (or [T,in]); h0/c0
    [L*nd, B, H] (or [L*nd, H]) or None.  Returns (y [B,T,nd*H], h_n [L*nd,B,H], c_n [L*nd,B,H]) (batch dimension dropped
    when x was 2-D).  More than 4 sequences are processed in groups of 4."""
    x, squeeze = _batched(x)
    if squeeze:
        h0 = None if h0 is None else h0.unsqueeze(1)
        c0 = None if c0 is None else c0.unsqueeze(1)
    nd = 2 if lstm.bidirectional else 1
    ys, hns, cns = [], [], []
    for b0 in range(0, x.shape[0], MAX_B):
        xi, hs, cs = x[b0:b0 + MAX_B], [], []
        for layer in range(lstm.num_layers):
            sl = slice(layer * nd, (layer + 1) * nd)
            xi, h_l, c_l = lstm_layer(cache, lstm, layer, xi, None if h0 is None else h0[sl, b0:b0 + MAX_B],
                                      None if c0 is None else c0[sl, b0:b0 + MAX_B])
            hs.append(h_l); cs.append(c_l)
        ys.append(xi); hns.append(torch.cat(hs, 0)); cns.append(torch.cat(cs, 0))
    y, h_n, c_n = torch.cat(ys, 0), torch.cat(hns, 1), torch.cat(cns, 1)
    if squeeze:
        return y[0], h_n[:, 0], c_n[:, 0]
    return y, h_n, c_n


class _DecodeShadow:
    def __init__(self, p0, p1):
        self.w = [_bf(p0[0]), _bf(p0[1]), _bf(p1[0]), _bf(p1[1])]                 # w_ih0, w_hh0, w_ih1, w_hh1
        self.wt = [_bf(p0[0].t()), _bf(p0[1].t()), _bf(p1[0].t()), _bf(p1[1].t())]
        self.bias = [(p0[2] + p0[3]).detach().float().contiguous(), (p1[2] + p1[3]).detach().float().contiguous()]


class _DecodeFn(torch.autograd.Function):
    """dLSTM.forward's recurrence (sumgan.py:106-112) for B <= 4 decodes that share the weights:
    (h_init [2,B,H], c_init [2,B,H]) -> top-layer outputs [B,T,H]."""

    @staticmethod
    def forward(ctx, h_init, c_init, meta, *flat):
        N.require_device()
        cache, key, T, H = meta
        p0, p1 = flat[:4], flat[4:]
        training = any(ctx.needs_input_grad)
        sh = cache.get(flat, lambda: _DecodeShadow(p0, p1), key=key, fresh=training)
        dev, B = h_init.device, h_init.shape[1]
        f32 = dict(dtype=torch.float32, device=dev)
        hi, ci = h_init.detach().float().contiguous(), c_init.detach().float().contiguous()
        hs0, hs1 = torch.empty(B, T, H, **f32), torch.empty(B, T, H, **f32)
        save = [torch.empty(B, T, 4 * H, **f32), torch.empty(B, T, 4 * H, **f32), torch.empty(B, T, H, **f32),
                torch.empty(B, T, H, **f32)] if training else [None] * 4
        d = LstmDecode()
        d.T, d.H, d.B = T, H, B
        d.w_ih0, d.w_hh0, d.w_ih1, d.w_hh1 = (w.data_ptr() for w in sh.w)
        d.bias0, d.bias1, d.h_init, d.c_init = sh.bias[0].data_ptr(), sh.bias[1].data_ptr(), hi.data_ptr(), ci.data_ptr()
        d.hs0, d.hs1 = hs0.data_ptr(), hs1.data_ptr()
        d.gates0, d.gates1, d.cs0, d.cs1 = (_off(t, 0) for t in save)
        N.check(N.lib().smz_lstm_decode_forward(C.byref(d), N.ptr(_sync_ws(dev)), N.current_stream()))
        ctx.meta, ctx.sh, ctx.saved = meta, sh, (hi, ci, hs0, hs1, save)
        return hs1

    @staticmethod
    def backward(ctx, dy):
        cache, key, T, H = ctx.meta
        sh = ctx.sh
        hi, ci, hs0, hs1, save = ctx.saved
        dev, B = hs1.device, hs1.shape[0]
        f32 = dict(dtype=torch.float32, device=dev)
        dy = dy.float().contiguous()
        dg0, dg1 = torch.empty(B, T, 4 * H, **f32), torch.empty(B, T, 4 * H, **f32)
        dh_init, dc_init = torch.empty(2, B, H, **f32), torch.empty(2, B, H, **f32)
        d = LstmDecode()
        d.T, d.H, d.B = T, H, B
        d.w_ih0_t, d.w_hh0_t, d.w_ih1_t, d.w_hh1_t = (w.data_ptr() for w in sh.wt)
        d.h_init, d.c_init, d.hs0, d.hs1 = hi.data_ptr(), ci.data_ptr(), hs0.data_ptr(), hs1.data_ptr()
        d.gates0, d.gates1, d.cs0, d.cs1 = (t.data_ptr() for t in save)
        d.dy, d.dgates0, d.dgates1 = dy.data_ptr(), dg0.data_ptr(), dg1.data_ptr()
        d.dh_init, d.dc_init = dh_init.data_ptr(), dc_init.data_ptr()
        N.check(N.lib().smz_lstm_decode_backward(C.byref(d), N.ptr(_sync_ws(dev)), N.current_stream()))
        rows = lambda t: _bf(t).reshape(B * T, -1)
        dgb0, dgb1 = rows(dg0), rows(dg1)
        in0 = rows(torch.cat([torch.zeros(B, 1, H, **f32), hs1[:, :-1]], 1))     # layer 0's input: previous top output, zeros first
        prev0 = rows(torch.cat([hi[0].unsqueeze(1), hs0[:, :-1]], 1))
        prev1 = rows(torch.cat([hi[1].unsqueeze(1), hs1[:, :-1]], 1))
        dw_ih0 = gemm(dgb0, in0, a_mn=True, b_mn=True)
        dw_hh0 = gemm(dgb0, prev0, a_mn=True, b_mn=True)
        dw_ih1 = gemm(dgb1, rows(hs0), a_mn=True, b_mn=True)
        dw_hh1 = gemm(dgb1, prev1, a_mn=True, b_mn=True)
        db0, db1 = dg0.sum((0, 1)), dg1.sum((0, 1))
        ctx.saved = None
        return dh_init, dc_init, None, dw_ih0, dw_hh0, db0, db0, dw_ih1, dw_hh1, db1, db1


def lstm_decode(cache, lstm, seq_len, h_init, c_init):
    """T steps of the 2-layer ``lstm`` fed with its own top-layer output (zeros first): h_init / c_init [2,B,H] (or [2,H])
    -> [B,T,H] (or [T,H]).  More than 4 decodes are processed in groups of 4."""
    if lstm.num_layers != 2 or lstm.bidirectional or lstm.input_size != lstm.hidden_size:
        raise NotImplementedError("the decode kernel implements the dLSTM shape: 2 unidirectional layers, input size = hidden size")
    squeeze = h_init.dim() == 2
    if squeeze:
        h_init, c_init = h_init.unsqueeze(1), c_init.unsqueeze(1)
    flat = [p for layer in (0, 1) for p in layer_params(lstm, layer)[0]]
    meta = (cache, (id(lstm), "decode"), int(seq_len), lstm.hidden_size)
    outs = [_DecodeFn.apply(h_init[:, b0:b0 + MAX_B], c_init[:, b0:b0 + MAX_B], meta, *flat)
            for b0 in range(0, h_init.shape[1], MAX_B)]
    top = torch.cat(outs, 0)
    return top[0] if squeeze else top
