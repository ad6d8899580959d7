"""VASNet — "Summarizing Videos with Attention" scorer with the reference's class, constructor,
parameter names and ``forward((T, B, 1024)) -> (T, B, 1)`` contract (models/vasnet.py:17-148), computed
by the sm_100a kernels of libsummarizer_b200.so (smz_vasnet_forward / smz_vasnet_backward).

The module keeps ordinary float32 ``nn.Parameter``s under the reference's names, so reference ``.pth``
files load unchanged (``layer_norm.{weight,bias}``, ``{K,Q,V,attention_head_projection}.weight``,
``k1.{weight,bias}``, ``k2.{weight,bias}``, optional ``pos_embed.weight``); bfloat16 copies for the
tensor cores are derived on the fly and never saved.  There is no CPU / eager fallback.
"""
import ctypes as C
import functools
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.init as init

from .. import _native as N
from ._packed import NativeModule, Workspace, cu_seqlens, packed_input, score_sequences, workspace_bytes
from ._packed import Workspace as _Workspace, cu_seqlens as _cu_seqlens  # noqa: F401 (earlier import location)


class VasnetParams(C.Structure):
    """struct smz_vasnet_params (include/summarizer_b200.h)."""
    _fields_ = [("wqk", C.c_void_p), ("wv", C.c_void_p), ("wo", C.c_void_p), ("w1", C.c_void_p),
                ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p), ("ln_g", C.c_void_p),
                ("ln_b", C.c_void_p), ("scale", C.c_float), ("eps", C.c_float), ("aperture", C.c_int32),
                ("ignore_self", C.c_int32), ("head_gw", C.c_void_p), ("head_c", C.c_void_p),
                ("w1g", C.c_void_p), ("ln_c", C.c_void_p), ("b1f", C.c_void_p), ("wgv", C.c_void_p), ("wgv16", C.c_void_p),
                ("status", C.c_void_p),
                ("wqk_lo", C.c_void_p), ("wv_lo", C.c_void_p), ("wo_lo", C.c_void_p), ("w1_lo", C.c_void_p)]

SPLIT = 4      # SMZ_VASNET_SPLIT: OR into `training` of smz_vasnet_workspace_bytes (room for the lo planes)
LO_KEYS = ("wqk_lo", "wv_lo", "wo_lo", "w1_lo")


class VASNet(NativeModule):
    def __init__(self, input_size=1024, max_length=None, pos_embed="simple", ignore_self=False,
                 attention_aperture=None, scale=None, epsilon=1e-6, weight_init="xavier", precision="bf16"):
        """Reference constructor (vasnet.py:18-21) + ``precision``: "bf16" (default: bf16 / float16 tensor-core operands,
        scores within 1e-2 of the float32 reference) or "fp32" (split-bf16 operands, every contraction as three
        tensor-core products: scores within 1e-4 of the float32 reference, forward AND backward; ~3 x the GEMM time)."""
        super().__init__()
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.precision = precision
        if input_size != 1024:
            raise ValueError("the sm_100a VASNet kernels are built for 1024-d features (GoogLeNet pool5)")
        self.input_size = input_size
        self.aperture = attention_aperture          # None = global attention, w = frames [t-w, t+w]
        self.ignore_self = ignore_self
        self.scale = scale if scale is not None else 1 / np.sqrt(self.input_size)
        self.epsilon = epsilon

        # optional positional information (vasnet.py:37-51): a learned table or the fixed sin/cos one,
        # which the reference keeps as a plain tensor outside the state dict
        self.max_length = max_length
        if self.max_length:
            self.pos_embed_type = pos_embed
            if pos_embed == "simple":
                self.pos_embed = nn.Embedding(self.max_length, self.input_size)
            elif pos_embed == "attention":
                pos = np.arange(self.max_length, dtype=np.float64)[:, None]
                i = np.arange(self.input_size, dtype=np.float64)[None, :]
                table = np.where(i % 2 == 0, np.sin(pos / 10000 ** (2 * i / self.input_size)),
                                 np.cos(pos / 10000 ** (2 * i / self.input_size)))
                self.pos_embed = torch.from_numpy(table).float()
            else:
                self.max_length = None

        self.dropout = nn.Dropout(0.5)
        self.layer_norm = nn.LayerNorm(self.input_size, epsilon)
        d = self.input_size
        self.K = nn.Linear(d, d, bias=False)
        self.Q = nn.Linear(d, d, bias=False)
        self.V = nn.Linear(d, d, bias=False)
        self.attention_head_projection = nn.Linear(d, d, bias=False)
        self.softmax = nn.Softmax(dim=2)
        self.k1 = nn.Linear(d, d)
        self.k2 = nn.Linear(d, 1)
        self.sigmoid = nn.Sigmoid()
        self.relu = nn.ReLU()

        mats = (self.K, self.Q, self.V, self.attention_head_projection, self.k1, self.k2)
        for m in mats:                               # vasnet.py:71-86
            if weight_init.lower() in ("he", "kaiming"):
                init.kaiming_uniform_(m.weight)
            else:
                init.xavier_uniform_(m.weight, gain=np.sqrt(2.0))
        init.constant_(self.k1.bias, 0.1)
        init.constant_(self.k2.bias, 0.1)

        self._status = None
        self._ws = Workspace()

    # ---------------------------------------------------------------------------------------------
    def _weights(self, inference=True, fast=True):
        """The kernels' weight copies (``_build_weights``, cached in ``self._cache``; a training forward,
        ``inference=False``, rebuilds them) and the parameter struct over them.  The fast inference path's fields are set
        when ``fast`` and its weights allow it."""
        ps = (self.Q.weight, self.K.weight, self.V.weight, self.attention_head_projection.weight,
              self.k1.weight, self.k1.bias, self.k2.weight, self.k2.bias, self.layer_norm.weight,
              self.layer_norm.bias)
        sh = self._cache.get(ps, lambda: self._build_weights(inference), config=(self.precision,), fresh=not inference)
        # the folded 16-bit fast path is the bf16 mode's
        fast = inference and fast and self.precision != "fp32" and sh["fast_ok"]
        st = VasnetParams(*(sh[k].data_ptr() for k in ("wqk", "wv", "wo", "w1", "b1", "w2", "b2", "ln_g", "ln_b")),
                          float(self.scale), float(self.epsilon),
                          -1 if self.aperture is None else int(self.aperture), int(bool(self.ignore_self)),
                          *((sh[k].data_ptr() if inference else None) for k in ("head_gw", "head_c", "w1g", "ln_c", "b1f")),
                          *((sh[k].data_ptr() if fast else None) for k in ("wgv", "wgv16")),
                          self._status_word(sh["ln_g"].device).data_ptr() if fast else None,
                          *((sh[k].data_ptr() if k in sh else None) for k in LO_KEYS))
        return sh, st

    def _build_weights(self, inference):
        """bfloat16 copies of the matrices (plus their lo planes in the float32-accurate mode) and float32 vectors.  The
        folded head constants and the fast path's folded projections are only derived for inference (the training path
        keeps the separate head kernel)."""
        big = (self.Q.weight, self.K.weight, self.V.weight, self.attention_head_projection.weight, self.k1.weight)
        lo = None
        if self.precision == "fp32":
            # float32-accurate mode: hi + lo bf16 planes of the five matrices in one launch
            src_t = [t.detach().float().contiguous() for t in big]
            flat = torch.empty(2, 5 * 1024 * 1024, dtype=torch.bfloat16, device=big[0].device)
            src = (C.c_void_p * 5)(*(t.data_ptr() for t in src_t))
            dst = (C.c_void_p * 5)(*(flat[0].data_ptr() + 2 * 1024 * 1024 * i for i in range(5)))
            dlo = (C.c_void_p * 5)(*(flat[1].data_ptr() + 2 * 1024 * 1024 * i for i in range(5)))
            cnt = (C.c_int64 * 5)(*([1024 * 1024] * 5))
            N.check(N.lib().smz_split_bf16_multi(src, dst, dlo, cnt, 5, N.current_stream()))
            w, wl = flat[0].view(5 * 1024, 1024), flat[1].view(5 * 1024, 1024)
            wqk, wv, wo, w1 = w[:2048], w[2048:3072], w[3072:4096], w[4096:]
            lo = dict(wqk_lo=wl[:2048], wv_lo=wl[2048:3072], wo_lo=wl[3072:4096], w1_lo=wl[4096:])
        elif all(t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() for t in big):
            # one launch: [Q;K] | V | O | k1 -> one bf16 buffer (no fp32 concatenation, no cast kernel per tensor)
            flat = torch.empty(5 * 1024 * 1024, dtype=torch.bfloat16, device=big[0].device)
            src = (C.c_void_p * 5)(*(t.data_ptr() for t in big))
            dst = (C.c_void_p * 5)(*(flat.data_ptr() + 2 * 1024 * 1024 * i for i in range(5)))
            cnt = (C.c_int64 * 5)(*([1024 * 1024] * 5))
            N.check(N.lib().smz_cvt_bf16_multi(src, dst, cnt, 5, N.current_stream()))
            w = flat.view(5 * 1024, 1024)
            wqk, wv, wo, w1 = w[:2048], w[2048:3072], w[3072:4096], w[4096:]
        else:
            wqk = torch.cat([self.Q.weight, self.K.weight], 0).to(torch.bfloat16).contiguous()
            wv, wo, w1 = (t.to(torch.bfloat16).contiguous() for t in big[2:])
        sh = dict(
            wqk=wqk, wv=wv, wo=wo, w1=w1,
            b1=self.k1.bias.float().contiguous(), w2=self.k2.weight.float().reshape(-1).contiguous(),
            b2=self.k2.bias.float().contiguous(), ln_g=self.layer_norm.weight.float().contiguous(),
            ln_b=self.layer_norm.bias.float().contiguous())
        if lo is not None:
            sh.update(lo)
        if not inference:
            return sh
        # regressor head folded into the k1 epilogue: z = rstd * (sum h*gw - mean * c0) + c1
        sh["head_gw"] = (sh["ln_g"] * sh["w2"]).contiguous()
        sh["head_c"] = torch.stack([sh["head_gw"].sum(), (sh["ln_b"] * sh["w2"]).sum() + sh["b2"][0]]).contiguous()
        # first LayerNorm folded into k1: W1.LN(y) + b1 = rstd * (W1g.y - mean * rowsum(W1g)) + (W1.ln_b + b1)
        w1 = self.k1.weight.float()
        sh["w1g"] = (w1 * sh["ln_g"][None, :]).to(torch.float16).contiguous()       # float16: y is handed over as float16
        sh["ln_c"] = sh["w1g"].float().sum(1).contiguous()
        sh["b1f"] = (w1 @ sh["ln_b"] + sh["b1"]).contiguous()
        # folded projections of the fast path (products in float32): rows 0..1023 = Wo Wv, 1024..2047 = Wk^T Wq.
        # The fast path is only offered when 16-bit floats hold them well (no overflow, the largest entries far
        # above the float16 subnormal range)
        wq, wk, wv, wo = (t.detach().float() for t in (self.Q.weight, self.K.weight, self.V.weight,
                                                       self.attention_head_projection.weight))
        gv = torch.cat([wo @ wv, wk.t() @ wq], 0)
        amax = torch.stack([gv[:1024].abs().max(), gv[1024:].abs().max(), (w1 * sh["ln_g"][None, :]).abs().max()])
        sh["fast_ok"] = bool((torch.isfinite(amax) & (amax < 6e4) & (amax > 1e-3)).all().item())
        sh["wgv"] = gv.to(torch.bfloat16).contiguous()
        sh["wgv16"] = gv.to(torch.float16).contiguous()
        return sh

    def _status_word(self, device):
        """Device word the fast inference path ORs SMZ_VASNET_STATUS_* into (include/summarizer_b200.h)."""
        if self._status is None or self._status.device != device:
            self._status = torch.zeros(1, dtype=torch.int32, device=device)
        return self._status

    def check_status(self):
        """True when every fast-path call since the last check stayed inside the checked value ranges (synchronises).
        ``score_packed(check=True)`` does this itself; callers that pipeline several ``check=False`` calls ask once at
        the end and, on False, repeat them with ``exact=True``."""
        if self._status is None:
            return True
        bad = int(self._status.item())
        if bad:
            self._status.zero_()
        return bad == 0

    def score_packed(self, x, lengths, check=True, exact=False):
        """Inference over a ragged batch: ``x`` packed [sum T, 1024] (float32 or bfloat16, device),
        ``lengths`` the per-video frame counts.  Returns float32 scores [sum T].

        The fast path (softmax without the max subtraction, float16 LayerNorm input) is exact inside value ranges the
        kernels check on the fly; ``check=True`` reads the status word after the call (one synchronisation, as the
        reference's own ``.cpu()`` per video) and repeats the call on the exact path if a range was left.
        ``check=False`` leaves that to a later ``check_status()``; ``exact=True`` takes the exact path directly."""
        x, cu, is_bf16 = packed_input(x, lengths, self.input_size)
        if self.precision == "fp32":
            return self._score_packed_split(x, lengths)
        _, st = self._weights(fast=not exact)
        cu_p = cu.ctypes.data_as(C.c_void_p)
        ws = self._ws.get(workspace_bytes(N.lib().smz_vasnet_workspace_bytes, cu_p, len(lengths), 0, is_bf16), x.device)
        scores = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        N.check(N.lib().smz_vasnet_forward(N.ptr(x), is_bf16, cu_p, len(lengths), C.byref(st), 0, None, None, None,
                                           N.ptr(scores), N.ptr(ws), ws.numel(), N.current_stream()))
        if check and not exact and not self.check_status():
            return self.score_packed(x, lengths, exact=True)
        return scores

    def _score_packed_split(self, x, lengths, max_rows=8192):
        """float32-accurate inference: the training-layout forward (every intermediate kept per video, no dropout) on
        split-bf16 operands, a few videos per call so that the doubled work buffer stays small."""
        _, st = self._weights()
        scores = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        is_bf16 = int(x.dtype == torch.bfloat16)
        v0, row0 = 0, 0
        while v0 < len(lengths):
            v1, rows = v0, 0
            while v1 < len(lengths) and (v1 == v0 or rows + lengths[v1] <= max_rows):
                rows += int(lengths[v1]); v1 += 1
            cu_p = cu_seqlens(lengths[v0:v1]).ctypes.data_as(C.c_void_p)
            ws = self._ws.get(workspace_bytes(N.lib().smz_vasnet_workspace_bytes, cu_p, v1 - v0, 1 | SPLIT, is_bf16), x.device)
            N.check(N.lib().smz_vasnet_forward(N.ptr(x[row0:row0 + rows]), is_bf16, cu_p, v1 - v0, C.byref(st), 1, None, None,
                                               None, N.ptr(scores[row0:row0 + rows]), N.ptr(ws), ws.numel(), N.current_stream()))
            v0, row0 = v1, row0 + rows
        return scores

    def forward(self, x):
        """
        Input
          x: (seq_len, batch_size, input_size)
        Output
          y: (seq_len, batch_size, 1)
        """
        seq_len, batch_size, input_size = x.shape
        assert self.input_size == input_size
        if not x.is_cuda:
            raise N.NativeError("summarizer_b200.VASNet runs on a CUDA (sm_100a) device only; move the input with .cuda()")
        if self.max_length is not None:
            assert self.max_length >= seq_len, "input sequence has higher length than max_length"
            xb = x.permute(1, 0, 2)                 # a view: the in-place add reaches the caller's tensor
            if self.pos_embed_type == "simple":     # (vasnet.py:110,112 quirk kept)
                pos = torch.arange(seq_len, device=x.device).repeat(1, batch_size).view(batch_size, seq_len)
                xb += self.pos_embed(pos)
            else:
                xb += self.pos_embed[:seq_len, :].repeat(1, batch_size).view(batch_size, seq_len, input_size).to(x.device)
        if torch.is_grad_enabled() and (self.training or any(p.requires_grad for p in self.parameters())):
            from .vasnet_autograd import vasnet_apply
            return score_sequences(functools.partial(vasnet_apply, self), x)
        return score_sequences(self.score_packed, x)


from . import Trainer  # noqa: E402


class VASNetTrainer(Trainer):
    """models/vasnet.py:151-238 — MSE regression of the (min-max normalised) ground-truth scores, one
    Adam step per video; extra parameters as the reference parses them (vasnet.py:153-161)."""

    def _init_model(self):
        ep = self.hps.extra_params or {}
        model = VASNet(
            max_length=int(ep["max_pos"]) if "max_pos" in ep else None,
            pos_embed=ep.get("pos_embed", "simple"),
            ignore_self=bool(ep.get("ignore_self", False)),
            attention_aperture=int(ep["local"]) if "local" in ep else None,
            scale=float(ep["scale"]) if "scale" in ep else None,
            epsilon=float(ep.get("epsilon", 1e-6)),
            weight_init=ep.get("weight_init", "xavier"),
            precision=str(ep.get("precision", "bf16")))
        if self.hps.use_cuda:
            self.log.info(f"Setting CUDA device: {self.hps.cuda_device}")
            torch.cuda.set_device(self.hps.cuda_device)
            model.cuda()
        return model

    def _packed_scorer(self):
        return self.model if self.model.max_length is None else None

    def train(self, fold):
        return self._train_supervised(fold)
