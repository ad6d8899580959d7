"""Autograd shell around smz_dsn_forward(training=1) / smz_dsn_backward (BPTT on the device)."""
import ctypes as C

import torch

from .. import _native as N
from ._packed import packed_input, workspace_bytes
from .dsn import DsnParams


class DsnGrads(C.Structure):
    """struct smz_dsn_grads (include/summarizer_b200.h)."""
    _fields_ = [(k, C.c_void_p) for k in ("w_ih", "w_hh", "bias", "w_out", "b_out")]


class _DsnFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, module, lengths, *params):
        x, cu, is_bf16 = packed_input(x, lengths, 1024)
        sh, st = module._weights(training=True)
        nbytes = workspace_bytes(N.lib().smz_dsn_workspace_bytes, int(cu[-1]), len(lengths), 1, is_bf16)
        ws = torch.empty(max(nbytes, 1024), dtype=torch.uint8, device=x.device)
        probs = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        N.check(N.lib().smz_dsn_forward(N.ptr(x), is_bf16, cu.ctypes.data_as(C.c_void_p), len(lengths), C.byref(st), 1,
                                        N.ptr(probs), N.ptr(ws), ws.numel(), N.current_stream()))
        ctx.cu, ctx.ws, ctx.shadow = cu, ws, sh
        ctx.save_for_backward(x, probs)
        return probs

    @staticmethod
    def backward(ctx, dprobs):
        x, probs = ctx.saved_tensors
        z = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=x.device)
        g = dict(w_ih=z(2048, 1024), w_hh=z(2048, 256), bias=z(2048), w_out=z(512), b_out=z(1))
        gs = DsnGrads(*(g[k].data_ptr() for k in ("w_ih", "w_hh", "bias", "w_out", "b_out")))
        sh = ctx.shadow
        st = DsnParams(*(sh[k].data_ptr() for k in ("w_ih", "bias", "whh", "whh_t", "w_out", "b_out")))
        cu = ctx.cu
        N.check(N.lib().smz_dsn_backward(N.ptr(x), int(x.dtype == torch.bfloat16), cu.ctypes.data_as(C.c_void_p), len(cu) - 1,
                                         C.byref(st), N.ptr(probs), N.ptr(dprobs.contiguous().float()), C.byref(gs),
                                         N.ptr(ctx.ws), ctx.ws.numel(), N.current_stream()))
        ctx.ws = None
        # parameter order of DSN._params(): forward direction, reverse direction, head
        return (None, None, None,
                g["w_ih"][:1024], g["w_hh"][:1024], g["bias"][:1024], g["bias"][:1024],
                g["w_ih"][1024:], g["w_hh"][1024:], g["bias"][1024:], g["bias"][1024:],
                g["w_out"].view(1, 512), g["b_out"])


def dsn_apply(module, packed, lengths):
    """probs [sum T] with autograd through the device BPTT."""
    return _DsnFunction.apply(packed, module, list(lengths), *module._params())
