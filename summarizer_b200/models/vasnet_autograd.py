"""Autograd shell around smz_vasnet_forward(training=1) / smz_vasnet_backward.

PyTorch only records the node and owns the buffers; forward and backward are the sm_100a kernels.  The three
p=0.5 dropouts of the reference (models/vasnet.py:130,136,142) are driven by torch's CUDA generator
(``torch.manual_seed`` reproduces them): the KEEP masks are drawn here and handed to the kernels, which is
also what lets the tests replay the very same masks through the float32 oracle.
"""
import ctypes as C

import torch

from .. import _native as N
from ._packed import packed_input, workspace_bytes
from .vasnet import LO_KEYS, SPLIT, VasnetParams


class VasnetGrads(C.Structure):
    """struct smz_vasnet_grads (include/summarizer_b200.h)."""
    _fields_ = [(k, C.c_void_p) for k in ("wqk", "wv", "wo", "w1", "b1", "w2", "b2", "ln_g", "ln_b", "dx")]


def mask_state(device, seed=None):
    """Draw state of smz_dropout_keep_masks: {Philox seed, call number, 0} as three device int64 words.  The seed comes
    from torch's CPU generator unless given, so ``torch.manual_seed`` reproduces the masks."""
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    return torch.tensor([seed, 0, 0], dtype=torch.int64, device=device)


def draw_keep_masks(lengths, device, generator=None):
    """KEEP masks (uint8, 1 = keep) of nn.Dropout(0.5) at the three sites, for a packed batch.  ``generator``: a
    ``mask_state`` tensor (the library's Philox kernel: one launch, graph-replayable, no process-wide generator — what the
    module uses), or a torch.Generator / None (torch's generator: tests that replay masks through the float32 oracle)."""
    rows = int(sum(lengths))
    n_att = int(sum(t * t for t in lengths))
    n_att_pad = (n_att + 15) // 16 * 16                     # keeps the row masks 16-byte aligned (uchar4 loads)
    if torch.is_tensor(generator):
        keep = torch.empty(n_att_pad + 2 * rows * 1024, dtype=torch.uint8, device=device)
        N.check(N.lib().smz_dropout_keep_masks(N.ptr(generator), N.ptr(keep), keep.numel(), N.current_stream()))
    else:
        keep = (torch.rand(n_att_pad + 2 * rows * 1024, device=device, generator=generator) >= 0.5).to(torch.uint8)   # one draw
    return (keep[:n_att], keep[n_att_pad:n_att_pad + rows * 1024].view(rows, 1024),
            keep[n_att_pad + rows * 1024:].view(rows, 1024))


class _VasnetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, module, lengths, masks, wq, wk, wv, wo, w1, b1, w2, b2, ln_g, ln_b):
        x, cu, is_bf16 = packed_input(x, lengths, 1024)
        cu_p = cu.ctypes.data_as(C.c_void_p)
        sh, st = module._weights(inference=False)
        split = SPLIT if module.precision == "fp32" else 0            # room for the activations' lo planes
        nbytes = workspace_bytes(N.lib().smz_vasnet_workspace_bytes, cu_p, len(lengths), 1 | split, is_bf16)
        ws = torch.empty(max(nbytes, 1024), dtype=torch.uint8, device=x.device)   # lives until backward
        scores = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        m_att, m_y, m_h = masks if masks is not None else (None, None, None)
        N.check(N.lib().smz_vasnet_forward(N.ptr(x), is_bf16, cu_p, len(lengths), C.byref(st), 1, N.ptr(m_att), N.ptr(m_y),
                                           N.ptr(m_h), N.ptr(scores), N.ptr(ws), ws.numel(), N.current_stream()))
        ctx.module, ctx.cu, ctx.masks, ctx.ws, ctx.shadow = module, cu, masks, ws, sh
        ctx.save_for_backward(x, scores)
        return scores

    @staticmethod
    def backward(ctx, dscores):
        x, scores = ctx.saved_tensors
        m = ctx.module
        dev = x.device
        shapes = dict(wqk=(2048, 1024), wv=(1024, 1024), wo=(1024, 1024), w1=(1024, 1024), b1=(1024,), w2=(1024,), b2=(1,),
                      ln_g=(1024,), ln_b=(1024,))
        sizes = {k: (int(torch.Size(v).numel()) + 3) // 4 * 4 for k, v in shapes.items()}    # 16-byte aligned slices
        flat = torch.zeros(sum(sizes.values()), dtype=torch.float32, device=dev)              # one memset for all gradients
        g, o = {}, 0
        for k, shp in shapes.items():
            g[k] = flat[o:o + int(torch.Size(shp).numel())].view(shp)
            o += sizes[k]
        z = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=dev)
        dx = z(x.shape[0], 1024) if ctx.needs_input_grad[0] else None
        gs = VasnetGrads(*(g[k].data_ptr() for k in ("wqk", "wv", "wo", "w1", "b1", "w2", "b2", "ln_g", "ln_b")),
                         dx.data_ptr() if dx is not None else None)
        sh = ctx.shadow   # the bf16 weights the forward used
        st = VasnetParams(*(sh[k].data_ptr() for k in ("wqk", "wv", "wo", "w1", "b1", "w2", "b2", "ln_g", "ln_b")),
                          float(m.scale), float(m.epsilon), -1 if m.aperture is None else int(m.aperture),
                          int(bool(m.ignore_self)), *([None] * 8), *((sh[k].data_ptr() if k in sh else None) for k in LO_KEYS))
        m_att, m_y, m_h = ctx.masks if ctx.masks is not None else (None, None, None)
        cu = ctx.cu
        N.check(N.lib().smz_vasnet_backward(N.ptr(x), int(x.dtype == torch.bfloat16), cu.ctypes.data_as(C.c_void_p),
                                            len(cu) - 1, C.byref(st), N.ptr(m_att), N.ptr(m_y), N.ptr(m_h), N.ptr(scores),
                                            N.ptr(dscores.contiguous().float()), C.byref(gs), N.ptr(ctx.ws), ctx.ws.numel(),
                                            N.current_stream()))
        ctx.ws = None
        return (dx, None, None, None, g["wqk"][:1024], g["wqk"][1024:], g["wv"], g["wo"], g["w1"], g["b1"],
                g["w2"].view(1, 1024), g["b2"], g["ln_g"], g["ln_b"])


def vasnet_apply(module, packed, lengths, masks="auto"):
    """scores [sum T] with autograd.  masks: "auto" draws dropout keep-masks when module.training,
    None disables dropout, or an explicit (att, y, h) tuple (tests)."""
    if masks == "auto":
        if module.training:
            if getattr(module, "_mask_state", None) is None or module._mask_state.device != packed.device:
                module._mask_state = mask_state(packed.device)
            masks = draw_keep_masks(lengths, packed.device, module._mask_state)
        else:
            masks = None
    return _VasnetFunction.apply(packed, module, list(lengths), masks, module.Q.weight, module.K.weight, module.V.weight,
                                 module.attention_head_projection.weight, module.k1.weight, module.k1.bias,
                                 module.k2.weight, module.k2.bias, module.layer_norm.weight, module.layer_norm.bias)
