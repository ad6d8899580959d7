"""Host-side plumbing shared by the modules that run on the library's kernels: the cache of the parameter copies the
kernels read (``ShadowCache``, owned by every ``NativeModule``) and the start of a packed (ragged-batch) call."""
import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from .. import _native as N


class ShadowCache:
    """bf16 / packed / folded copies of parameters for the kernels, one entry per ``key``.

    An entry is reused while every parameter keeps its storage and ``Tensor._version`` and ``config`` (module settings
    the copies depend on) is unchanged, so ``load_state_dict`` and ``.cuda()`` rebuild it.  ``fresh=True`` (training
    forwards) always rebuilds and leaves the entry dirty: an optimizer step follows, and the library's Adam and torch's
    fused optimizers update parameters in place without bumping ``_version``.  ``clear()`` drops every entry."""

    def __init__(self):
        self._store = {}

    def get(self, params, build, key=None, config=(), fresh=False):
        tag = tuple((p.data_ptr(), p._version) for p in params) + config
        ent = self._store.get(key)
        if fresh or ent is None or ent[0] != tag:
            with torch.no_grad():
                ent = (None if fresh else tag, build())
            self._store[key] = ent
        return ent[1]

    def peek(self, key=None):
        """The copies last built for ``key``, or None; no check that they are current."""
        ent = self._store.get(key)
        return None if ent is None else ent[1]

    def clear(self):
        self._store.clear()


class NativeModule(nn.Module):
    """A module whose kernels read cached copies of its parameters (``self._cache``).  ``Trainer`` clears the cache of
    every such module around captured and replayed training steps."""

    def __init__(self):
        super().__init__()
        self._cache = ShadowCache()

    # older spellings, kept for scripts and tests that use them: ``m._shadow_key = None`` is ``m._cache.clear()``,
    # ``m._shadow`` the copies the last call built
    _shadow_key = property(None, lambda self, _: self._cache.clear())
    _shadow = property(lambda self: self._cache.peek())


def cu_seqlens(lengths):
    """Host int32 prefix offsets of ``lengths`` ([0, T0, T0+T1, ...]), the ``h_cu_seqlens`` of the packed calls."""
    cu = np.zeros(len(lengths) + 1, dtype=np.int32)
    np.cumsum(np.asarray(lengths, dtype=np.int64), out=cu[1:])
    return cu


class Workspace:
    """Grow-only device work buffer, one per (device, purpose)."""

    def __init__(self):
        self.buf = None

    def get(self, nbytes, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(max(int(nbytes), 1024), dtype=torch.uint8, device=device)
        return self.buf


def workspace_bytes(query, *args):
    """Work-buffer bytes from one of the library's ``smz_*_workspace_bytes(..., int64_t *bytes)`` queries."""
    nbytes = C.c_int64(0)
    N.check(query(*args, C.byref(nbytes)))
    return nbytes.value


def packed_input(x, lengths, width):
    """The start of every packed call: ``x`` [sum T, width] as a contiguous float32 / bfloat16 device tensor, the host
    prefix offsets of ``lengths`` and the kernels' ``x_is_bf16`` flag."""
    N.require_device()
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.contiguous()
    cu = cu_seqlens(lengths)
    assert x.shape == (int(cu[-1]), width)
    return x, cu, int(x.dtype == torch.bfloat16)


def score_sequences(score_packed, x):
    """The reference's ``forward`` contract over a packed scorer: x (T, B, D) -> ``score_packed(rows [B*T, D], [T] * B)``
    -> scores (T, B, 1)."""
    seq_len, batch_size, width = x.shape
    s = score_packed(x.permute(1, 0, 2).reshape(batch_size * seq_len, width), [seq_len] * batch_size)
    return s.view(batch_size, seq_len, 1).permute(1, 0, 2)
