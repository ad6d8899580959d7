"""The cache of the parameter copies the kernels read (``ShadowCache``, models/_packed.py): when an entry is reused and
when it is rebuilt.  CPU tensors and a build function that counts its calls; no device, no library."""
from types import SimpleNamespace

import torch
import torch.nn as nn

from summarizer_b200.models import Trainer
from summarizer_b200.models._packed import NativeModule, ShadowCache


class Scorer(NativeModule):
    """A module whose "copies" are the number of builds so far."""

    def __init__(self):
        super().__init__()
        self.lin = nn.Linear(3, 2)
        self.builds = 0

    def copies(self, fresh=False, config=()):
        return self._cache.get(list(self.parameters()), self._build, config=config, fresh=fresh)

    def _build(self):
        assert not torch.is_grad_enabled()
        self.builds += 1
        return self.builds


def test_reused_when_nothing_changed():
    m = Scorer()
    assert [m.copies() for _ in range(3)] == [1, 1, 1]
    assert m.builds == 1


def test_rebuilt_after_an_in_place_update():
    m = Scorer()
    m.copies()
    with torch.no_grad():
        m.lin.weight.add_(1.0)                       # bumps Tensor._version, same storage
    assert [m.copies(), m.copies()] == [2, 2]


def test_rebuilt_after_a_storage_change():
    a, b = torch.zeros(4), torch.ones(2, 3)
    b2 = b.clone()                                   # same values and version, other storage
    assert b2._version == b._version and b2.data_ptr() != b.data_ptr()
    cache, calls = ShadowCache(), []
    build = lambda: calls.append(1) or len(calls)
    assert cache.get([a, b], build) == 1
    assert cache.get([a, b2], build) == 2
    assert cache.get([a, b2], build) == 2


def test_rebuilt_after_a_config_change():
    m = Scorer()
    assert [m.copies(config=("bf16",)), m.copies(config=("fp32",)), m.copies(config=("fp32",))] == [1, 2, 2]


def test_fresh_rebuilds_and_leaves_the_entry_dirty():
    """A training forward: an optimizer step that does not bump ``_version`` may follow, so the next call rebuilds."""
    m = Scorer()
    assert m.copies() == 1
    assert m.copies(fresh=True) == 2
    assert m.copies(fresh=True) == 3
    assert [m.copies(), m.copies()] == [4, 4]


def test_rebuilt_after_clear():
    m = Scorer()
    m.copies()
    m._cache.clear()
    assert [m.copies(), m.copies()] == [2, 2]
    assert m._shadow == 2                            # the older spelling of the last copies built
    m._shadow_key = None                             # the older spelling of clear()
    assert m._shadow is None and m.copies() == 3


def test_entries_are_kept_per_key():
    p = [torch.zeros(2)]
    cache, calls = ShadowCache(), []
    build = lambda: calls.append(1) or len(calls)
    assert [cache.get(p, build, key="a"), cache.get(p, build, key="b"), cache.get(p, build, key="a")] == [1, 2, 1]


def test_trainer_clears_every_native_module():
    """Trainer._invalidate_shadows reaches native modules at any depth of the model."""
    outer = nn.Module()
    outer.inner = nn.Sequential(Scorer(), nn.Linear(2, 2))
    outer.top = Scorer()
    scorers = [outer.inner[0], outer.top]
    for s in scorers:
        s.copies()
    Trainer._invalidate_shadows(SimpleNamespace(model=outer))
    assert [s.copies() for s in scorers] == [2, 2]
