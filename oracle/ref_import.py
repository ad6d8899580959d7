"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Imports the UNMODIFIED reference (sylvainma/Summarizer) from a checkout of it, so the oracle
restatement can be validated against it and golden vectors can be generated (oracle/gen_golden.py).
The checkout is not part of this repository: $SMZ_REFERENCE_ROOT names its root directory (the one
holding the reference's ``summarizer/`` package).  Without it ``available()`` is False and the tests
marked ``reference`` skip.

Two third-party modules the reference imports are absent from this image and are stubbed in
``sys.modules`` before import (SURVEY.md §8c):
  * ``h5py``     — only ``h5py.File`` is used (models/__init__.py:15,149); the stub's File is a
                   dict-backed shim over an in-memory dataset.
  * ``ortools``  — ``pywrapknapsack_solver.KnapsackSolver`` (utils/knapsack.py:7-21); the stub
                   serves it from the restatement in oracle/eval_np.py, so anything the reference
                   computes THROUGH the knapsack is "reference code + restated solver".
``np.int`` (utils/knapsack.py:14-15) was removed in numpy 1.24; it is restored as an alias of
``int`` for the duration of the import only.
"""
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("SMZ_REFERENCE_ROOT", "")


def available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "summarizer"))


class _DictDataset(dict):
    """h5py.Dataset stand-in: ``d[...]`` / ``d[()]`` return the stored array/scalar."""


class _Field:
    def __init__(self, value):
        self.value = value

    def __getitem__(self, idx):
        if idx is Ellipsis:
            return np.array(self.value, copy=True)
        if idx == ():
            return self.value
        return np.asarray(self.value)[idx]


class DictFile:
    """h5py.File stand-in over {video_key: {field: ndarray}} (read-only use)."""
    registry = {}

    def __init__(self, path, mode="r"):
        self._data = DictFile.registry[path]

    def __getitem__(self, key):
        return {k: _Field(v) for k, v in self._data[key].items()}

    def keys(self):
        return self._data.keys()


class _KnapsackSolver:
    KNAPSACK_DYNAMIC_PROGRAMMING_SOLVER = 2

    def __init__(self, kind, name):
        assert kind == self.KNAPSACK_DYNAMIC_PROGRAMMING_SOLVER

    def Init(self, profits, weights, capacities):
        self._p, self._w, self._c = profits, weights[0], capacities[0]

    def Solve(self):
        from oracle.eval_np import knapsack_dp_takebits
        self._best = set(knapsack_dp_takebits(self._p, self._w, self._c))
        return sum(self._p[i] for i in self._best)

    def BestSolutionContains(self, i):
        return i in self._best


_loaded = {}


def load():
    """Returns a namespace with the reference modules (cached)."""
    if _loaded:
        return _loaded["ns"]
    if not available():
        raise RuntimeError("no reference checkout: set SMZ_REFERENCE_ROOT to the root of a sylvainma/Summarizer "
                           "checkout")
    h5 = types.ModuleType("h5py")
    h5.File = DictFile
    sys.modules.setdefault("h5py", h5)
    ort = types.ModuleType("ortools")
    alg = types.ModuleType("ortools.algorithms")
    pw = types.ModuleType("ortools.algorithms.pywrapknapsack_solver")
    pw.KnapsackSolver = _KnapsackSolver
    alg.pywrapknapsack_solver = pw
    ort.algorithms = alg
    sys.modules.setdefault("ortools", ort)
    sys.modules.setdefault("ortools.algorithms", alg)
    sys.modules.setdefault("ortools.algorithms.pywrapknapsack_solver", pw)
    if not hasattr(np, "int"):
        np.int = int  # utils/knapsack.py:14-15

    # The product ships an alias package also called ``summarizer``; make sure the reference
    # one is what gets imported here, under a private name space, then restore sys.modules.
    saved = {k: v for k, v in sys.modules.items() if k == "summarizer" or k.startswith("summarizer.")}
    for k in saved:
        del sys.modules[k]
    alias = [f for f in sys.meta_path if type(f).__name__ == "_AliasFinder"]   # the product's `summarizer` alias
    for f in alias:
        sys.meta_path.remove(f)
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        import importlib
        ns = types.SimpleNamespace()
        ns.eval = importlib.import_module("summarizer.utils.eval")
        ns.knapsack = importlib.import_module("summarizer.utils.knapsack")
        ns.models = importlib.import_module("summarizer.models")
        ns.vasnet = importlib.import_module("summarizer.models.vasnet")
        ns.dsn = importlib.import_module("summarizer.models.dsn")
        ns.sumgan = importlib.import_module("summarizer.models.sumgan")
        ns.logistic = importlib.import_module("summarizer.models.logistic")
        ns.utils = importlib.import_module("summarizer.utils")
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for f in alias:
            sys.meta_path.insert(0, f)
        ref_mods = {k: v for k, v in sys.modules.items() if k == "summarizer" or k.startswith("summarizer.")}
        for k in ref_mods:
            del sys.modules[k]
        sys.modules.update(saved)
    ns._modules = ref_mods
    _loaded["ns"] = ns
    return ns
