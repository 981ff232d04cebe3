"""Locate and import the host framework (LibKGE, package `kge`) that kge_b200.plugin plugs into.

The plugin classes subclass the reference's own `KgeModel` / `TrainingJob*` classes, so `kge` must be
importable.  In a LibKGE deployment it simply is (`pip install -e .`).  In this repository's test and bench
environment build() installs the unmodified LibKGE into `oracle/_ref` (git-ignored; oracle/install_ref.py)
when its source tree is present, and a handful of optional third-party modules that `kge` imports at
module level but never touches on the training / evaluation path (`path`, `igraph`, `ConfigSpace`, `ax`,
`hpbandster`, `sqlalchemy`, `torchviz`; SURVEY.md 8c) may be missing: those are replaced by empty stub
modules — the reference code itself is not modified.

Search order for the `kge` tree: `$KGE_REFERENCE_ROOT`, `<repo>/oracle/_ref`, an already importable `kge`.
"""
from __future__ import annotations

import importlib.abc
import importlib.machinery
import importlib.util
import os
import sys
import types
import warnings

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_OPTIONAL = ("path", "igraph", "ConfigSpace", "ax", "hpbandster", "sqlalchemy", "torchviz")


class _StubModule(types.ModuleType):
    __path__: list = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return type(name, (object,), {})


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def __init__(self, roots):
        self.roots = set(roots)

    def find_spec(self, name, path, target=None):
        if name.split(".")[0] in self.roots:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)
        return None

    def create_module(self, spec):
        return _StubModule(spec.name)

    def exec_module(self, module):
        pass


def locate() -> str | None:
    """Directory that contains the `kge` package, or None if `kge` is importable as is / not found."""
    cands = [os.environ.get("KGE_REFERENCE_ROOT"), os.path.join(_REPO, "oracle", "_ref")]
    for c in cands:
        if c and os.path.isdir(os.path.join(c, "kge", "model")):
            return c
    return None


def available() -> bool:
    return locate() is not None or "kge" in sys.modules or importlib.util.find_spec("kge") is not None


_done = False


def import_kge():
    """Imports `kge` (+ kge.model, kge.job) and returns the package."""
    global _done
    if not _done:
        root = locate()
        if root is None and importlib.util.find_spec("kge") is None:
            raise ImportError(
                "LibKGE (`kge`) is not importable: install it, set KGE_REFERENCE_ROOT, or run "
                "oracle/install_ref.py (installs it into oracle/_ref)")
        if root is not None and root not in sys.path:
            sys.path.insert(0, root)
        missing = []
        for name in _OPTIONAL:
            try:
                if importlib.util.find_spec(name) is None:
                    missing.append(name)
            except (ImportError, ValueError):
                missing.append(name)
        if missing:
            sys.meta_path.append(_StubFinder(missing))
        _done = True
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import kge  # noqa: F401
        import kge.job  # noqa: F401
        import kge.model  # noqa: F401
    return sys.modules["kge"]
