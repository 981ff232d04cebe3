"""Import the live reference (uma-pi1/kge, installed into oracle/_ref by oracle/install_ref.py).

TEST INFRASTRUCTURE.  Used only by tests/golden/gen_golden.py (to produce the committed
golden vectors) and by CPU tests that are skipped when the reference is not installed.
Nothing is copied from the reference into the repository: it is imported
read-only, with the five optional third-party modules it imports at module level but
never touches on the scoring path (`path`, `igraph`, `ConfigSpace`, `ax`, `hpbandster`;
SURVEY.md 8c) replaced by empty stub modules.
"""
from __future__ import annotations

import importlib.abc
import importlib.machinery
import os
import sys
import types
import warnings

REFERENCE_ROOT = os.environ.get("KGE_REFERENCE_ROOT",
                                os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


class _StubModule(types.ModuleType):
    __path__: list = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return type(name, (object,), {})


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    roots = {"path", "igraph", "ConfigSpace", "ax", "hpbandster", "sqlalchemy", "torchviz"}

    def find_spec(self, name, path, target=None):
        if name.split(".")[0] in self.roots:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)
        return None

    def create_module(self, spec):
        return _StubModule(spec.name)

    def exec_module(self, module):
        pass


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "kge"))


_installed = False


def import_reference():
    """Returns the imported reference package `kge` (raises if the tree is absent)."""
    global _installed
    if not available():
        raise ImportError(f"reference tree not found at {REFERENCE_ROOT}")
    if not _installed:
        for root in list(_StubFinder.roots):
            try:
                __import__(root)
                _StubFinder.roots.discard(root)  # the real one exists; do not shadow it
            except Exception:
                pass
        sys.meta_path.insert(0, _StubFinder())
        if REFERENCE_ROOT not in sys.path:
            sys.path.insert(0, REFERENCE_ROOT)
        _installed = True
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import kge  # noqa: F401

        import kge.model  # noqa: F401
        import kge.job  # noqa: F401
    return sys.modules["kge"]


def make_reference_model(model: str, E: int, R: int, D: int, ent=None, rel=None,
                         l_norm: float | None = None, extra: dict | None = None, imports=()):
    """Builds a reference KgeModel on CPU over an in-memory dataset of the given shape and
    (optionally) injects seeded embedding tables."""
    import torch

    kge = import_reference()
    from kge import Config, Dataset
    from kge.model import KgeModel

    config = Config()
    config.folder = None
    config.set("console.quiet", True)
    config.set("model", model)
    config._import(model)
    for extra_model in imports:          # e.g. the base model of reciprocal_relations_model
        config._import(extra_model)
    config.set("dataset.name", "synthetic")
    config.set("dataset.num_entities", E)
    config.set("dataset.num_relations", R)
    config.set("dataset.pickle", False)
    config.set("job.device", "cpu")
    config.set_all({"lookup_embedder.dim": D})
    if l_norm is not None:
        config.set(f"{model}.l_norm", float(l_norm))
    if extra:
        config.set_all(extra)
    dataset = Dataset(config, None)
    # in-memory dataset: no files to read (the reciprocal-relations wrapper looks these up)
    dataset._meta["entity_ids"] = [f"e{i}" for i in range(E)]
    dataset._meta["relation_ids"] = [f"r{i}" for i in range(R)]
    m = KgeModel.create(config, dataset)
    m.eval()
    with torch.no_grad():
        if ent is not None:
            m.get_s_embedder()._embeddings.weight.copy_(ent)
        if rel is not None:
            m.get_p_embedder()._embeddings.weight.copy_(rel)
    return m, config, dataset
