"""The LibKGE plugin loads through the reference's own plugin mechanism (config `modules:` +
`<model>.yaml` class_name, kge/misc.py:13-42, kge_model.py:473-503).  Needs the live reference
(installed into oracle/_ref by oracle/install_ref.py); skipped where it is not installed."""
import pytest
import torch

from oracle import ref_shim

pytestmark = pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")

MODELS = ["complex", "distmult", "simple", "cp", "rescal", "transe", "rotate"]


def _create(model, extra=None):
    ref_shim.import_reference()
    from kge import Config, Dataset
    from kge.model import KgeModel

    config = Config()
    config.folder = None
    config.set("console.quiet", True)
    config.set("modules", ["kge.job", "kge.model", "kge.model.embedder", "kge_b200.plugin"])
    config.set("model", model)
    config._import(model)
    config.set("dataset.name", "synthetic")
    config.set("dataset.num_entities", 30)
    config.set("dataset.num_relations", 4)
    config.set("dataset.pickle", False)
    config.set("job.device", "cpu")
    config.set_all({"lookup_embedder.dim": 8})
    if extra:
        config.set_all(extra)
    ds = Dataset(config, None)
    ds._meta["relation_ids"] = [f"r{i}" for i in range(4)]    # in-memory dataset: no files to read
    ds._meta["entity_ids"] = [f"e{i}" for i in range(30)]
    return KgeModel.create(config, ds), config


@pytest.mark.parametrize("name", MODELS)
def test_plugin_model_loads_with_reference_parameter_names(name):
    m, _ = _create("b200_" + name)
    import kge_b200.plugin as plug

    assert type(m).__name__.startswith("B200")
    assert isinstance(m, getattr(plug, type(m).__name__))
    keys = set(m.state_dict().keys())
    assert "_entity_embedder._embeddings.weight" in keys       # lookup_embedder.py:44
    assert "_relation_embedder._embeddings.weight" in keys
    assert type(m.get_scorer()).__name__.startswith("B200")
    # same relation-embedder sizing rules as the reference models
    D = 8
    want = {"cp": D // 2, "rotate": D // 2, "rescal": D * D}.get(name, D)
    assert m.get_p_embedder()._embeddings.weight.shape == (4, want)


def test_plugin_refuses_cpu_tensors():
    m, _ = _create("b200_complex")
    idx = torch.tensor([0, 1, 2])
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU path"):
            m.score_sp(idx, idx % 4)
        with pytest.raises(RuntimeError, match="no CPU path"):
            m.score_spo(idx, idx % 4, idx)
        with pytest.raises(RuntimeError, match="no CPU path"):
            m.get_scorer().score_emb(torch.zeros(3, 8), torch.zeros(3, 8), torch.zeros(5, 8), "sp_")


def test_reciprocal_relations_model_uses_plugin_scorer():
    m, _ = _create("reciprocal_relations_model",
                   {"reciprocal_relations_model.base_model.type": "b200_distmult"})
    assert type(m._base_model.get_scorer()).__name__ == "B200DistMultScorer"


def test_plugin_options_propagate():
    m, _ = _create("b200_transe", {"b200_transe.l_norm": 2.0, "b200_transe.precision": "3xtf32"})
    sc = m.get_scorer()
    assert sc._b200_l_norm() == 2.0 and sc._b200_precision() == "3xtf32" and sc._b200_name == "transe"
    r, _ = _create("b200_rotate")
    w = r.get_p_embedder()._embeddings.weight
    assert float(w.abs().max()) <= 3.1416 and r.get_scorer()._b200_l_norm() == 1.0     # uniform(-pi, pi) phases
    assert r._normalize_phases is True


def test_native_indexes_serve_the_reference_jobs():
    """The reference's own KvsAll training job (collate + label construction) and entity-ranking job (filter
    label lookup) run on kge_b200's native KvsAllIndex and produce the same traces as on their own index."""
    import tempfile

    ref_shim.import_reference()
    from kge import Config, Dataset
    from kge.job import Job
    import kge_b200.plugin as plugin
    from kge_b200.indexing import KvsAllIndex

    E, R, D = 40, 4, 8
    g = torch.Generator().manual_seed(4)
    tri = lambda n: torch.stack([torch.randint(0, E, (n,), generator=g), torch.randint(0, R, (n,), generator=g),
                                 torch.randint(0, E, (n,), generator=g)], 1).int()
    splits = {"train": tri(120), "valid": tri(15), "test": tri(15)}

    def run(native):
        torch.manual_seed(0)
        config = Config()
        config.folder = tempfile.mkdtemp()
        config.set("console.quiet", True)
        config.set("model", "distmult")
        config._import("distmult")
        config.set("dataset.name", "synthetic")
        config.set("dataset.num_entities", E)
        config.set("dataset.num_relations", R)
        config.set("dataset.pickle", False)
        config.set("job.device", "cpu")
        config.set("job.type", "train")
        config.set("train.type", "KvsAll")
        config.set("train.loss", "kl")
        config.set("train.batch_size", 16)
        config.set("KvsAll.label_smoothing", 0.1)
        config.set("eval.batch_size", 8)
        config.set_all({"lookup_embedder.dim": D})
        ds = Dataset(config, None)
        ds._triples = dict(splits)
        ds._meta = {"entity_ids": [f"e{i}" for i in range(E)], "relation_ids": [f"r{i}" for i in range(R)]}
        if native:
            plugin.install_native_indexes(ds)
        job = Job.create(config, ds)
        job.is_forward_only = True
        job._prepare()
        if native:
            assert all(isinstance(ix, KvsAllIndex) for ix in job.query_indexes)
        torch.manual_seed(1)               # same shuffling of the batches
        loss = job.run_epoch()["avg_loss"]
        ev = job.valid_job
        ev._prepare()
        tr = ev._run()
        return loss, tr["mean_reciprocal_rank_filtered"], tr["mean_rank_filtered"], tr["hits_at_10_filtered"]

    a, b = run(False), run(True)
    assert a[0] == pytest.approx(b[0], rel=1e-6)
    assert a[1:] == b[1:]
