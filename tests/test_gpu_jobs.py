"""SURVEY 8(b): the UNMODIFIED reference jobs run on CUDA through the kge_b200 plugin.

For every case the same job is run twice on the same in-memory graph with the same tables and batch order:
  (ref)  the reference itself:  model: <m>,       job.device: cpu
  (b200) through the plugin:    model: b200_<m>,  job.device: cuda   [+ optionally <type>.class_name: B200TrainingJob*]
and the trace values are compared (avg_loss 1e-4 relative; ranking metrics: ranks agree for >= 99.5 % of the
triples, which at these sizes means identical metrics).  Needs the reference installed in oracle/_ref
(oracle/install_ref.py, run by build() when the LibKGE source tree is present) and a B200.
"""
import pytest
import torch

from kge_b200 import hostenv

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not hostenv.available(), reason="LibKGE not installed (oracle/install_ref.py)")]

import jobs_util as ju  # noqa: E402

MODELS = ["complex", "distmult", "simple", "cp", "rescal", "transe", "rotate"]
E, R, D = 211, 5, 32
REL = 1e-4


@pytest.fixture(scope="module")
def splits():
    return ju.synthetic_splits(E, R, 600, 60, 60)


def _pair(model, splits, **kw):
    torch.manual_seed(0)
    ref = ju.make_job(model, E, R, D, splits, device="cpu", **{k: v for k, v in kw.items() if k != "job_class"})
    dev = ju.make_job("b200_" + model, E, R, D, splits, device="cuda", **kw)
    ju.copy_tables(ref, dev)
    return ref, dev


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("loss", ["bce", "kl"])
def test_unmodified_1vsall_job(model, loss, splits):
    """TrainingJob1vsAll (train_1vsAll.py:48-82), forward-only epoch: model.score_sp / score_po + KgeLoss."""
    ref, dev = _pair(model, splits, train_type="1vsAll", loss=loss, batch_size=64)
    assert type(dev).__name__ == "TrainingJob1vsAll" and type(dev.model).__name__.startswith("B200")
    a = ju.run_forward_epoch(ref)["avg_loss"]
    b = ju.run_forward_epoch(dev)["avg_loss"]
    assert b == pytest.approx(a, rel=REL)


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("loss", ["bce", "kl"])
def test_fused_1vsall_job(model, loss, splits):
    """B200TrainingJob1vsAll selected through `1vsAll.class_name` (train.py:127-137): same trace, fused step."""
    from kge_b200 import engine

    ref, dev = _pair(model, splits, train_type="1vsAll", loss=loss, batch_size=64,
                     job_class="B200TrainingJob1vsAll")
    assert type(dev).__name__ == "B200TrainingJob1vsAll"
    a = ju.run_forward_epoch(ref)["avg_loss"]
    engine.launch_count(reset=True)
    tr = ju.run_forward_epoch(dev)
    assert engine.launch_count() > 0
    assert tr["avg_loss"] == pytest.approx(a, rel=REL)
    # sub-batching changes nothing (tests/test_train.py:33-53 of the reference)
    dev.config.set("train.subbatch_size", 24)
    dev._max_subbatch_size = 24
    assert ju.run_forward_epoch(dev)["avg_loss"] == pytest.approx(a, rel=REL)


@pytest.mark.parametrize("model", ["complex", "rescal", "transe"])
@pytest.mark.parametrize("loss,eps", [("kl", 0.0), ("kl", 0.2), ("bce", 0.0), ("bce", 0.2)])
def test_kvsall_jobs(model, loss, eps, splits):
    """TrainingJobKvsAll unmodified (dense labels built by the reference, scores by the plugin) and the fused
    B200TrainingJobKvsAll (CSR labels)."""
    extra = {"KvsAll.label_smoothing": eps}
    ref, dev = _pair(model, splits, train_type="KvsAll", loss=loss, batch_size=32, extra=extra)
    a = ju.run_forward_epoch(ref)["avg_loss"]
    assert ju.run_forward_epoch(dev)["avg_loss"] == pytest.approx(a, rel=REL)
    if eps > 0 and model == "transe":
        return      # label smoothing over CSR labels needs the dot family's column-sum identity
    _, fused = _pair(model, splits, train_type="KvsAll", loss=loss, batch_size=32, extra=extra,
                     job_class="B200TrainingJobKvsAll")
    assert type(fused).__name__ == "B200TrainingJobKvsAll"
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)
    fused._max_subbatch_size = 10
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)


@pytest.mark.parametrize("model", ["complex", "transe", "rotate"])
@pytest.mark.parametrize("impl", ["triple", "batch"])
def test_negative_sampling_jobs(model, impl, splits):
    """TrainingJobNegativeSampling unmodified (both sampler implementations) and the fused job; the samples are
    drawn by the reference's CPU sampler in the main process, so both runs see the same negatives."""
    extra = {"negative_sampling.implementation": impl, "negative_sampling.num_samples.s": 7,
             "negative_sampling.num_samples.o": 9, "negative_sampling.num_samples.p": 3,
             "train.loss_arg": 2.0}
    ref, dev = _pair(model, splits, train_type="negative_sampling", loss="bce", batch_size=32, extra=extra)
    a = ju.run_forward_epoch(ref)["avg_loss"]
    assert ju.run_forward_epoch(dev)["avg_loss"] == pytest.approx(a, rel=REL)
    _, fused = _pair(model, splits, train_type="negative_sampling", loss="bce", batch_size=32, extra=extra,
                     job_class="B200TrainingJobNegativeSampling")
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)


@pytest.mark.parametrize("model", MODELS)
def test_unmodified_entity_ranking_job(model, splits):
    """EntityRankingJob (eval_entity_ranking.py:103-487): score_sp/score_po on the unique targets for the true
    scores, score_sp_po per chunk, its own tie-handling consistency check — all on the plugin model."""
    ref, dev = _pair(model, splits, train_type="1vsAll", loss="kl", batch_size=64,
                     extra={"entity_ranking.chunk_size": 64, "entity_ranking.filter_with_test": True})
    a, b = ju.run_valid(ref), ju.run_valid(dev)
    for suffix in ("", "_filtered", "_filtered_with_test"):
        for k in ("mean_rank", "mean_reciprocal_rank", "hits_at_1", "hits_at_3", "hits_at_10"):
            assert b[k + suffix] == pytest.approx(a[k + suffix], rel=5e-3, abs=5e-3), (k + suffix)
    assert b["mean_reciprocal_rank_filtered"] == pytest.approx(a["mean_reciprocal_rank_filtered"], rel=2e-3)


@pytest.mark.parametrize("model", ["complex", "transe", "rotate"])
def test_training_epoch_through_plugin(model, splits):
    """Two full training epochs (forward, backward, Adagrad step) of the unmodified job and of the fused job move
    the tables as the reference does: same avg_loss in epoch 1 AND in epoch 2 (i.e. after the updates)."""
    torch.manual_seed(0)
    init = ju.make_job(model, E, R, D, splits, device="cpu", train_type="1vsAll", loss="kl", batch_size=64)
    losses = {}
    for tag, kw, dev in (("ref", {}, "cpu"), ("plugin", {}, "cuda"),
                         ("fused", {"job_class": "B200TrainingJob1vsAll"}, "cuda")):
        name = model if tag == "ref" else "b200_" + model
        job = ju.make_job(name, E, R, D, splits, device=dev, train_type="1vsAll", loss="kl", batch_size=64,
                          forward_only=False, **kw)
        ju.copy_tables(init, job)
        out = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            out.append(job.run_epoch()["avg_loss"])
        losses[tag] = out
    assert losses["ref"][1] < losses["ref"][0]
    for tag in ("plugin", "fused"):
        assert losses[tag][0] == pytest.approx(losses["ref"][0], rel=REL)
        assert losses[tag][1] == pytest.approx(losses["ref"][1], rel=1e-3)


@pytest.mark.parametrize("model", ["complex", "distmult", "simple", "cp", "rescal", "transe", "rotate"])
@pytest.mark.parametrize("loss", ["kl", "bce"])
def test_training_epoch_native_backward(model, loss, splits):
    """The fused job with the gradient kernels of libb200kge (b200kge_train_1vsall_backward: recompute, G planes,
    two split-K tensor-core GEMMs, unfold; TransE / RotatE: the row-gradient passes of grad_distance.cu) instead of the
    reference's autograd: two epochs track the reference."""
    torch.manual_seed(0)
    init = ju.make_job(model, E, R, D, splits, device="cpu", train_type="1vsAll", loss=loss, batch_size=64)
    losses = {}
    for tag, dev in (("ref", "cpu"), ("native", "cuda")):
        name = model if tag == "ref" else "b200_" + model
        kw = {"job_class": "B200TrainingJob1vsAll"} if tag == "native" else {}
        job = ju.make_job(name, E, R, D, splits, device=dev, train_type="1vsAll", loss=loss, batch_size=64,
                          forward_only=False, **kw)
        if tag == "native":
            job.model.b200_backward = "native"
        ju.copy_tables(init, job)
        out = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            out.append(job.run_epoch()["avg_loss"])
        losses[tag] = out
    assert losses["native"][0] == pytest.approx(losses["ref"][0], rel=REL)
    assert losses["native"][1] == pytest.approx(losses["ref"][1], rel=1e-3)


@pytest.mark.parametrize("model,extra", [
    ("complex", {"entity_embedder.regularize": "n3", "entity_embedder.regularize_weight": 0.05,
                 "entity_embedder.regularize_args.weighted": True,
                 "relation_embedder.regularize": "lp", "relation_embedder.regularize_weight": 0.01}),
    ("distmult", {"entity_embedder.regularize": "lp", "entity_embedder.regularize_weight": 0.02,
                  "entity_embedder.regularize_args.p": 3, "entity_embedder.regularize_args.weighted": True}),
    ("transe", {"entity_embedder.normalize.p": 2.0, "relation_embedder.regularize": "lp",
                "relation_embedder.regularize_weight": 0.01}),
])
def test_training_with_penalties_and_normalisation(model, extra, splits):
    """SURVEY 8f-3 through the jobs: Lp / N3 penalties (weighted and unweighted; forward by the row kernel, backward by
    autograd of the reference expression) and the post-batch row normalisation hook on the plugin model reproduce the
    reference's avg_penalty / avg_cost over two training epochs."""
    torch.manual_seed(0)
    init = ju.make_job(model, E, R, D, splits, device="cpu", train_type="1vsAll", loss="kl", batch_size=64)
    traces = {}
    for tag, dev in (("ref", "cpu"), ("plugin", "cuda")):
        name = model if tag == "ref" else "b200_" + model
        ex = {f"{name}.{k}": v for k, v in extra.items()}
        kw = {"job_class": "B200TrainingJob1vsAll"} if tag == "plugin" else {}
        job = ju.make_job(name, E, R, D, splits, device=dev, train_type="1vsAll", loss="kl", batch_size=64,
                          forward_only=False, extra=ex, **kw)
        ju.copy_tables(init, job)
        if tag == "plugin":
            assert getattr(job.model.get_s_embedder(), "_b200_patched", False)
        out = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
                for f in job.pre_run_hooks:          # Job.run() would call these (initial normalisation)
                    f(job)
            ju.seed_all(10 + ep)
            tr = job.run_epoch()
            out.append((tr["avg_loss"], tr["avg_penalty"], tr["avg_cost"]))
        traces[tag] = out
    for ep in range(2):
        for a, b in zip(traces["plugin"][ep], traces["ref"][ep]):
            assert a == pytest.approx(b, rel=1e-3 if ep else REL, abs=1e-7)


@pytest.mark.parametrize("model", ["complex", "transe", "rotate"])
def test_negative_sampling_training_native_backward(model, splits):
    """B200TrainingJobNegativeSampling in TRAINING mode: per slot one autograd node whose backward is the fused NS
    gradient kernel (b200kge_ns_backward); two epochs (forward, backward, Adagrad) track the reference job, which draws
    the same negatives from the same CPU sampler."""
    extra = {"negative_sampling.num_samples.s": 11, "negative_sampling.num_samples.o": 13, "train.loss_arg": 1.0,
             "negative_sampling.implementation": "triple"}
    torch.manual_seed(0)
    init = ju.make_job(model, E, R, D, splits, device="cpu", train_type="negative_sampling", loss="bce", batch_size=64,
                       extra=extra)
    losses = {}
    for tag, dev in (("ref", "cpu"), ("native", "cuda")):
        name = model if tag == "ref" else "b200_" + model
        kw = {"job_class": "B200TrainingJobNegativeSampling"} if tag == "native" else {}
        job = ju.make_job(name, E, R, D, splits, device=dev, train_type="negative_sampling", loss="bce", batch_size=64,
                          forward_only=False, extra=extra, **kw)
        ju.copy_tables(init, job)
        out = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            out.append(job.run_epoch()["avg_loss"])
        losses[tag] = out
    assert losses["ref"][1] < losses["ref"][0]
    assert losses["native"][0] == pytest.approx(losses["ref"][0], rel=REL)
    assert losses["native"][1] == pytest.approx(losses["ref"][1], rel=1e-3)


@pytest.mark.parametrize("base", ["distmult", "complex"])
def test_reciprocal_relations_model_through_plugin(base, splits):
    """The reference's own ReciprocalRelationsModel wrapper (reciprocal_relations_model.py:85-124: score_po as sp_ with a
    relation offset; it calls the scorer's score_emb directly) over a b200 base model: two 1vsAll training epochs and
    the entity-ranking job agree with the same wrapper over the reference base model."""
    def make(bm, dev):
        return ju.make_job("reciprocal_relations_model", E, R, D, splits, device=dev, train_type="1vsAll", loss="kl",
                           batch_size=64, forward_only=False, imports=(bm,),
                           extra={"reciprocal_relations_model.base_model.type": bm})
    torch.manual_seed(0)
    init = make(base, "cpu")
    out = {}
    for tag, dev, bm in (("ref", "cpu", base), ("plugin", "cuda", "b200_" + base)):
        job = make(bm, dev)
        with torch.no_grad():
            for a, b in zip(init.model.parameters(), job.model.parameters()):
                b.copy_(a.to(b.device))
        if tag == "plugin":
            assert type(job.model._base_model.get_scorer()).__name__.startswith("B200")
        losses = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(20 + ep)
            losses.append(job.run_epoch()["avg_loss"])
        out[tag] = (losses, ju.run_valid(job))
    assert out["plugin"][0][0] == pytest.approx(out["ref"][0][0], rel=REL)
    assert out["plugin"][0][1] == pytest.approx(out["ref"][0][1], rel=1e-3)
    for k in ("mean_reciprocal_rank_filtered", "hits_at_10_filtered", "mean_rank"):
        assert out["plugin"][1][k] == pytest.approx(out["ref"][1][k], rel=1e-2, abs=1e-2)


@pytest.mark.parametrize("model", ["complex", "rescal"])
@pytest.mark.parametrize("loss,eps", [("kl", 0.0), ("kl", 0.2), ("bce", 0.1)])
def test_kvsall_training_native_backward(model, loss, eps, splits):
    """B200TrainingJobKvsAll in TRAINING mode: CSR labels in the forward epilogue and in the gradient planes
    (b200kge_score_1vsN_loss_csr_backward); two epochs (forward, backward, Adagrad) track the reference job."""
    extra = {"KvsAll.label_smoothing": eps}
    torch.manual_seed(0)
    init = ju.make_job(model, E, R, D, splits, device="cpu", train_type="KvsAll", loss=loss, batch_size=32, extra=extra)
    losses = {}
    for tag, dev in (("ref", "cpu"), ("native", "cuda")):
        name = model if tag == "ref" else "b200_" + model
        kw = {"job_class": "B200TrainingJobKvsAll"} if tag == "native" else {}
        job = ju.make_job(name, E, R, D, splits, device=dev, train_type="KvsAll", loss=loss, batch_size=32,
                          forward_only=False, extra=extra, **kw)
        ju.copy_tables(init, job)
        out = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            out.append(job.run_epoch()["avg_loss"])
        losses[tag] = out
    assert losses["native"][0] == pytest.approx(losses["ref"][0], rel=REL)
    assert losses["native"][1] == pytest.approx(losses["ref"][1], rel=1e-3)
