"""Host logic of the LibKGE plugin on CPU: the reference's job factory finds the job plugins, the plugin models
route index-level calls to the engine with the right operands, the fused job steps (CSR construction, sub-batch
scaling, positive-first NS blocks) reproduce the reference job's trace, and the autograd wrappers deliver the
reference's gradients.  kge_b200.engine is replaced by an oracle-backed stand-in (tests/engine_stub.py) — the CUDA
path itself runs the same jobs in tests/test_gpu_jobs.py."""
import pytest
import torch

from kge_b200 import hostenv

pytestmark = pytest.mark.skipif(not hostenv.available(), reason="LibKGE not installed (oracle/install_ref.py)")

import engine_stub  # noqa: E402
import jobs_util as ju  # noqa: E402

E, R, D = 53, 4, 16
REL = 2e-5


@pytest.fixture(scope="module")
def splits():
    return ju.synthetic_splits(E, R, 150, 20, 20)


@pytest.fixture()
def stub():
    with engine_stub.installed():
        yield


def _pair(model, splits, **kw):
    torch.manual_seed(0)
    ref = ju.make_job(model, E, R, D, splits, **{k: v for k, v in kw.items() if k != "job_class"})
    dev = ju.make_job("b200_" + model, E, R, D, splits, **kw)
    ju.copy_tables(ref, dev)
    return ref, dev


@pytest.mark.parametrize("model", ["complex", "cp", "transe"])
@pytest.mark.parametrize("loss", ["bce", "kl"])
def test_1vsall_jobs(model, loss, splits, stub):
    ref, dev = _pair(model, splits, loss=loss, batch_size=32)
    a = ju.run_forward_epoch(ref)["avg_loss"]
    assert ju.run_forward_epoch(dev)["avg_loss"] == pytest.approx(a, rel=REL)
    _, fused = _pair(model, splits, loss=loss, batch_size=32, job_class="B200TrainingJob1vsAll")
    assert type(fused).__name__ == "B200TrainingJob1vsAll"
    engine_stub.launch_count(reset=True)
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)
    assert engine_stub.launch_count() == len(fused.loader)          # ONE fused call per batch
    fused._max_subbatch_size = 10
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)


@pytest.mark.parametrize("loss,eps", [("kl", 0.0), ("kl", 0.2), ("bce", 0.2)])
def test_kvsall_jobs(loss, eps, splits, stub):
    extra = {"KvsAll.label_smoothing": eps}
    ref, dev = _pair("distmult", splits, train_type="KvsAll", loss=loss, batch_size=16, extra=extra)
    a = ju.run_forward_epoch(ref)["avg_loss"]
    assert ju.run_forward_epoch(dev)["avg_loss"] == pytest.approx(a, rel=REL)
    _, fused = _pair("distmult", splits, train_type="KvsAll", loss=loss, batch_size=16, extra=extra,
                     job_class="B200TrainingJobKvsAll")
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)
    fused._max_subbatch_size = 5
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)


@pytest.mark.parametrize("impl", ["triple", "batch"])
@pytest.mark.parametrize("shared", [False, True])
def test_negative_sampling_jobs(impl, shared, splits, stub):
    extra = {"negative_sampling.implementation": impl, "negative_sampling.num_samples.s": 5,
             "negative_sampling.num_samples.o": 6, "negative_sampling.num_samples.p": 2,
             "negative_sampling.shared": shared, "train.loss_arg": 1.5}
    ref, dev = _pair("complex", splits, train_type="negative_sampling", loss="bce", batch_size=16, extra=extra)
    a = ju.run_forward_epoch(ref)["avg_loss"]
    assert ju.run_forward_epoch(dev)["avg_loss"] == pytest.approx(a, rel=REL)
    _, fused = _pair("complex", splits, train_type="negative_sampling", loss="bce", batch_size=16, extra=extra,
                     job_class="B200TrainingJobNegativeSampling")
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)
    fused._max_subbatch_size = 5
    assert ju.run_forward_epoch(fused)["avg_loss"] == pytest.approx(a, rel=REL)


def test_entity_ranking_job(splits, stub):
    ref, dev = _pair("rescal", splits, loss="kl", batch_size=32,
                     extra={"entity_ranking.chunk_size": 20, "entity_ranking.filter_with_test": True})
    a, b = ju.run_valid(ref), ju.run_valid(dev)
    for k in ("mean_rank", "mean_reciprocal_rank_filtered", "hits_at_10_filtered_with_test"):
        assert b[k] == pytest.approx(a[k], rel=1e-6)


@pytest.mark.parametrize("job_class", [None, "B200TrainingJob1vsAll"])
def test_training_epoch_gradients(job_class, splits, stub):
    """Two full training epochs (backward through the autograd wrappers + Adagrad) track the reference."""
    out = {}
    torch.manual_seed(0)
    init = ju.make_job("complex", E, R, D, splits, loss="kl", batch_size=32)
    for tag in ("ref", "plugin"):
        kw = {"job_class": job_class} if (tag == "plugin" and job_class) else {}
        job = ju.make_job("complex" if tag == "ref" else "b200_complex", E, R, D, splits, loss="kl", batch_size=32,
                          forward_only=False, **kw)
        ju.copy_tables(init, job)
        losses = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            losses.append(job.run_epoch()["avg_loss"])
        out[tag] = losses
    assert out["plugin"] == pytest.approx(out["ref"], rel=1e-5)
    assert out["ref"][1] < out["ref"][0]


def test_job_plugins_fall_through_for_reference_models(splits):
    """A job plugin over a non-b200 model runs the reference implementation (no engine involved: no stub here)."""
    ref = ju.make_job("distmult", E, R, D, splits, loss="kl", batch_size=32)
    plug = ju.make_job("distmult", E, R, D, splits, loss="kl", batch_size=32, job_class="B200TrainingJob1vsAll")
    ju.copy_tables(ref, plug)
    assert type(plug).__name__ == "B200TrainingJob1vsAll"
    assert ju.run_forward_epoch(plug)["avg_loss"] == pytest.approx(ju.run_forward_epoch(ref)["avg_loss"], rel=1e-7)


def test_kvsall_training_through_the_job_plugin(splits, stub):
    """B200TrainingJobKvsAll in training mode (autograd node per query type over the CSR labels) tracks the reference."""
    out = {}
    torch.manual_seed(0)
    init = ju.make_job("distmult", E, R, D, splits, train_type="KvsAll", loss="kl", batch_size=16,
                       extra={"KvsAll.label_smoothing": 0.1})
    for tag in ("ref", "plugin"):
        kw = {"job_class": "B200TrainingJobKvsAll"} if tag == "plugin" else {}
        job = ju.make_job("distmult" if tag == "ref" else "b200_distmult", E, R, D, splits, train_type="KvsAll", loss="kl",
                          batch_size=16, forward_only=False, extra={"KvsAll.label_smoothing": 0.1}, **kw)
        ju.copy_tables(init, job)
        losses = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            losses.append(job.run_epoch()["avg_loss"])
        out[tag] = losses
    assert out["plugin"] == pytest.approx(out["ref"], rel=1e-5)
