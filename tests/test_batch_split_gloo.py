"""`user.b200_batch_split` of the job plugins with world_size = 2 on CPU (gloo): every rank scores its rows of each
batch, the dense table gradients and the batch loss are all-reduced, and the replicas take identical optimizer steps —
the two-process run must reproduce the single-process run of the same job (loss trajectory and final tables).  The
engine is the oracle-backed stand-in (tests/engine_stub.py); tests/test_gpu_sharded.py runs the CUDA path."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from kge_b200 import hostenv

pytestmark = pytest.mark.skipif(not hostenv.available(), reason="LibKGE not installed (oracle/install_ref.py)")

HERE = os.path.dirname(os.path.abspath(__file__))
E, R, D = 53, 4, 16
CASES = {
    "1vsAll": dict(model="complex", train_type="1vsAll", loss="kl", batch_size=30, job_class="B200TrainingJob1vsAll"),
    "KvsAll": dict(model="distmult", train_type="KvsAll", loss="bce", batch_size=15, job_class="B200TrainingJobKvsAll"),
    "negative_sampling": dict(model="complex", train_type="negative_sampling", loss="bce", batch_size=30,
                              job_class="B200TrainingJobNegativeSampling",
                              extra={"negative_sampling.num_samples.s": 6, "negative_sampling.num_samples.o": 5}),
}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _train(case, split):
    """Two epochs of the plugin job; returns (avg_loss per epoch, entity table, relation table)."""
    sys.path.insert(0, HERE)
    import engine_stub
    import jobs_util as ju

    kw = dict(CASES[case])
    model = kw.pop("model")
    extra = dict(kw.pop("extra", {}))
    extra["user.b200_batch_split"] = split
    splits = ju.synthetic_splits(E, R, 150, 20, 20)
    with engine_stub.installed():
        torch.manual_seed(0)
        init = ju.make_job(model, E, R, D, splits, **{k: v for k, v in kw.items() if k != "job_class"})
        job = ju.make_job("b200_" + model, E, R, D, splits, forward_only=False, extra=extra, **kw)
        ju.copy_tables(init, job)
        losses = []
        for ep in range(2):
            job.epoch += 1
            if job.loader is None:
                job._prepare()
            ju.seed_all(10 + ep)
            losses.append(job.run_epoch()["avg_loss"])
    return (losses, job.model.get_s_embedder()._embeddings.weight.detach().clone(),
            job.model.get_p_embedder()._embeddings.weight.detach().clone())


def _worker(rank, world, port, case, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        losses, ent, rel = _train(case, True)
        both = [None, None]
        dist.all_gather_object(both, (losses, ent, rel))
        assert torch.equal(both[0][1], both[1][1]) and torch.equal(both[0][2], both[1][2]), "replicas diverged"
        assert both[0][0] == both[1][0]
        if rank == 0:
            torch.save({"losses": losses, "ent": ent, "rel": rel}, out)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case", list(CASES))
def test_two_ranks_reproduce_the_single_process_job(case, tmp_path):
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, _free_port(), case, out), nprocs=2, join=True)
    got = torch.load(out)
    losses, ent, rel = _train(case, False)
    assert got["losses"] == pytest.approx(losses, rel=1e-5)
    assert losses[1] < losses[0]
    for a, b in ((got["ent"], ent), (got["rel"], rel)):
        assert float((a - b).abs().max()) <= 1e-5 * float(b.abs().max())


def test_option_without_process_group_is_single_process():
    losses, _, _ = _train("1vsAll", True)          # no group initialised: the whole batch stays on this process
    ref, _, _ = _train("1vsAll", False)
    assert losses == ref


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("batch_size", [1, 7, 30, 64])
def test_rank_slices_partition_every_subbatch(world, batch_size):
    """The ranks' row ranges tile [0, B) exactly — also inside sub-batches and when B < world."""
    hostenv.import_kge()
    from kge_b200.plugin.jobs import _BatchSplit

    class Probe(_BatchSplit):
        def __init__(self, rank):
            self._b200_rank_world = (rank, world)

    for sub in (batch_size, 5, 16):
        seen = []
        for start in range(0, batch_size, sub):
            sl = slice(start, min(start + sub, batch_size))
            for rank in range(world):
                mine = Probe(rank)._b200_my_rows(sl, batch_size)
                if mine is not None:
                    assert sl.start <= mine.start < mine.stop <= sl.stop
                    seen.extend(range(mine.start, mine.stop))
        assert sorted(seen) == list(range(batch_size))
