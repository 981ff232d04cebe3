"""Helpers to run the UNMODIFIED reference jobs (LibKGE, installed by oracle/install_ref.py into oracle/_ref)
on in-memory synthetic graphs — once as the reference itself (`model: <m>`, job.device cpu) and once through the
kge_b200 plugin (`model: b200_<m>`, job.device cuda), with identical tables and identical batch order."""
from __future__ import annotations

import tempfile

import torch

from kge_b200 import hostenv

MODULES = ["kge.job", "kge.model", "kge.model.embedder", "kge_b200.plugin"]


def synthetic_splits(E, R, n_train, n_valid=40, n_test=40, seed=1):
    def tri(n, sd):
        g = torch.Generator().manual_seed(sd)
        return torch.stack([torch.randint(0, E, (n,), generator=g), torch.randint(0, R, (n,), generator=g),
                            torch.randint(0, E, (n,), generator=g)], 1).int()
    return {"train": tri(n_train, seed), "valid": tri(n_valid, seed + 1), "test": tri(n_test, seed + 2)}


def make_job(model, E, R, D, splits, device="cpu", train_type="1vsAll", loss="bce", batch_size=16, extra=None,
             job_class=None, forward_only=True, imports=()):
    """A reference TrainingJob (with its validation EntityRankingJob) over an in-memory dataset."""
    hostenv.import_kge()
    from kge import Config, Dataset
    from kge.job import Job

    config = Config()
    config.folder = tempfile.mkdtemp()
    config.set("console.quiet", True)
    config.set("modules", MODULES)
    config.set("model", model)
    config._import(model)
    for extra_model in imports:           # e.g. the base model of reciprocal_relations_model
        config._import(extra_model)
    config.set("dataset.name", "synthetic")
    config.set("dataset.num_entities", E)
    config.set("dataset.num_relations", R)
    config.set("dataset.pickle", False)
    config.set("job.device", device)
    config.set("job.type", "train")
    config.set("train.type", train_type)
    config.set("train.loss", loss)
    config.set("train.batch_size", batch_size)
    config.set("eval.batch_size", 8)
    config.set_all({"lookup_embedder.dim": D})
    if job_class:
        config.set(f"{train_type}.class_name", job_class)
    if extra:
        config.set_all(extra)
    ds = Dataset(config, None)
    ds._triples = dict(splits)
    ds._meta = {"entity_ids": [f"e{i}" for i in range(E)], "relation_ids": [f"r{i}" for i in range(R)]}
    job = Job.create(config, ds)
    if forward_only:
        job.is_forward_only = True
    return job


def copy_tables(src_job, dst_job):
    with torch.no_grad():
        for get in ("get_s_embedder", "get_p_embedder"):
            a = getattr(src_job.model, get)()._embeddings.weight
            b = getattr(dst_job.model, get)()._embeddings.weight
            b.copy_(a.to(b.device))


def run_forward_epoch(job, seed=1):
    """One forward-only epoch with a fixed batch order; returns the epoch trace entry."""
    if job.loader is None:
        job._prepare()
    seed_all(seed)
    return job.run_epoch()


def seed_all(seed):
    """torch (batch order, uniform sampling) + python/numpy RNGs (shared negative sampling, sampler.py:620-680)."""
    import random

    import numpy as np

    torch.manual_seed(seed)
    random.seed(seed)
    np.random.seed(seed)


def run_valid(job):
    ev = job.valid_job
    ev._prepare()
    return ev._run()
