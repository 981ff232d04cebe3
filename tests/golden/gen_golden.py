"""Generate golden vectors by running the LIVE reference (uma-pi1/kge, installed into oracle/_ref by
oracle/install_ref.py).

    python tests/golden/gen_golden.py          # writes tests/golden/*.npz

The reference holds no golden vectors of its own for the scoring path (SURVEY.md 8c), so
these files — outputs of the unmodified reference on seeded inputs — are what pins the
oracle (tests/test_oracle_golden.py) and, through it and directly, the CUDA path
(tests/test_gpu_*.py).  The tests need no reference installed: the committed .npz
files stand in for it.  Inputs are stored with the outputs so replay needs no RNG parity.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import kge_oracle as orc  # noqa: E402
from oracle import ref_shim  # noqa: E402

S, P, O = 0, 1, 2


def _np(t):
    return t.detach().cpu().numpy()


def gen_scores(model, E, R, D, n, l_norm, sigma, tag):
    ent, rel = orc.make_tables(model, E, R, D, sigma=sigma, seed=1234)
    tri = orc.make_triples(E, R, n, seed=0)
    m, _, _ = ref_shim.make_reference_model(
        model, E, R, D, ent, rel, l_norm=l_norm if model in ("transe", "rotate") else None
    )
    s, p, o = tri[:, S], tri[:, P], tri[:, O]
    g = torch.Generator().manual_seed(7)
    subset = torch.randperm(E, generator=g)[: max(3, E // 3)]
    psub = torch.randperm(R, generator=g)[: max(2, R // 2)]
    with torch.no_grad():
        out = dict(
            ent=_np(ent), rel=_np(rel), triples=_np(tri), subset=_np(subset), psub=_np(psub),
            l_norm=np.float64(l_norm),
            spo=_np(m.score_spo(s, p, o)),
            sp=_np(m.score_sp(s, p)),
            po=_np(m.score_po(p, o)),
            sp_subset=_np(m.score_sp(s, p, subset)),
            po_subset=_np(m.score_po(p, o, subset)),
            so=_np(m.score_so(s, o)),
            so_subset=_np(m.score_so(s, o, psub)),
            sp_po=_np(m.score_sp_po(s, p, o)),
            sp_po_subset=_np(m.score_sp_po(s, p, o, subset)),
        )
    np.savez_compressed(os.path.join(HERE, f"scores_{tag}.npz"), **out)
    print("wrote", tag, {k: v.shape for k, v in out.items() if hasattr(v, "shape")})


def gen_losses():
    ref_shim.import_reference()
    from kge import Config
    from kge.util.loss import KgeLoss

    g = torch.Generator().manual_seed(11)
    n, E = 9, 57
    scores = torch.randn((n, E), generator=g) * 3.0
    idx = torch.randint(0, E, (n,), generator=g)
    multi = (torch.rand((n, E), generator=g) < 0.08).float()
    multi[torch.arange(n), idx] = 1.0
    smooth = (1.0 - 0.1) * multi + 1.0 / E  # train_KvsAll.py:260-266
    out = dict(scores=_np(scores), idx=_np(idx), multi=_np(multi), smooth=_np(smooth))

    def make(loss, arg=float("nan")):
        c = Config()
        c.folder = None
        c.set("console.quiet", True)
        c.set("job.device", "cpu")
        c.set("train.loss", loss)
        c.set("train.loss_arg", arg)
        return KgeLoss.create(c)

    out["bce_idx"] = _np(make("bce")(scores, idx))
    out["bce_idx_off2"] = _np(make("bce", 2.0)(scores, idx))
    out["bce_multi"] = _np(make("bce")(scores, multi))
    out["bce_smooth"] = _np(make("bce")(scores, smooth))
    out["kl_idx"] = _np(make("kl")(scores, idx))
    out["kl_multi"] = _np(make("kl")(scores, multi))
    out["kl_smooth"] = _np(make("kl")(scores, smooth))
    np.savez_compressed(os.path.join(HERE, "losses.npz"), **out)
    print("wrote losses")


def gen_ranks():
    ref_shim.import_reference()
    from kge.job import EntityRankingJob

    class _Self:
        tie_rtol = 1e-4
        tie_atol = 1e-5
        tie_handling = "rounded_mean_rank"

    me = _Self()
    me._get_ranks_and_num_ties = lambda a, b: EntityRankingJob._get_ranks_and_num_ties(me, a, b)
    g = torch.Generator().manual_seed(13)
    n, E = 11, 83
    sp = torch.randn((n, E), generator=g) * 2.0
    po = torch.randn((n, E), generator=g) * 2.0
    # exercise ties, near-ties, NaN, +-inf
    sp[0, 3] = sp[0, 5]
    sp[1, 7] = sp[1, 9] * (1 + 5e-5)
    sp[2, 4] = float("nan")
    sp[3, 6] = float("inf")
    po[4, 2] = float("-inf")
    po[5, :] = 1.25
    true_o_idx = torch.randint(0, E, (n,), generator=g)
    true_s_idx = torch.randint(0, E, (n,), generator=g)
    true_o_idx[0], true_o_idx[1], true_o_idx[2] = 5, 9, 4  # true answer is the tied / NaN one
    o_true = sp[torch.arange(n), true_o_idx].clone()
    s_true = po[torch.arange(n), true_s_idx].clone()
    labels = torch.zeros((n, 2 * E))
    mask = torch.rand((n, 2 * E), generator=g) < 0.05
    labels[mask] = float("inf")
    labels[torch.arange(n), true_o_idx] = 0.0  # own answer zeroed :287-290
    labels[torch.arange(n), E + true_s_idx] = 0.0
    out = dict(sp=_np(sp), po=_np(po), labels=_np(labels), o_true=_np(o_true), s_true=_np(s_true),
               true_o_idx=_np(true_o_idx), true_s_idx=_np(true_s_idx))
    r, t = EntityRankingJob._get_ranks_and_num_ties(me, sp, o_true)
    out["raw_o_rank"], out["raw_o_ties"] = _np(r), _np(t)
    r, t = EntityRankingJob._get_ranks_and_num_ties(me, po, s_true)
    out["raw_s_rank"], out["raw_s_ties"] = _np(r), _np(t)
    s_rank, s_ties, o_rank, o_ties, _, _ = EntityRankingJob._filter_and_rank(
        me, sp, po, labels, o_true, s_true
    )
    out.update(filt_s_rank=_np(s_rank), filt_s_ties=_np(s_ties),
               filt_o_rank=_np(o_rank), filt_o_ties=_np(o_ties))
    out["final_o"] = _np(EntityRankingJob._get_ranks(me, o_rank, o_ties))
    np.savez_compressed(os.path.join(HERE, "ranks.npz"), **out)
    print("wrote ranks")


def gen_ns(model, E, R, D, n, K, l_norm, tag):
    ref_shim.import_reference()
    from kge.util.sampler import DefaultBatchNegativeSample

    ent, rel = orc.make_tables(model, E, R, D, sigma=1.0, seed=1234)
    tri = orc.make_triples(E, R, n, seed=3)
    m, config, _ = ref_shim.make_reference_model(
        model, E, R, D, ent, rel, l_norm=l_norm if model in ("transe", "rotate") else None
    )
    g = torch.Generator().manual_seed(5)
    out = dict(ent=_np(ent), rel=_np(rel), triples=_np(tri), l_norm=np.float64(l_norm))
    with torch.no_grad():
        out["pos"] = _np(m.score_spo(tri[:, S], tri[:, P], tri[:, O]))
        for slot, nm in ((S, "s"), (P, "p"), (O, "o")):
            hi = R if slot == P else E
            neg = torch.randint(0, hi, (n, K), generator=g)
            out[f"neg_{nm}"] = _np(neg)
            for impl in ("triple", "batch"):
                config.set("negative_sampling.implementation", impl)
                bns = DefaultBatchNegativeSample(config, "negative_sampling", tri, slot, K, neg)
                out[f"ns_{nm}_{impl}"] = _np(bns.score(m))
    np.savez_compressed(os.path.join(HERE, f"ns_{tag}.npz"), **out)
    print("wrote ns", tag)


def gen_jobs(model, tag):
    """Run the reference's OWN jobs (TrainingJob1vsAll forward-only epoch, EntityRankingJob) on an
    in-memory synthetic graph with seeded tables; record the trace values the oracle must reproduce."""
    import tempfile

    ref_shim.import_reference()
    from kge import Config, Dataset
    from kge.job import Job

    E, R, D = 20, 3, 16          # dense enough that the filters change the ranks

    def triples(n, seed):
        g = torch.Generator().manual_seed(seed)
        return torch.stack([torch.randint(0, E, (n,), generator=g), torch.randint(0, R, (n,), generator=g),
                            torch.randint(0, E, (n,), generator=g)], 1).int()

    out = {}
    splits = {"train": triples(200, 1), "valid": triples(40, 2), "test": triples(40, 3)}
    ent, rel = orc.make_tables(model, E, R, D, sigma=0.5)
    for loss in ("bce", "kl"):
        config = Config()
        config.folder = tempfile.mkdtemp()
        config.set("console.quiet", True)
        config.set("model", model)
        config._import(model)
        config.set("dataset.name", "synthetic")
        config.set("dataset.num_entities", E)
        config.set("dataset.num_relations", R)
        config.set("dataset.pickle", False)
        config.set("job.device", "cpu")
        config.set("job.type", "train")
        config.set("train.type", "1vsAll")
        config.set("train.loss", loss)
        config.set("train.batch_size", 16)
        config.set("eval.batch_size", 8)
        config.set_all({"lookup_embedder.dim": D})
        ds = Dataset(config, None)
        ds._triples = dict(splits)
        ds._meta = {"entity_ids": [f"e{i}" for i in range(E)], "relation_ids": [f"r{i}" for i in range(R)]}
        job = Job.create(config, ds)
        with torch.no_grad():
            job.model.get_s_embedder()._embeddings.weight.copy_(ent)
            job.model.get_p_embedder()._embeddings.weight.copy_(rel)
        job.is_forward_only = True
        job._prepare()
        out[f"avg_loss_{loss}"] = np.float64(job.run_epoch()["avg_loss"])
        if loss == "bce":
            ev = job.valid_job
            ev._prepare()
            tr = ev._run()
            for suffix in ("", "_filtered", "_filtered_with_test"):
                for k in ("mean_rank", "mean_reciprocal_rank", "hits_at_1", "hits_at_3", "hits_at_10"):
                    out["valid_" + k + suffix] = np.float64(tr[k + suffix])
    # KvsAll forward-only epochs (default query types sp_ and _po), with and without label smoothing
    for loss, eps in (("kl", 0.0), ("kl", 0.2), ("bce", 0.2)):
        config = Config()
        config.folder = tempfile.mkdtemp()
        config.set("console.quiet", True)
        config.set("model", model)
        config._import(model)
        config.set("dataset.name", "synthetic")
        config.set("dataset.num_entities", E)
        config.set("dataset.num_relations", R)
        config.set("dataset.pickle", False)
        config.set("job.device", "cpu")
        config.set("job.type", "train")
        config.set("train.type", "KvsAll")
        config.set("train.loss", loss)
        config.set("train.batch_size", 16)
        config.set("KvsAll.label_smoothing", eps)
        config.set_all({"lookup_embedder.dim": D})
        ds = Dataset(config, None)
        ds._triples = dict(splits)
        ds._meta = {"entity_ids": [f"e{i}" for i in range(E)], "relation_ids": [f"r{i}" for i in range(R)]}
        job = Job.create(config, ds)
        with torch.no_grad():
            job.model.get_s_embedder()._embeddings.weight.copy_(ent)
            job.model.get_p_embedder()._embeddings.weight.copy_(rel)
        job.is_forward_only = True
        job._prepare()
        out[f"kvsall_avg_loss_{loss}_{int(eps * 10)}"] = np.float64(job.run_epoch()["avg_loss"])
    out.update(ent=_np(ent), rel=_np(rel), train=_np(splits["train"]), valid=_np(splits["valid"]),
               test=_np(splits["test"]))
    np.savez_compressed(os.path.join(HERE, f"jobs_{tag}.npz"), **out)
    print("wrote jobs", tag, {k: float(v) for k, v in out.items() if np.ndim(v) == 0})


def gen_index():
    """KvsAllIndex (kge/indexing.py) and the sp/po coordinate lookup (kge/job/util.py) of the live reference on
    random triples with duplicate triples, duplicate keys and query keys absent from the index."""
    ref_shim.import_reference()
    from kge.indexing import KvsAllIndex
    from kge.job.util import get_sp_po_coords_from_spo_batch

    g = torch.Generator().manual_seed(21)
    E, R, n = 23, 4, 300
    tri = torch.stack([torch.randint(0, E, (n,), generator=g), torch.randint(0, R, (n,), generator=g),
                       torch.randint(0, E, (n,), generator=g)], 1).int()
    tri[10:20] = tri[0:10]                       # exact duplicate triples
    out = dict(triples=_np(tri), num_entities=np.int64(E))
    idx = {}
    for key, (cols, val) in (("sp", ([S, P], O)), ("po", ([P, O], S)), ("so", ([S, O], P))):
        ix = KvsAllIndex(tri, cols, val, list)
        idx[key] = ix
        out[f"{key}_keys"] = _np(ix._keys)
        out[f"{key}_offsets"] = _np(ix._values_offset)
        out[f"{key}_values"] = _np(ix._values)
    batch = torch.stack([torch.randint(0, E + 3, (40,), generator=g), torch.randint(0, R, (40,), generator=g),
                         torch.randint(0, E + 3, (40,), generator=g)], 1).int()   # some keys do not exist
    batch[:8] = tri[:8]
    out["batch"] = _np(batch)
    out["sp_get_all"] = _np(idx["sp"].get_all(batch[:, [S, P]]))
    out["po_get_all"] = _np(idx["po"].get_all(batch[:, [P, O]]))
    out["sp_po_coords"] = _np(get_sp_po_coords_from_spo_batch(batch, E, idx["sp"], idx["po"]))
    np.savez_compressed(os.path.join(HERE, "index.npz"), **out)
    print("wrote index", {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim})


def gen_ns_job(model, tag):
    """One batch of the reference's TrainingJobNegativeSampling (collate -> _process_batch, forward only) with
    the sampled negatives recorded, for all three slots and a BCE offset (train_negative_sampling.py:64-170)."""
    import tempfile

    ref_shim.import_reference()
    from kge import Config, Dataset
    from kge.job import Job

    E, R, D = 30, 4, 16
    g = torch.Generator().manual_seed(8)
    tri = lambda n: torch.stack([torch.randint(0, E, (n,), generator=g), torch.randint(0, R, (n,), generator=g),
                                 torch.randint(0, E, (n,), generator=g)], 1).int()
    splits = {"train": tri(64), "valid": tri(8), "test": tri(8)}
    ent, rel = orc.make_tables(model, E, R, D, sigma=0.5)
    config = Config()
    config.folder = tempfile.mkdtemp()
    config.set("console.quiet", True)
    config.set("model", model)
    config._import(model)
    config.set("dataset.name", "synthetic")
    config.set("dataset.num_entities", E)
    config.set("dataset.num_relations", R)
    config.set("dataset.pickle", False)
    config.set("job.device", "cpu")
    config.set("job.type", "train")
    config.set("train.type", "negative_sampling")
    config.set("train.loss", "bce")
    config.set("train.loss_arg", 0.5)
    config.set("train.batch_size", 16)
    config.set("negative_sampling.num_samples.s", 5)
    config.set("negative_sampling.num_samples.p", 2)
    config.set("negative_sampling.num_samples.o", 7)
    config.set_all({"lookup_embedder.dim": D})
    ds = Dataset(config, None)
    ds._triples = dict(splits)
    ds._meta = {"entity_ids": [f"e{i}" for i in range(E)], "relation_ids": [f"r{i}" for i in range(R)]}
    torch.manual_seed(3)
    job = Job.create(config, ds)
    with torch.no_grad():
        job.model.get_s_embedder()._embeddings.weight.copy_(ent)
        job.model.get_p_embedder()._embeddings.weight.copy_(rel)
    job.is_forward_only = True
    job._prepare()
    batch = job._get_collate_fun()(list(range(5, 21)))
    res = job._process_batch(0, batch)
    # the same batch once more with the backward pass (train_negative_sampling.py:160-164): table gradients
    job.is_forward_only = False
    job.model.zero_grad()
    job._process_batch(0, batch)
    out = dict(ent=_np(ent), rel=_np(rel), triples=_np(batch["triples"]), avg_loss=np.float64(res.avg_loss),
               size=np.int64(res.size), offset=np.float64(0.5),
               d_ent=_np(job.model.get_s_embedder()._embeddings.weight.grad),
               d_rel=_np(job.model.get_p_embedder()._embeddings.weight.grad))
    for slot, nm in ((S, "s"), (P, "p"), (O, "o")):
        out[f"neg_{nm}"] = _np(batch["negative_samples"][slot].samples())
    np.savez_compressed(os.path.join(HERE, f"nsjob_{tag}.npz"), **out)
    print("wrote nsjob", tag, float(out["avg_loss"]), {k: v.shape for k, v in out.items() if k.startswith("neg")})


PENALTY_CASES = [
    # (tag, model, entity options, relation options)   options: regularize, regularize_weight, p, weighted
    ("complex_l2", "complex", dict(regularize="lp", regularize_weight=0.1, p=2, weighted=False),
     dict(regularize="lp", regularize_weight=0.2, p=2, weighted=False)),
    ("complex_l3w", "complex", dict(regularize="lp", regularize_weight=0.1, p=3, weighted=True),
     dict(regularize="lp", regularize_weight=0.05, p=3, weighted=True)),
    ("complex_n3w", "complex", dict(regularize="n3", regularize_weight=0.3, p=3, weighted=True),
     dict(regularize="n3", regularize_weight=0.2, p=3, weighted=True)),
    ("complex_n3", "complex", dict(regularize="n3", regularize_weight=0.3, p=3, weighted=False),
     dict(regularize="n3", regularize_weight=0.0, p=3, weighted=False)),
    ("distmult_l1w", "distmult", dict(regularize="lp", regularize_weight=0.4, p=1, weighted=True),
     dict(regularize="lp", regularize_weight=0.1, p=2, weighted=False)),
]


def gen_penalties():
    """KgeModel.penalty(batch=...) of the live reference (kge_model.py:603-649, lookup_embedder.py:123-177) and
    the row normalisation hook (lookup_embedder.py:64-69)."""
    E, R, D, n = 37, 5, 16, 40
    out = {}
    for tag, model, eo, ro in PENALTY_CASES:
        ent, rel = orc.make_tables(model, E, R, D, sigma=0.7)
        tri = orc.make_triples(E, R, n, seed=4)
        tri[1] = tri[0]
        extra = {}
        for key, o in (("entity_embedder", eo), ("relation_embedder", ro)):
            extra[f"{model}.{key}.regularize"] = o["regularize"]
            extra[f"{model}.{key}.regularize_weight"] = o["regularize_weight"]
            extra[f"{model}.{key}.regularize_args.p"] = o["p"]
            extra[f"{model}.{key}.regularize_args.weighted"] = o["weighted"]
        m, _, _ = ref_shim.make_reference_model(model, E, R, D, ent, rel, extra=extra)
        pen = m.penalty(batch={"triples": tri})
        out[f"{tag}_total"] = np.float64(sum(float(v) for _, v in pen))
        out[f"{tag}_ent"], out[f"{tag}_rel"], out[f"{tag}_triples"] = _np(ent), _np(rel), _np(tri)
    ent, _ = orc.make_tables("transe", E, R, D, sigma=0.7)
    for pn in (1.0, 2.0):
        m, _, _ = ref_shim.make_reference_model("transe", E, R, D, ent, None, l_norm=1.0,
                                                extra={"transe.entity_embedder.normalize.p": pn})
        m.get_s_embedder()._normalize_embeddings()
        out[f"normalize_p{int(pn)}"] = _np(m.get_s_embedder()._embeddings.weight)
    out["normalize_in"] = _np(ent)
    np.savez_compressed(os.path.join(HERE, "penalties.npz"), **out)
    print("wrote penalties", {k: float(v) for k, v in out.items() if np.ndim(v) == 0})


def gen_reciprocal(base, tag):
    """ReciprocalRelationsModel over `base` (reciprocal_relations_model.py): relation table with 2R rows."""
    E, R, D, n = 53, 4, 16, 11
    ent, rel2 = orc.make_tables(base, E, 2 * R, D, sigma=0.8)
    tri = orc.make_triples(E, R, n, seed=6)
    m, _, _ = ref_shim.make_reference_model(
        "reciprocal_relations_model", E, R, D, ent, rel2,
        extra={"reciprocal_relations_model.base_model.type": base}, imports=[base])
    s, p, o = tri[:, S], tri[:, P], tri[:, O]
    sub = torch.randperm(E, generator=torch.Generator().manual_seed(2))[:17]
    with torch.no_grad():
        out = dict(ent=_np(ent), rel2=_np(rel2), triples=_np(tri), subset=_np(sub), num_relations=np.int64(R),
                   spo_o=_np(m.score_spo(s, p, o, "o")), spo_s=_np(m.score_spo(s, p, o, "s")),
                   sp=_np(m.score_sp(s, p)), po=_np(m.score_po(p, o)), po_subset=_np(m.score_po(p, o, sub)),
                   sp_po=_np(m.score_sp_po(s, p, o)), sp_po_subset=_np(m.score_sp_po(s, p, o, sub)))
    np.savez_compressed(os.path.join(HERE, f"reciprocal_{tag}.npz"), **out)
    print("wrote reciprocal", tag)


def gen_grads(model, D, loss, tag):
    """Entity / relation table gradients of one 1vsAll step of the LIVE reference: loss(score_sp, o)/n and
    loss(score_po, s)/n with sum reduction, backward through the reference's own autograd graph
    (train_1vsAll.py:59-82)."""
    ref_shim.import_reference()
    from kge import Config
    from kge.util.loss import KgeLoss

    E, R, n = 83, 5, 17
    ent, rel = orc.make_tables(model, E, R, D, sigma=0.5)
    tri = orc.make_triples(E, R, n, seed=9)
    m, _, _ = ref_shim.make_reference_model(model, E, R, D, ent, rel, l_norm=1.0 if model in ("transe", "rotate") else None)
    m.train()
    c = Config()
    c.folder = None
    c.set("console.quiet", True)
    c.set("job.device", "cpu")
    c.set("train.loss", loss)
    offset = 1.5 if loss == "bce" else float("nan")
    c.set("train.loss_arg", offset)
    fn = KgeLoss.create(c)
    s, p, o = tri[:, S], tri[:, P], tri[:, O]
    l_sp = fn(m.score_sp(s, p), o) / n
    l_sp.backward()
    l_po = fn(m.score_po(p, o), s) / n
    l_po.backward()
    out = dict(ent=_np(ent), rel=_np(rel), triples=_np(tri), loss=np.float64(float(l_sp) + float(l_po)),
               offset=np.float64(0.0 if loss == "kl" else offset),
               d_ent=_np(m.get_s_embedder()._embeddings.weight.grad),
               d_rel=_np(m.get_p_embedder()._embeddings.weight.grad))
    np.savez_compressed(os.path.join(HERE, f"grads_{tag}.npz"), **out)
    print("wrote grads", tag, float(out["loss"]))


def gen_mid(model, E=5003, R=11, D=128, n=300, ncols=64):
    """Mid-size outputs of the live reference (several K chunks and several tiles of the tensor-core kernels): the
    tables are regenerated from seeds at replay time (kge_b200.synthetic / the oracle share the generator), only
    sampled score columns, row sums and the row-wise scores are stored."""
    if model == "rescal":
        D = 48
    ent, rel = orc.make_tables(model, E, R, D, sigma=0.5, seed=4321)
    tri = orc.make_triples(E, R, n, seed=17)
    m, _, _ = ref_shim.make_reference_model(model, E, R, D, ent, rel)
    s, p, o = tri[:, S], tri[:, P], tri[:, O]
    cols = torch.sort(torch.randperm(E, generator=torch.Generator().manual_seed(23))[:ncols]).values
    with torch.no_grad():
        sp, po = m.score_sp(s, p), m.score_po(p, o)
        out = dict(E=np.int64(E), R=np.int64(R), D=np.int64(D), n=np.int64(n), cols=_np(cols),
                   sp_cols=_np(sp[:, cols]), po_cols=_np(po[:, cols]),
                   sp_rowsum=_np(sp.double().sum(1)), po_rowsum=_np(po.double().sum(1)),
                   sp_rms=np.float64(sp.double().pow(2).mean().sqrt()), po_rms=np.float64(po.double().pow(2).mean().sqrt()),
                   spo=_np(m.score_spo(s, p, o)))
    np.savez_compressed(os.path.join(HERE, f"mid_{model}.npz"), **out)
    print("wrote mid", model, {k: getattr(v, "shape", v) for k, v in out.items()})


def main():
    torch.manual_seed(0)
    E, R, n = 97, 7, 13
    for model in orc.MODELS:
        D = 16 if model == "rescal" else 32
        gen_scores(model, E, R, D, n, 1.0, 1.0, model)
    gen_scores("transe", E, R, 32, n, 2.0, 1.0, "transe_l2")
    gen_scores("rotate", E, R, 32, n, 2.0, 1.0, "rotate_l2")
    gen_scores("complex", 301, 5, 64, 33, 1.0, 0.1, "complex_sigma01")
    gen_losses()
    gen_ranks()
    for model in ("complex", "rotate", "transe", "rescal"):
        gen_ns(model, 61, 5, 16 if model == "rescal" else 32, 6, 10, 1.0, model)
    for model in ("complex", "transe"):
        gen_jobs(model, model)
    gen_index()
    gen_penalties()
    for base in ("complex", "transe"):
        gen_reciprocal(base, base)
    for model in ("complex", "rotate"):
        gen_ns_job(model, model)
    for model in orc.MODELS:
        gen_grads(model, 8 if model == "rescal" else 16, "bce", f"{model}_bce")
    gen_grads("complex", 16, "kl", "complex_kl")
    gen_grads("rescal", 8, "kl", "rescal_kl")
    for model in orc.MODELS:
        gen_mid(model)


if __name__ == "__main__":
    main()
