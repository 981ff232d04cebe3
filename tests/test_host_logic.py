"""CPU tests of host-side logic that needs no GPU: argument validation in the Python layer, label
packing, relation-dim rules, model construction errors, the reference arm of bench.py."""
import json
import subprocess
import sys
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_relation_dim_rules():
    from kge_b200.model import relation_dim
    from oracle import kge_oracle as orc

    for m in orc.MODELS:
        for D in (8, 32, 200):
            assert relation_dim(m, D) == orc.relation_dim(m, D)
    assert relation_dim("rescal", 200) == 40000 and relation_dim("rotate", 512) == 256


def test_model_construction_errors_match_reference():
    from kge_b200 import KgeModel, KgeLoss

    for name in ("complex", "simple", "cp", "rotate"):
        with pytest.raises(ValueError, match="even dimensionality"):
            KgeModel(name, 10, 2, 7)                      # simple.py:46-50, cp.py:44-48, rotate.py:87-91
    with pytest.raises(ValueError):
        KgeModel("conve", 10, 2, 8)
    with pytest.raises(ValueError, match="invalid value train.loss"):
        KgeLoss.create("soft_margin")                     # loss.py:87-89
    m = KgeModel("rescal", 10, 3, 6, seed=0)
    assert m.state_dict()["_relation_embedder._embeddings.weight"].shape == (3, 36)
    assert set(m.state_dict()) == {"_entity_embedder._embeddings.weight", "_relation_embedder._embeddings.weight"}
    r = KgeModel("rotate", 10, 3, 8, seed=0)
    w = r._relation_embedder.weight
    assert w.shape == (3, 4) and float(w.abs().max()) <= 3.1416


def test_engine_rejects_bad_inputs_before_touching_the_gpu():
    from kge_b200 import engine

    x = torch.zeros(4, 8)
    with pytest.raises(RuntimeError, match="no CPU path"):
        engine.score_spo("complex", x, x, x)
    with pytest.raises(ValueError):
        engine.score_1vsN("complex", "s_o", x, x, x)


def test_bench_reference_arm_runs_on_cpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "triples/s" and line["value"] > 0
    from kge_b200 import hostenv
    # the live reference's own job when it is installed (oracle/install_ref.py), else the oracle's restatement
    assert line["cpu_baseline"]["kind"] == ("reference" if hostenv.available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["config"]["workload"].startswith("ComplEx d=512 1vsAll+BCE")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True


def test_topk_tie_break_is_lowest_index():
    from kge_b200.sharded import _topk_lowest_index

    v = torch.tensor([[1.0, 3.0, 3.0, 2.0, 3.0]])
    vals, idx = _topk_lowest_index(v, 3)
    assert idx.tolist() == [[1, 2, 4]] and vals.tolist() == [[3.0, 3.0, 3.0]]
    ids = torch.tensor([[9, 4, 7, 1, 2]])
    vals, pos = _topk_lowest_index(v, 2, ids)
    assert torch.gather(ids, 1, pos).tolist() == [[2, 4]]      # among the 3.0s, ids 4,7,2 -> 2 then 4


def test_fp16_presplit_scheme_is_fp32_equivalent():
    """Numerics premise of the experimental pre-split kernel (kge_b200/csrc/presplit.cu): per-row power-of-two
    scaling to [2^13, 2^14), hi = fp16(x), lo = fp16(x - hi), three products hi*hi + hi*lo + lo*hi.  Emulated
    here with exact products (fp64): the representation error must sit far below the 1e-4 * rms parity bar for
    any table magnitude, including rows dominated by one outlier."""
    import torch

    def split(x):
        amax = x.abs().amax(1, keepdim=True)
        e = torch.floor(torch.log2(torch.where(amax > 0, amax, torch.full_like(amax, 2.0 ** 13)))).clamp(-60, 60)
        mul = torch.pow(2.0, 13 - e)
        xs = x * mul
        hi = xs.half()
        lo = (xs - hi.float()).half()
        assert torch.isfinite(hi.float()).all()
        return hi.double(), lo.double(), (1.0 / mul).double()

    g = torch.Generator().manual_seed(0)
    for sigma in (1.0, 1e-3, 1e-6):
        q = torch.randn((64, 256), generator=g) * sigma * torch.randn((64, 256), generator=g) * sigma
        t = torch.randn((500, 256), generator=g) * sigma
        t[7, 3] = 1000.0 * sigma          # outlier row: everything else in it loses 10 bits of lo, still fine
        t[8] = 0.0
        ref = q.double() @ t.double().t()
        qh, ql, qs = split(q)
        th, tl, ts = split(t)
        rec = (th + tl) * ts
        assert float((rec - t.double()).abs().max() / t.abs().max()) < 2.0 ** -21
        got = (qh @ th.t() + qh @ tl.t() + ql @ th.t()) * qs * ts.t()
        rms = float(ref.pow(2).mean().sqrt())
        assert float((got - ref).abs().max()) <= 1e-5 * rms, sigma   # an fp32 GEMM itself sits at ~2.5e-6


def test_reciprocal_model_index_arithmetic(monkeypatch):
    """kge_b200.ReciprocalRelationsModel routes every subject-side query through the `sp_` entry points with
    relation p + R (reciprocal_relations_model.py:72-124); checked on CPU with the engine calls recorded."""
    import torch
    import kge_b200
    from kge_b200 import engine

    calls = []

    def fake_1vsN(model, combine, q_tab, rel, cand_tab, q=None, p=None, cand=None, l_norm=1.0, precision="auto", out=None):
        calls.append(("1vsN", combine, q.tolist(), p.tolist(), None if cand is None else cand.tolist()))
        m = cand_tab.shape[0] if cand is None else cand.numel()
        res = torch.full((q.numel(), m), float(len(calls)))
        if out is not None:
            out.copy_(res)
            return out
        return res

    def fake_spo(model, ent_s, rel, ent_o, s=None, p=None, o=None, l_norm=1.0):
        calls.append(("spo", s.tolist(), p.tolist(), o.tolist()))
        return torch.zeros(s.numel())

    monkeypatch.setattr(engine, "score_1vsN", fake_1vsN)
    monkeypatch.setattr(engine, "score_spo", fake_spo)
    m = kge_b200.ReciprocalRelationsModel("distmult", 10, 3, 8)
    assert m.get_p_embedder().weight.shape[0] == 6 and m.num_relations == 3
    s, p, o = torch.tensor([1, 2]), torch.tensor([0, 2]), torch.tensor([5, 7])
    m.score_po(p, o)
    assert calls[-1] == ("1vsN", "sp_", [5, 7], [3, 5], None)
    m.score_spo(s, p, o, "s")
    assert calls[-1] == ("spo", [5, 7], [3, 5], [1, 2])
    m.score_spo(s, p, o, "o")
    assert calls[-1] == ("spo", [1, 2], [0, 2], [5, 7])
    out = m.score_sp_po(s, p, o, torch.tensor([4, 5, 6]))
    assert out.shape == (2, 6) and calls[-2][1:4] == ("sp_", [1, 2], [0, 2]) and calls[-1][1:4] == ("sp_", [5, 7], [3, 5])
    assert bool((out[:, :3] != out[:, 3:]).all())          # the two halves came from the two calls
    import pytest
    with pytest.raises(Exception, match="undirected"):
        m.score_spo(s, p, o)
    with pytest.raises(Exception, match="cannot score relations"):
        m.score_so(s, o)


def test_csr_loss_decomposition_matches_dense_losses():
    """The algebra of kge_b200/csrc/csr_loss.cu: with labels y = a*count + b the KvsAll losses split into a
    label-free per-row term (what the fused scorer produces) and sums over the listed columns only.  Emulated in
    torch and compared with the oracle's losses on the densified label matrix (duplicates, empty rows, smoothing)."""
    import math
    import torch
    from oracle import kge_oracle as orc

    g = torch.Generator().manual_seed(2)
    n, E = 9, 41
    z = torch.randn((n, E), generator=g, dtype=torch.float64) * 2
    counts = (torch.rand((n, E), generator=g) < 0.1).double()
    counts[2, 5] = 3.0
    counts[4] = 0.0
    for eps in (0.0, 0.2):
        a, b = 1.0 - eps, (1.0 / E if eps > 0 else 0.0)
        y = a * counts + b
        off = 0.7
        # BCE
        A = torch.nn.functional.softplus(z + off).sum(1)
        B = (counts * (z + off)).sum(1)
        Cs = (z + off).sum(1)
        got = float((A - a * B - b * Cs).sum())
        assert abs(got - float(orc.bce_loss(z, y, off))) <= 1e-9 * abs(got)
        # KL
        lse = torch.logsumexp(z, 1)
        Bz, Zs, nnz = (counts * z).sum(1), z.sum(1), counts.sum(1)
        Y = a * nnz + b * E
        total = 0.0
        for i in range(n):
            if float(Y[i]) <= 0:
                continue
            listed = counts[i][counts[i] > 0]
            ylogy = float(((a * listed + b) * torch.log(a * listed + b)).sum())
            rest = (E - listed.numel()) * b * math.log(b) if b > 0 else 0.0
            total += (ylogy + rest) / float(Y[i]) - math.log(float(Y[i])) - (a * float(Bz[i]) + b * float(Zs[i])) / float(Y[i]) + float(lse[i])
        assert abs(total - float(orc.kl_loss(z, y))) <= 1e-9 * abs(total)


def test_synthetic_inputs_match_the_checkers_copy():
    """kge_b200.synthetic (used by bench.py's device arm and the scripts, which must not import oracle/) and the
    oracle's own generators produce identical tensors."""
    import torch
    from kge_b200 import synthetic
    from oracle import kge_oracle as orc

    for model in orc.MODELS:
        D = 8 if model == "rescal" else 16
        a, b = synthetic.make_tables(model, 23, 4, D, sigma=0.3, seed=7), orc.make_tables(model, 23, 4, D, sigma=0.3, seed=7)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert synthetic.relation_dim(model, D) == orc.relation_dim(model, D)
    assert torch.equal(synthetic.make_triples(23, 4, 9, seed=3), orc.make_triples(23, 4, 9, seed=3))


def test_philox_reference_known_answers():
    """Known-answer vectors of Philox4x32-10 (Random123 kat_vectors) pin the Python mirror that checks the device
    sampler (tests/test_gpu_rows.py::test_device_uniform_sampler)."""
    from philox_ref import philox4x32_10

    assert philox4x32_10([0, 0, 0, 0], (0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert philox4x32_10([0xffffffff] * 4, (0xffffffff, 0xffffffff)) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert philox4x32_10([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], (0xa4093822, 0x299f31d0)) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_reference_install_copies_modules_and_yaml_only(tmp_path, monkeypatch):
    """oracle/install_ref.py installs LibKGE's modules and yaml data from a source tree, nothing else."""
    from oracle import install_ref

    src = tmp_path / "src"
    for f in ("kge/__init__.py", "kge/model/__init__.py", "kge/model/complex.yaml", "kge/README.md", "setup.py"):
        (src / f).parent.mkdir(parents=True, exist_ok=True)
        (src / f).write_text(f)
    monkeypatch.setattr(install_ref, "HERE", str(tmp_path))
    monkeypatch.setattr(install_ref, "TARGET", str(tmp_path / "_ref"))
    monkeypatch.setenv("KGE_REFERENCE_SRC", str(src))
    assert install_ref.source_tree() == str(src) and not install_ref.installed()
    install_ref.install(str(src))
    got = sorted(str(p.relative_to(tmp_path / "_ref")) for p in (tmp_path / "_ref").rglob("*") if p.is_file())
    assert got == ["kge/__init__.py", "kge/model/__init__.py", "kge/model/complex.yaml"]
    assert install_ref.installed() and sorted(os.listdir(tmp_path)) == ["_ref", "src"]
    with pytest.raises(RuntimeError):
        install_ref.install(str(tmp_path / "_ref" / "kge"))      # no kge/model package below it
