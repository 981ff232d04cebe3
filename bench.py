#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the KGE scoring hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (BASELINE.json configs[1]): ComplEx dim=512, 1vsAll + BCE, FB15k-237-shaped synthetic graph (14 541
entities / 237 relations), batch n = 1024 triples per GPU.  One "step" = one 1vsAll forward pass over one batch
(train_1vsAll.py:48-82 without backward): score_sp + BCE against all entities and score_po + BCE against all
entities = 2*n*E candidate triples scored.  metric = candidate triples scored per second (whole job, all GPUs).

  value        : batch indexes already resident in HBM; the fused step entry point; CUDA events per step
  e2e          : the SAME step through the reference-facing plugin: the reference's own job object
                 (`1vsAll.class_name: B200TrainingJob1vsAll`, `model: b200_complex`, job.device cuda) processes a
                 pinned HOST batch with `job._process_batch` — H2D of the triples, kernels, `.item()` D2H inside the
                 timed region (falls back to the C-ABI host entry point when LibKGE is not importable; `e2e.api` says)
  roofline     : dominant kernel, CUDA events on its launch stream, against MEASURED_PEAKS.json
  cpu_baseline : the UNMODIFIED reference job (`model: complex`, job.device cpu, installed in oracle/_ref by
                 oracle/install_ref.py) processing the same batches on the host cores, bounded sample
  configs      : (N=1) the other BASELINE.json configs — RotatE negative sampling, RESCAL KvsAll with CSR labels,
                 one Wikidata5M-shaped TransE shard — kernel ms, rate, roofline fraction, parity vs the live reference
  sharded      : (N>1) BASELINE config 5: TransE d=512, 600 k rows per GPU, entity-sharded across the N ranks with
                 NCCL (query-row all-reduce, int64 rank all-reduce, logits all-gather); per-phase ms

`--impl reference` runs the reference arm alone (rank 0 only under torchrun).
L2 is flushed (a 256 MiB buffer is overwritten) before every timed step, outside the timed bracket.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL, E, R, D, N_BATCH = "complex", 14541, 237, 512, 1024
LOSS = "bce"
METRIC = "triples scored/sec 1vsAll ComplEx d=512"
UNIT = "triples/s"
WORKLOAD = ("ComplEx d=512 1vsAll+BCE forward (score_sp+loss, score_po+loss), FB15k-237-shaped synthetic: "
            "14541 ent / 237 rel, n=1024 triples per GPU per step")
MODULES = ["kge.job", "kge.model", "kge.model.embedder", "kge_b200.plugin"]


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return {"hbm_gbs": float(j["hbm_gbs"]), "bf16_tflops": float(j["bf16_tflops"]),
                    "bf16_tflops_sustained": float(j.get("bf16_tflops_sustained", j["bf16_tflops"])),
                    "source": "measured (MEASURED_PEAKS.json)"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------
# The reference's own job objects (LibKGE), on CPU (reference arm) or on CUDA through the plugin (e2e)
def _have_kge():
    try:
        from kge_b200 import hostenv

        return hostenv.available()
    except Exception:
        return False


def make_job(model_name, device, job_class=None, E_=E, R_=R, D_=D, n_batch=N_BATCH, train_type="1vsAll", loss=LOSS,
             extra=None, tables=None):
    """A forward-only reference TrainingJob over an in-memory dataset of the bench shape, tables = synthetic."""
    import torch

    from kge_b200 import hostenv, synthetic

    hostenv.import_kge()
    from kge import Config, Dataset
    from kge.job import TrainingJob

    config = Config()
    config.folder = tempfile.mkdtemp(prefix="kge_bench_")
    config.set("console.quiet", True)
    config.set("modules", MODULES)
    config.set("model", model_name)
    config._import(model_name)
    config.set("dataset.name", "synthetic")
    config.set("dataset.num_entities", E_)
    config.set("dataset.num_relations", R_)
    config.set("dataset.pickle", False)
    config.set("job.device", device)
    config.set("job.type", "train")
    config.set("train.type", train_type)
    config.set("train.loss", loss)
    config.set("train.batch_size", n_batch)
    config.set("train.num_workers", 0)
    config.set_all({"lookup_embedder.dim": D_})
    if job_class:
        config.set(f"{train_type}.class_name", job_class)
    if extra:
        config.set_all(extra)
    ds = Dataset(config, None)
    ds._triples = {"train": synthetic.make_triples(E_, R_, 4 * n_batch, seed=99).int()}
    ds._meta = {"entity_ids": [str(i) for i in range(E_)], "relation_ids": [str(i) for i in range(R_)]}
    job = TrainingJob.create(config, ds, forward_only=True)
    base = model_name[5:] if model_name.startswith("b200_") else model_name
    ent, rel = tables if tables is not None else synthetic.make_tables(base, E_, R_, D_, sigma=1.0)
    with torch.no_grad():
        w = job.model.get_s_embedder()._embeddings.weight
        w.copy_(ent.to(w.device))
        w = job.model.get_p_embedder()._embeddings.weight
        w.copy_(rel.to(w.device))
    return job


def _time_reference_job(steps, warmup, budget_s):
    """The reference's TrainingJob1vsAll._process_batch (forward only) on the host cores."""
    import torch

    from kge_b200 import synthetic

    cores_all = os.cpu_count() or 1
    job = make_job(MODEL, "cpu")
    batches = [{"triples": synthetic.make_triples(E, R, N_BATCH, seed=i)} for i in range(4)]
    # give the reference its best shot: oversubscribing a many-core host slows MKL/ATen down
    best_t, best_thr = None, cores_all
    for thr in sorted({cores_all, max(1, cores_all // 2), 32, 16, 8} & set(range(1, cores_all + 1)), reverse=True):
        torch.set_num_threads(thr)
        job._process_batch(0, dict(batches[0]))
        t0 = time.perf_counter()
        job._process_batch(0, dict(batches[1]))
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, best_thr = dt, thr
    torch.set_num_threads(best_thr)
    for i in range(max(1, min(warmup, 3))):
        job._process_batch(i, dict(batches[i % 4]))
    times, t_begin, loss = [], time.perf_counter(), None
    for i in range(steps):
        t0 = time.perf_counter()
        res = job._process_batch(i, dict(batches[i % 4]))
        times.append(time.perf_counter() - t0)
        loss = res.avg_loss
        if time.perf_counter() - t_begin > budget_s:
            break
    per = sum(times) / len(times)
    return {"value": 2.0 * N_BATCH * E / per, "unit": UNIT, "cores": best_thr, "kind": "reference",
            "sample": f"{len(times)} x TrainingJob1vsAll._process_batch (forward only; n={N_BATCH}, E={E}, D={D}, BCE) "
                      f"of the unmodified reference (oracle/_ref) on the host CPU, torch {torch.__version__}, "
                      f"{best_thr} threads (fastest of the probed thread counts on {cores_all} host cores)",
            "ms_per_step": per * 1e3, "avg_loss_last": loss}, len(times)


def _time_oracle_port(steps, warmup, budget_s):
    """Fallback when the reference is not installed: the oracle's restatement of the same step."""
    import torch

    from oracle import kge_oracle as orc

    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    ent, rel = orc.make_tables(MODEL, E, R, D, sigma=1.0)
    tri = orc.make_triples(E, R, N_BATCH, seed=0)
    with torch.no_grad():
        for _ in range(max(1, min(warmup, 2))):
            orc.train_1vsall_forward(MODEL, ent, rel, tri, LOSS)
        times, t_begin = [], time.perf_counter()
        for _ in range(steps):
            t0 = time.perf_counter()
            orc.train_1vsall_forward(MODEL, ent, rel, tri, LOSS)
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_begin > budget_s:
                break
    per = sum(times) / len(times)
    return {"value": 2.0 * N_BATCH * E / per, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} x one 1vsAll forward step with the oracle's torch-CPU restatement of the reference "
                      f"path (reference not installed), {cores} threads", "ms_per_step": per * 1e3}, len(times)


def cpu_reference(steps, warmup, budget_s):
    if _have_kge():
        try:
            return _time_reference_job(steps, warmup, budget_s)
        except Exception as ex:      # never lose the line: fall back to the port and say why
            base, done = _time_oracle_port(steps, warmup, budget_s)
            base["sample"] += f" [live reference failed: {ex!r}]"
            return base, done
    return _time_oracle_port(steps, warmup, budget_s)


def _config(world):
    """The SAME config object in both arms (the driver compares them): the workload, and how the device arm times it."""
    return {"workload": WORKLOAD, "global_batch": N_BATCH * world,
            "parallelism": f"replicas x{world} (batch split, no data-path collective)",
            "l2": "device arm: flushed before every timed step (256 MiB write)",
            "precision": "device arm: f16x3 split (parity mode); reference arm: torch fp32 on the host"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W = max(args.warmup, 3)
    base, done = cpu_reference(max(1, args.steps), W, budget_s=90.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": done, "warmup": W, "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(max(1, args.gpus)),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


# ------------------------------------------------------------------------------------------------------------
def _flops_cfg2():
    # both directions: 2 * (2 n E D)    (SURVEY 8d: ops_alg = 2nED per direction)
    return 2.0 * 2.0 * N_BATCH * E * D


def _timed_kernel(engine, torch, fn, flush, iters=8, warm=3):
    """(kernel_ms of the profiled dominant kernel, call_ms) averaged over `iters` L2-flushed calls."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    engine.profile_enable(True)
    ks, ts = [], []
    for i in range(iters):
        flush.fill_(i & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
        try:
            ks.append(engine.profile_last_ms())
        except Exception:
            ks.append(float("nan"))
    engine.profile_enable(False)
    return sum(ks) / len(ks), sum(ts) / len(ts)


def _ref_model(name, E_, R_, D_, ent, rel, extra=None):
    """The reference KgeModel on CPU over given tables (parity checker of the `configs` section)."""
    import torch

    from kge_b200 import hostenv

    hostenv.import_kge()
    from kge import Config, Dataset
    from kge.model import KgeModel

    config = Config()
    config.folder = None
    config.set("console.quiet", True)
    config.set("model", name)
    config._import(name)
    config.set("dataset.name", "synthetic")
    config.set("dataset.num_entities", E_)
    config.set("dataset.num_relations", R_)
    config.set("dataset.pickle", False)
    config.set("job.device", "cpu")
    config.set_all({"lookup_embedder.dim": D_})
    if extra:
        config.set_all(extra)
    ds = Dataset(config, None)
    ds._meta = {"entity_ids": [str(i) for i in range(E_)], "relation_ids": [str(i) for i in range(R_)]}
    m = KgeModel.create(config, ds)
    m.eval()
    with torch.no_grad():
        m.get_s_embedder()._embeddings.weight.copy_(ent)
        m.get_p_embedder()._embeddings.weight.copy_(rel)
    return m


def _parity(got, ref):
    rms = float(ref.double().pow(2).mean().sqrt())
    err = float((got.double() - ref.double()).abs().max())
    return {"max_abs_err_over_rms": err / max(rms, 1e-30), "ok": bool(err <= 1e-4 * rms), "tolerance": 1e-4}


def headline_parity(engine, torch, dev, ent_c, rel_c, rows=256):
    """The headline shape against the LIVE reference on the CPU for a row sample: score error, and how often the rank
    of the true answer (reference rank arithmetic, eval_entity_ranking.py:571-618) agrees — reported, not asserted."""
    from kge_b200 import synthetic

    tri = synthetic.make_triples(E, R, rows, seed=4242)
    m = _ref_model(MODEL, E, R, D, ent_c, rel_c)
    with torch.no_grad():
        ref = m.score_sp(tri[:, 0], tri[:, 1])
    ent, rel = ent_c.to(dev), rel_c.to(dev)
    t = tri.to(dev)
    got = engine.score_1vsN(MODEL, "sp_", ent, rel, ent, t[:, 0].contiguous(), t[:, 1].contiguous()).cpu()
    out = _parity(got, ref)

    def final_ranks(x):
        tr = x[torch.arange(rows), tri[:, 2]].view(-1, 1)
        close = torch.isclose(x, tr, rtol=1e-4, atol=1e-5)
        rank = ((x > tr) & ~close).sum(1)
        return rank + close.sum(1) // 2
    a, b = final_ranks(got), final_ranks(ref)
    out.update({"rows": rows, "rank_agreement": float((a == b).float().mean()), "max_rank_delta": int((a - b).abs().max()),
                "against": f"reference ComplEx.score_sp on the CPU for {rows} rows of the headline shape; ranks = rounded "
                           "mean rank of the true object with the reference's tolerance band (rtol 1e-4, atol 1e-5)"})
    return out


def other_configs(engine, torch, dev, flush, peaks):
    """BASELINE.json configs 3-5 on one GPU: kernel ms, rate, roofline fraction, parity vs the live reference."""
    from kge_b200 import synthetic

    have_ref = _have_kge()
    sm_clock_ghz, sms = 1.965, 148
    fma_peak = sms * 128 * sm_clock_ghz * 1e9          # fp32 lanes x clock: FADD/FFMA issue slots per second
    out = {}

    # ---- cfg3: RotatE d=512, negative sampling K=1000 (s and o slots), WN18RR-shaped, n=512 ------------------
    try:
        E3, R3, D3, n3, K3 = 40943, 11, 512, 512, 1000
        ent, rel = synthetic.make_tables("rotate", E3, R3, D3)
        ce, cr = ent.to(dev), rel.to(dev)
        tri = synthetic.make_triples(E3, R3, n3, seed=3).to(dev)
        g = torch.Generator().manual_seed(5)
        neg = {0: torch.randint(0, E3, (n3, K3), generator=g).to(dev), 2: torch.randint(0, E3, (n3, K3), generator=g).to(dev)}
        lab = torch.zeros(n3, dtype=torch.int64, device=dev)

        def step3():
            tot = None
            for slot in (0, 2):
                sc = engine.ns_score("rotate", ce, cr, tri, neg[slot], slot, True)
                l = engine.loss_dense(sc, lab, "bce", 5.0)
                tot = l if tot is None else tot + l
            return tot
        _, call_ms = _timed_kernel(engine, torch, step3, flush)
        gathered = 2.0 * n3 * K3 * D3 * 4            # bytes of sampled rows (both slots)
        entry = {"workload": f"RotatE d={D3} negative sampling K={K3} (s and o slots) + BCE(offset 5), WN18RR-shaped "
                             f"{E3} ent, n={n3}: fused gather+score [n,1+K] per slot",
                 "ms_per_step": call_ms, "value": 2.0 * n3 * (1 + K3) / (call_ms * 1e-3), "unit": "needed scores/s",
                 "roofline": {"bound": "hbm", "achieved": gathered / (call_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                              "unit": "GB/s", "frac": gathered / (call_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                              "note": "algorithmic bytes = 4*n*K*D gathered rows per slot (SURVEY 8d); the 84 MB table is "
                                      "L2-resident, so this is gather bandwidth against the HBM peak"}}
        if have_ref:
            m = _ref_model("rotate", E3, R3, D3, ent, rel)
            rows = 3
            t = tri[:rows].cpu()
            ng = neg[2][:rows].cpu()
            with torch.no_grad():
                trip = t.repeat(1, K3).view(-1, 3).clone()
                trip[:, 2] = ng.reshape(-1)
                ref = m.score_spo(trip[:, 0], trip[:, 1], trip[:, 2], "o").view(rows, K3)
            got = engine.ns_score("rotate", ce, cr, tri[:rows], neg[2][:rows], 2, False).cpu()
            entry["parity"] = dict(_parity(got, ref), against="reference RotatE.score_spo on the expanded triples of "
                                   f"{rows} rows x {K3} negatives (the `triple` implementation, sampler.py:294-305)")
        out["cfg3_rotate_ns"] = entry
        del ce, cr, neg
    except Exception as ex:
        out["cfg3_rotate_ns"] = {"error": repr(ex)}

    # ---- cfg4: RESCAL d=200 KvsAll (sp_ queries, KL, CSR multi-hot labels), YAGO3-10-shaped -------------------
    try:
        E4, R4, D4, n4 = 123182, 37, 200, 1024
        ent, rel = synthetic.make_tables("rescal", E4, R4, D4, sigma=0.3)
        ce, cr = ent.to(dev), rel.to(dev)
        tri = synthetic.make_triples(E4, R4, n4, seed=4)
        g = torch.Generator().manual_seed(6)
        counts = torch.randint(1, 20, (n4,), generator=g)
        offs = torch.zeros(n4 + 1, dtype=torch.int64)
        offs[1:] = torch.cumsum(counts, 0)
        cols = torch.cat([torch.sort(torch.randperm(E4, generator=g)[:c]).values for c in counts.tolist()])
        s, p = tri[:, 0].to(dev), tri[:, 1].to(dev)
        doffs, dcols = offs.to(dev), cols.to(dev)

        def step4():
            return engine.score_1vsN_loss_csr("rescal", "sp_", ce, cr, ce, doffs, dcols, s, p, "kl")
        k_ms, call_ms = _timed_kernel(engine, torch, step4, flush)
        flops = 2.0 * n4 * E4 * D4 + 2.0 * n4 * D4 * D4
        entry = {"workload": f"RESCAL d={D4} KvsAll sp_ queries + KL with CSR multi-hot labels (no dense [n,E] label "
                             f"matrix), YAGO3-10-shaped {E4} ent / {R4} rel, n={n4}",
                 "ms_per_step": call_ms, "kernel_ms": k_ms, "value": n4 * E4 / (call_ms * 1e-3), "unit": UNIT,
                 "roofline": {"bound": "tensor", "achieved": flops / (k_ms * 1e-3) / 1e12, "peak": peaks["bf16_tflops"],
                              "unit": "TFLOP/s", "frac": flops / (k_ms * 1e-3) / 1e12 / peaks["bf16_tflops"],
                              "note": "algorithmic 2nEd + 2nd^2 FLOP over the scoring kernel; 3 f16 MMA passes => ceiling 1/3"}}
        if have_ref:
            rows = 24
            m = _ref_model("rescal", E4, R4, D4, ent, rel)
            with torch.no_grad():
                x = m.score_sp(tri[:rows, 0], tri[:rows, 1])
                y = torch.zeros((rows, E4))
                for i in range(rows):
                    y[i, cols[offs[i]:offs[i + 1]]] = 1.0
                ref = torch.nn.functional.kl_div(torch.log_softmax(x, 1), torch.nn.functional.normalize(y, p=1, dim=1),
                                                 reduction="sum")
            got = engine.score_1vsN_loss_csr("rescal", "sp_", ce, cr, ce, doffs[:rows + 1], dcols[: int(offs[rows])],
                                             s[:rows], p[:rows], "kl")
            rel_err = abs(float(got) - float(ref)) / abs(float(ref))
            entry["parity"] = {"rel_err_loss": rel_err, "ok": bool(rel_err <= 1e-4), "tolerance": 1e-4,
                               "against": f"reference Rescal.score_sp + KLDivWithSoftmaxKgeLoss on {rows} rows"}
        out["cfg4_rescal_kvsall"] = entry
        del ce, cr
    except Exception as ex:
        out["cfg4_rescal_kvsall"] = {"error": repr(ex)}

    # ---- cfg5: one Wikidata5M-shaped TransE shard (600 k rows), 1vsAll scores + entity-ranking counts --------
    try:
        out["cfg5_transe_shard"] = transe_shard_bench(engine, torch, dev, flush, peaks, have_ref, fma_peak)
    except Exception as ex:
        out["cfg5_transe_shard"] = {"error": repr(ex)}
    return out


def train_step_bench(torch, local, ent_c, rel_c, batches_host, flush, iters=10):
    """The headline workload as a TRAINING step (forward + backward, no optimizer step) through the reference job's
    `_process_batch` on the plugin with the gradient kernels (SURVEY 8f-1); informational, not part of `value`."""
    import torch as _t

    if not _have_kge():
        return {"skipped": "reference not installed"}
    from kge_b200 import hostenv

    hostenv.import_kge()
    job = make_job("b200_" + MODEL, f"cuda:{local}", job_class="B200TrainingJob1vsAll", tables=(ent_c, rel_c))
    job.is_forward_only = False
    for i in range(3):
        job._process_batch(i, {"triples": batches_host[i % 4]})
    _t.cuda.synchronize()
    ts = []
    for i in range(iters):
        flush.fill_(i & 0xFF)
        _t.cuda.synchronize()
        t0 = time.perf_counter()
        job._process_batch(i, {"triples": batches_host[i % 4]})
        _t.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    per = sum(ts) / len(ts)
    g = job.model.get_s_embedder()._embeddings.weight.grad
    return {"workload": "the headline batch as a training step: fused forward + native backward (recompute, G planes, two "
                        "split-K tensor-core GEMMs, unfold) through B200TrainingJob1vsAll._process_batch; gradients "
                        "accumulate into .grad, no optimizer step",
            "ms_per_step": per * 1e3, "value": N_BATCH / per, "unit": "train triples/s",
            "grad_finite": bool(g is not None and bool(_t.isfinite(g).all()))}


def reference_on_gpu_bench(torch, local, ent_c, rel_c, batches_host, flush, iters=20):
    """SURVEY 8d "PyTorch-on-B200" bar: the UNMODIFIED reference job and model (`model: complex`, no plugin module on the
    path) with job.device cuda — torch's own kernels (cuBLAS sgemm, elementwise, BCEWithLogits) on the same GPU, same
    batches, same harness as `e2e` (host batch in, .item() out, wall clock between synchronisations)."""
    if not _have_kge():
        return {"skipped": "reference not installed"}
    job = make_job(MODEL, f"cuda:{local}", tables=(ent_c, rel_c))
    assert type(job).__name__ == "TrainingJob1vsAll" and type(job.model).__name__ == "ComplEx"
    for i in range(3):
        loss = job._process_batch(i, {"triples": batches_host[i % 4]}).avg_loss
    torch.cuda.synchronize()
    ts = []
    for i in range(iters):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = job._process_batch(i, {"triples": batches_host[i % 4]}).avg_loss
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    per = sum(ts) / len(ts)
    return {"workload": "the headline step through the unmodified reference TrainingJob1vsAll._process_batch (forward only) "
                        "with the reference's own ComplEx model on job.device cuda (torch eager: fp32 cuBLAS GEMMs with "
                        f"torch.backends.cuda.matmul.allow_tf32={torch.backends.cuda.matmul.allow_tf32}, embed_all copy, "
                        "[n,E] logits and BCE through HBM)",
            "ms_per_step": per * 1e3, "value": 2.0 * N_BATCH * E / per, "unit": UNIT, "loss_last": float(loss)}


def batch_split_train_bench(torch, dist, local, rank, world, ent_c, rel_c, flush, iters=10):
    """SURVEY 8e "small tables": replicas + batch split as a TRAINING step.  Every rank holds the whole ComplEx tables
    and runs B200TrainingJob1vsAll._process_batch with `user.b200_batch_split` on the SAME global batch of
    N_BATCH * world triples: fused forward + native backward on its N_BATCH rows, then ncclAllReduce of the dense table
    gradients (and of the batch loss).  Weak scaling; wall clock between device synchronisations, max over ranks."""
    if not _have_kge():
        return {"skipped": "reference not installed"}
    from kge_b200 import hostenv, synthetic

    hostenv.import_kge()
    nb = N_BATCH * world
    dev = torch.device("cuda", local)
    out = {}
    for tag, split in (("batch_split", True), ("one_rank_own_batch", False)):
        job = make_job("b200_" + MODEL, f"cuda:{local}", job_class="B200TrainingJob1vsAll", tables=(ent_c, rel_c),
                       n_batch=nb if split else N_BATCH, extra={"user.b200_batch_split": split})
        job.is_forward_only = False
        batches = [{"triples": synthetic.make_triples(E, R, nb if split else N_BATCH, seed=50 + i).contiguous().pin_memory()}
                   for i in range(4)]
        for i in range(3):
            job.model.zero_grad(set_to_none=False)
            job._process_batch(i, batches[i % 4])
        torch.cuda.synchronize()
        dist.barrier()
        ts = []
        for i in range(iters):
            flush.fill_(i & 0xFF)
            job.model.zero_grad(set_to_none=False)
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            res = job._process_batch(i, batches[i % 4])
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        t = torch.tensor([sum(ts) / len(ts)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[tag] = {"ms_per_step": float(t) * 1e3, "loss": float(res.avg_loss)}
        if split:       # replicas must hold identical gradients after the all-reduce
            g = job.model.get_s_embedder()._embeddings.weight.grad
            ck = torch.stack([g.double().sum(), g.double().abs().sum()])
            lo, hi = ck.clone(), ck.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            out[tag]["replica_gradients_identical"] = bool(torch.equal(lo, hi))
            out[tag]["grad_bytes_all_reduced"] = int(sum(p.numel() * 4 for p in job.model.parameters()))
        del job
    per = out["batch_split"]["ms_per_step"] * 1e-3
    return {"workload": f"ComplEx d={D} 1vsAll+{LOSS.upper()} training step, global batch {nb} = {N_BATCH} rows per GPU, tables "
                        f"replicated x{world}: fused forward + native backward per rank, dense-gradient ncclAllReduce "
                        "(B200TrainingJob1vsAll, user.b200_batch_split)",
            "parallelism": f"replicas + batch split x{world} (NCCL all-reduce of gradients)", "scaling": "weak",
            "ms_per_step": per * 1e3, "value": nb / per, "unit": "train triples/s",
            "same_step_without_collective_ms": out["one_rank_own_batch"]["ms_per_step"], "detail": out}


def transe_shard_bench(engine, torch, dev, flush, peaks, have_ref, fma_peak):
    rows, D5, n5, R5 = 600000, 512, 128, 822
    g = torch.Generator(device=dev).manual_seed(1234)
    shard = torch.randn((rows, D5), generator=g, device=dev)
    rel = torch.randn((R5, D5), generator=torch.Generator(device=dev).manual_seed(7), device=dev)
    gi = torch.Generator().manual_seed(3)
    tri = torch.stack([torch.randint(0, rows, (n5,), generator=gi), torch.randint(0, R5, (n5,), generator=gi),
                       torch.randint(0, rows, (n5,), generator=gi)], 1).to(dev)
    s, p, o = tri[:, 0].contiguous(), tri[:, 1].contiguous(), tri[:, 2].contiguous()
    both = torch.cat([s, o])
    x = engine.score_sp_po("transe", shard, rel, s, p, o, both)          # true scores via the 1-vs-N path
    ar = torch.arange(n5, device=dev)
    true2n = torch.cat([x[ar, n5 + ar], x[ar, 2 * n5 + ar]]).contiguous()

    def step5():
        return engine.rank_sp_po("transe", shard, rel, shard, shard, true2n, s, p, o)
    k_ms, call_ms = _timed_kernel(engine, torch, step5, flush, iters=5, warm=2)
    # SURVEY 8d counts 3 fp32 ops per (i, j, k) (sub, abs, add); the kernel issues 2 instructions for them (|a - b| is a
    # FADD with an operand modifier, then the accumulate), so the issue-slot roofline uses 2
    ops = 2.0 * 2.0 * n5 * rows * D5
    byts = rows * D5 * 4.0
    entry = {"workload": f"TransE d={D5} L1, one Wikidata5M-shaped shard of {rows} entity rows, n={n5}: fused score_sp_po + "
                         "rank/tie counting (both directions stacked in one launch)",
             "ms_per_step": call_ms, "kernel_ms": k_ms, "value": 2.0 * n5 * rows / (call_ms * 1e-3), "unit": UNIT,
             "roofline": {"bound": "fp32 CUDA-core pipe (SURVEY 8d: ALU-bound for n >= 12)",
                          "achieved": ops / (k_ms * 1e-3) / 1e12, "peak": fma_peak / 1e12, "unit": "T instr/s (fp32 issue slots)",
                          "frac": ops / (k_ms * 1e-3) / fma_peak,
                          "hbm_frac": byts / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                          "note": "north_star asks for the HBM fraction (hbm_frac: 1.23 GB table stream per call); the "
                                  "binding roofline is the fp32 pipe: 148 SM x 128 lanes x 1.965 GHz issue slots"}}
    if have_ref:
        sub = torch.randperm(rows, generator=torch.Generator().manual_seed(9))[:4096]
        m = _ref_model("transe", 4096, R5, D5, shard[sub.to(dev)].cpu(), rel.cpu())
        q = 8
        with torch.no_grad():
            loc = torch.arange(q)                    # queries: the first q sampled rows as subjects
            ref = m.score_sp(loc, p[:q].cpu())
        got = engine.score_1vsN("transe", "sp_", shard, rel, shard, sub[:q].to(dev), p[:q], sub.to(dev)).cpu()
        entry["parity"] = dict(_parity(got, ref), against=f"reference TransE.score_sp (torch.cdist) for {q} queries x 4096 "
                               "sampled rows of the shard")
    return entry


def sharded_bench(engine, torch, dist, dev, rank, world, flush, peaks, iters=6):
    """BASELINE config 5 across the N ranks: entity-sharded TransE, NCCL collectives, per-phase CUDA-event times
    (max over ranks)."""
    from kge_b200.sharded import ShardedKgeModel

    rows, D5, n5, R5 = 600000, 512, 128, 822
    Etot = rows * world
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    shard = torch.randn((rows, D5), generator=g, device=dev)
    rel = torch.randn((R5, D5), generator=torch.Generator(device=dev).manual_seed(7), device=dev)
    m = ShardedKgeModel("transe", shard, rel, Etot)
    gi = torch.Generator().manual_seed(3)
    tri = torch.stack([torch.randint(0, Etot, (n5,), generator=gi), torch.randint(0, R5, (n5,), generator=gi),
                       torch.randint(0, Etot, (n5,), generator=gi)], 1).to(dev)
    s, p, o = tri[:, 0].contiguous(), tri[:, 1].contiguous(), tri[:, 2].contiguous()

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def phases():
        """rank_sp_po spelled out with events between its phases (same calls as ShardedKgeModel.rank_sp_po)."""
        e0 = ev()
        both = m.backend.exchange_rows(m.ent, m.lo, torch.cat([s, o]))
        e1 = ev()
        dist.all_reduce(both)
        e2 = ev()
        s_emb, o_emb = both[:n5], both[n5:]
        x = m.backend.score_sp_po("transe", s_emb, rel, p, o_emb, both, 1.0, "auto")
        ar = torch.arange(n5, device=dev)
        true2n = torch.cat([x[ar, n5 + ar], x[ar, 2 * n5 + ar]]).contiguous()
        e3 = ev()
        r, t = m.backend.rank_sp_po("transe", s_emb, rel, p, o_emb, m.ent, true2n, None, 1e-4, 1e-5, 1.0, "auto")
        e4 = ev()
        counts = torch.stack([r, t])
        dist.all_reduce(counts)
        e5 = ev()
        return (e0, e1, e2, e3, e4, e5), counts

    for _ in range(2):
        phases()
    torch.cuda.synchronize()
    dist.barrier()
    acc = [0.0] * 5
    total = 0.0
    for i in range(iters):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        es, _ = phases()
        torch.cuda.synchronize()
        for j in range(5):
            acc[j] += es[j].elapsed_time(es[j + 1])
        total += es[0].elapsed_time(es[5])
    t = torch.tensor(acc + [total], dtype=torch.float64, device=dev) / iters
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ph = [float(v) for v in t[:5]]
    total_ms = float(t[5])

    # full logits (north_star: "local-shard scoring + NCCL all-gather of per-shard logits"), n reduced to bound memory
    nl = 32
    for _ in range(2):
        full = m.score_sp_po(s[:nl], p[:nl], o[:nl])
    torch.cuda.synchronize()
    dist.barrier()
    a = ev()
    full = m.score_sp_po(s[:nl], p[:nl], o[:nl])
    b = ev()
    torch.cuda.synchronize()
    lg = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    dist.all_reduce(lg, op=dist.ReduceOp.MAX)
    shape = list(full.shape)
    # the same logits with the all-gather fused into the scoring kernel (epilogue stores to the peers' symmetric
    # buffers): must be bit-identical
    fused = None
    try:
        for _ in range(2):
            ff = m.score_sp_po_fused(s[:nl], p[:nl], o[:nl])
        same_logits = bool(torch.equal(ff, full))
        torch.cuda.synchronize()
        dist.barrier()
        a2 = ev()
        ff = m.score_sp_po_fused(s[:nl], p[:nl], o[:nl])
        b2 = ev()
        torch.cuda.synchronize()
        lf = torch.tensor([a2.elapsed_time(b2)], dtype=torch.float64, device=dev)
        dist.all_reduce(lf, op=dist.ReduceOp.MAX)
        ok = torch.tensor([1 if same_logits else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        fused = {"op": "scoring kernel whose epilogue stores into every rank's symmetric [n, 2E] buffer over NVLink "
                       "(peer-mapped pointers; torch symmetric memory for allocation + barriers)",
                 "ms_per_call": float(lf), "bit_identical_to_nccl_path": bool(int(ok) == 1),
                 "bytes_stored_to_peers_per_rank": nl * 2 * rows * 4 * (world - 1)}
        del ff
    except Exception as ex:
        fused = {"error": repr(ex)}
    del full

    # exactness at a small shape: N-rank ranks / logits == the same quantities on one rank over the whole table
    from kge_b200 import synthetic
    E0, R0, n0 = 4001, 7, 50
    ent0, rel0 = synthetic.make_tables("transe", E0, R0, 64, sigma=0.5)
    tri0 = synthetic.make_triples(E0, R0, n0).to(dev)
    lo, hi = ShardedKgeModel.shard_bounds(E0, world, rank)
    ms = ShardedKgeModel("transe", ent0[lo:hi].to(dev), rel0.to(dev), E0)
    one = ShardedKgeModel("transe", ent0.to(dev), rel0.to(dev), E0, rank=0, world=1)
    ra = ms.rank_sp_po(tri0[:, 0], tri0[:, 1], tri0[:, 2])
    rb = one.rank_sp_po(tri0[:, 0], tri0[:, 1], tri0[:, 2])
    same = all(bool(torch.equal(x, y)) for x, y in zip(ra, rb))
    same = same and bool(torch.equal(ms.score_sp_po(tri0[:, 0], tri0[:, 1], tri0[:, 2]),
                                     one.score_sp_po(tri0[:, 0], tri0[:, 1], tri0[:, 2])))
    flag = torch.tensor([1 if same else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {
        "workload": f"TransE d={D5} L1 entity-sharded x{world}: {rows} rows per GPU (E={Etot}, weak scaling in E), n={n5}: "
                    "rank_sp_po = query-row exchange + local fused score+rank on the shard + int64 all-reduce",
        "parallelism": f"entity-sharded x{world} (NCCL)", "scaling": "weak",
        "value": 2.0 * n5 * Etot / (total_ms * 1e-3), "unit": UNIT, "ms_per_call": total_ms,
        "phases_ms": {"exchange_gather_kernel": ph[0], "exchange_all_reduce": ph[1], "true_scores": ph[2],
                      "local_score_rank_kernel": ph[3], "counts_all_reduce": ph[4]},
        "collective": {"exchange": {"op": "ncclAllReduce(sum, f32)", "bytes_per_call": 2 * n5 * D5 * 4},
                       "counts": {"op": "ncclAllReduce(sum, i64)", "bytes_per_call": 2 * 2 * n5 * 8}},
        "logits_all_gather": {"op": "ncclAllGather(f32) + one re-layout copy", "n": nl, "shape": shape,
                              "bytes_gathered_per_rank": nl * 2 * rows * 4 * world, "ms_per_call": float(lg)},
        "logits_fused_all_gather": fused,
        "ranks_bit_identical_to_single_gpu": bool(int(flag) == 1),
    }


def run_ours(args):
    import torch

    from kge_b200 import engine, synthetic          # the device arm never touches oracle/

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist  # noqa: F811

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if not engine.device_ok():
        raise RuntimeError("bench.py needs an sm_100 (B200) device; kge_b200 has no fallback path")

    ent_c, rel_c = synthetic.make_tables(MODEL, E, R, D, sigma=1.0)
    ent, rel = ent_c.to(dev), rel_c.to(dev)
    K, W = args.steps, max(args.warmup, 3)
    # every rank scores its own batches (weak scaling: per-GPU work fixed, no data-path collective)
    batches_host = [synthetic.make_triples(E, R, N_BATCH, seed=1000 * rank + i).contiguous().pin_memory()
                    for i in range(4)]
    batches_dev = [b.to(dev) for b in batches_host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident step: the fused entry point, batch indexes already in HBM ----------------------
    ws = engine._workspace(0, N_BATCH, E, D, False, dev)
    loss_dev = torch.zeros((), dtype=torch.float32, device=dev)

    def device_step(i):
        return engine.train_1vsall_forward(MODEL, ent, rel, batches_dev[i % 4], LOSS, 0.0, out=loss_dev,
                                           workspace=ws)

    for i in range(W):
        device_step(i)
    barrier()
    engine.profile_enable(True)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    kern_ms = []
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    engine.launch_count(reset=True)
    barrier()
    for i in range(K):
        flush.fill_(i & 0xFF)                       # evict L2 (outside the timed bracket)
        ev[i][0].record()
        device_step(i)
        ev[i][1].record()
        ev[i][1].synchronize()
        kern_ms.append(engine.profile_last_ms())   # the stacked (2n-row) pairwise kernel of this step
    barrier()
    launches = engine.launch_count()
    engine.profile_enable(False)
    outputs = {"loss": loss_dev.cpu().numpy()}      # the 0-d loss the last timed step returned
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms)
    value = world * K * 2.0 * N_BATCH * E / (total_ms * 1e-3)

    # ---- end to end through the reference-facing plugin: the reference's job object on CUDA -----------------
    e2e_api, h2d, d2h = None, N_BATCH * 3 * 8, 8
    job_loss = None
    step = None
    if _have_kge():
        try:
            job = make_job("b200_" + MODEL, f"cuda:{local}", job_class="B200TrainingJob1vsAll", tables=(ent_c, rel_c))
            assert type(job).__name__ == "B200TrainingJob1vsAll"

            def step(i):
                return job._process_batch(i, {"triples": batches_host[i % 4]}).avg_loss
            e2e_api = ("kge.job.TrainingJob._process_batch of B200TrainingJob1vsAll (1vsAll.class_name) with model "
                       "b200_complex on job.device cuda: pinned host batch -> one library call (H2D copy, fused step, "
                       "4-byte read-back, stream sync) -> float")
            d2h = 4
        except Exception as ex:
            step, e2e_api = None, f"job plugin unavailable ({ex!r}); "
    if step is None:
        host = engine.HostStep(MODEL, ent, rel, N_BATCH, LOSS)

        def step(i):
            return host(batches_host[i % 4])
        e2e_api = (e2e_api or "") + "C ABI b200kge_train_1vsall_forward_host (pinned host triples -> loss on the host)"
        d2h = 4
    for i in range(W):
        job_loss = step(i)
    barrier()
    e2e_t = []
    for i in range(K):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        job_loss = step(i)                          # H2D + kernels + D2H (+ the job's own bookkeeping) inside
        e2e_t.append(time.perf_counter() - t0)
    barrier()
    outputs["e2e_loss"] = np.float64(job_loss)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, "" if world == 1 else f"_rank{rank}")
    clocks = sampler.stop() if rank == 0 else None
    e2e_total = torch.tensor([sum(e2e_t)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_value = world * K * 2.0 * N_BATCH * E / float(e2e_total)

    sharded = None
    if dist is not None:
        try:
            sharded = sharded_bench(engine, torch, dist, dev, rank, world, flush, _peaks())
        except Exception as ex:
            sharded = {"error": repr(ex)}
        barrier()
        try:
            sharded["batch_split_training"] = batch_split_train_bench(torch, dist, local, rank, world, ent_c, rel_c, flush)
        except Exception as ex:
            sharded["batch_split_training"] = {"error": repr(ex)}
        barrier()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = _peaks()
    k_ms = sum(kern_ms) / len(kern_ms)
    achieved = _flops_cfg2() / (k_ms * 1e-3) / 1e12
    peak = peaks["bf16_tflops"]
    pair = os.environ.get("B200KGE_TC_VERSION", "4") == "4"        # n = 1024 >= 128: the CTA-pair kernel is the default
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
        "traffic": 34.1e6,
        "traffic_from": "profiles/r2c_raw_tc4.csv / r2_raw_tc3.csv (ncu --set full of this command: dram__bytes_read.sum 34.11 MB + "
                        "dram__bytes_write.sum 0 per launch) — NOT measured in this run; algorithmic bytes = table "
                        "planes 29.8 MB + query planes 4.2 MB",
        "kernel": "pairwise_tc4_kernel<BCE> (CTA pair)" if pair else "pairwise_tc3_kernel<BCE>",
        "kernel_ms": k_ms,
        "peak_name": f"dense bf16 burst, {peaks['source']}",
        "note": "algorithmic fp32 FLOPs (2nED per direction, both directions in one launch).  For fp32-equivalent "
                "results the operands are split once per call into fp16 hi/lo planes and the kernel issues hi*hi + "
                "hi*lo + lo*hi: 3 f16 MMAs per 16 reduction elements where a plain bf16 GEMM needs 1, so the ceiling "
                "of `frac` is 1/3; tensor_pipe_frac_executed = 3 * frac is the share of the measured bf16 peak the "
                "kernel's executed MMAs reach",
        "tensor_pipe_frac_executed": 3.0 * achieved / peak,
    }
    cpu, _ = cpu_reference(40, 1, budget_s=12.0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (fp16 hi/lo split products hi*hi + hi*lo + lo*hi on tcgen05, fp32 accumulate; ~2.5e-5 of score rms vs fp64)",
        "data": "synthetic",
        "config": _config(world),
        "roofline": roofline,
        "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * float(e2e_total) / K, "api": e2e_api, "loss_last": job_loss},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if world == 1 and _have_kge():
        try:
            line["parity"] = headline_parity(engine, torch, dev, ent_c, rel_c)
        except Exception as ex:
            line["parity"] = {"error": repr(ex)}
    if sharded is not None:
        line["sharded"] = sharded
    if world == 1 and not args.no_configs:
        try:
            line["configs"] = other_configs(engine, torch, dev, flush, peaks)
        except Exception as ex:
            line["configs"] = {"error": repr(ex)}
        try:
            line["configs"]["cfg2_train_fwd_bwd"] = train_step_bench(torch, local, ent_c, rel_c, batches_host, flush)
        except Exception as ex:
            line["configs"]["cfg2_train_fwd_bwd"] = {"error": repr(ex)}
        try:
            line["reference_on_b200"] = reference_on_gpu_bench(torch, local, ent_c, rel_c, batches_host, flush)
        except Exception as ex:
            line["reference_on_b200"] = {"error": repr(ex)}
    _emit(line)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, outputs, suffix=""):
    """Writes each output as out_dir/<name><suffix>.npy (float32 / float64, at most 64 MB in all), so that two builds
    run with the same arguments, and therefore the same seeded inputs, can be compared output for output."""
    arrays = {name: np.asarray(a) for name, a in outputs.items()}
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"output {name} has dtype {a.dtype}; only float32 / float64 are dumped")
    if sum(a.nbytes for a in arrays.values()) > 64 << 20:
        raise ValueError("outputs exceed 64 MB; dump a seeded sample instead")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


_OUT_FD = None


def _stdout_for_the_json_line_only():
    """Libraries print to stdout too (NCCL's version banner under NCCL_DEBUG=VERSION): route fd 1 to stderr for the whole
    run and keep the original for the ONE json line the contract asks for."""
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _OUT_FD is None:
        os.write(1, data)
    else:
        os.write(_OUT_FD, data)


def main():
    _stdout_for_the_json_line_only()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs (N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy: loss (the "
                         "device-resident step) and e2e_loss (the host-batch step); with N > 1 each rank adds _rank<r>")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the device arm; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
