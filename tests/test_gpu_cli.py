"""BASELINE.json configs[0] — `kge start examples/toy-complex-train.yaml` with `--train.type 1vsAll
--lookup_embedder.dim 128` — through LibKGE's OWN COMMAND LINE (kge/cli.py, launched by scripts/kge_cli.py):

  (ref)    model: complex,       job.device: cpu                      — the reference's CPU-runnable case
  (plugin) model: b200_complex,  job.device: cuda, 1vsAll.class_name: B200TrainingJob1vsAll, modules + kge_b200.plugin

on a toy-shaped synthetic dataset on disk (280 entities / 112 relations / 4565 train / 109 valid / 152 test: the toy
dataset itself is not in the reference repository, data/download_all.sh).  Same seed => same initial tables and batch
order; the per-epoch avg_loss and the validation metrics of the two trace files must agree.  Everything between
`kge start` and the scoring kernels — config loading, plugin discovery (kge/misc.py:13-42, kge_model.py:473-503,
train.py:127-137), dataset loading, DataLoader, optimizer, checkpoints, the entity-ranking validation job — is the
reference's code."""
import os
import subprocess
import sys

import pytest
import torch
import yaml

from kge_b200 import hostenv

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not hostenv.available(), reason="LibKGE not installed (oracle/install_ref.py)")]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E, R, SIZES = 280, 112, {"train": 4565, "valid": 109, "test": 152}

BASE = """job.type: train
dataset.name: {data}
dataset.pickle: False
random_seed.default: 42
train:
  type: 1vsAll
  max_epochs: 3
  optimizer.default:
    type: Adagrad
    args:
      lr: 0.2
valid.every: 3
lookup_embedder:
  dim: 128
  regularize_weight: 0.8e-7
  initialize: normal_
  initialize_args:
    normal_:
      mean: 0.0
      std: 0.1
"""


def _write_dataset(d):
    os.makedirs(d, exist_ok=True)
    g = torch.Generator().manual_seed(5)
    for k, n in SIZES.items():
        t = torch.stack([torch.randint(0, E, (n,), generator=g), torch.randint(0, R, (n,), generator=g),
                         torch.randint(0, E, (n,), generator=g)], 1)
        with open(os.path.join(d, f"{k}.del"), "w") as f:
            f.writelines(f"{s}\t{p}\t{o}\n" for s, p, o in t.tolist())
    for nm, cnt, pre in (("entity_ids", E, "e"), ("relation_ids", R, "r")):
        with open(os.path.join(d, f"{nm}.del"), "w") as f:
            f.writelines(f"{i}\t{pre}{i}\n" for i in range(cnt))
    files = {f"files.{k}.{a}": v for k, n in SIZES.items()
             for a, v in (("filename", f"{k}.del"), ("size", n), ("type", "triples"))}
    files.update({"files.entity_ids.filename": "entity_ids.del", "files.entity_ids.type": "map",
                  "files.relation_ids.filename": "relation_ids.del", "files.relation_ids.type": "map",
                  "name": "toy", "num_entities": E, "num_relations": R})
    with open(os.path.join(d, "dataset.yaml"), "w") as f:
        yaml.safe_dump({"dataset": files}, f)


def _run(tmp, tag, extra_yaml, device):
    cfg = os.path.join(tmp, f"{tag}.yaml")
    with open(cfg, "w") as f:
        f.write(BASE.format(data=os.path.join(tmp, "toy")) + extra_yaml)
    out = os.path.join(tmp, f"out_{tag}")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "kge_cli.py"), "start", cfg, "--folder", out,
                        "--job.device", device, "--console.quiet", "True"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    entries = []
    for line in open(os.path.join(out, "trace.yaml")):      # one flow-style yaml dict per line (kge/config.py trace)
        try:
            entries.append(yaml.safe_load(line))
        except yaml.YAMLError:                               # the job_created entry carries a python-tagged torch version
            continue
    entries = [e for e in entries if isinstance(e, dict)]
    epochs = [e["avg_loss"] for e in entries if e.get("job") == "train" and e.get("scope") == "epoch"
              and e.get("event") == "epoch_completed"]
    valid = [e for e in entries if e.get("job") == "eval" and e.get("scope") == "epoch"][-1]
    log = open(os.path.join(out, "kge.log")).read()
    return epochs, valid, log, os.path.exists(os.path.join(out, "checkpoint_best.pt"))


def test_kge_start_toy_complex_1vsall(tmp_path):
    tmp = str(tmp_path)
    _write_dataset(os.path.join(tmp, "toy"))
    ref_ep, ref_valid, _, _ = _run(tmp, "ref", "model: complex\n", "cpu")
    plug_ep, plug_valid, log, ckpt = _run(
        tmp, "plugin",
        "modules: [kge.job, kge.model, kge.model.embedder, kge_b200.plugin]\nmodel: b200_complex\n"
        "1vsAll.class_name: B200TrainingJob1vsAll\n", "cuda")
    assert ckpt and len(ref_ep) == 3 and len(plug_ep) == 3
    for a, b in zip(plug_ep, ref_ep):      # every batch after the first already runs on natively updated tables
        assert a == pytest.approx(b, rel=2e-3)
    assert ref_ep[-1] < ref_ep[0]
    for k in ("mean_reciprocal_rank_filtered", "mean_rank_filtered", "hits_at_10_filtered"):
        assert plug_valid[k] == pytest.approx(ref_valid[k], rel=0.05, abs=0.01), k
