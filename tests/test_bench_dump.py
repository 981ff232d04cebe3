"""bench.py --dump-outputs: what the last timed step returned, written as .npy files so that two builds run with the
same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_dump_outputs_writes_float_arrays(tmp_path):
    bench.dump_outputs(str(tmp_path / "out"), {"loss": np.float32(1.5), "e2e_loss": np.float64(2.5)}, "_rank1")
    a, b = np.load(tmp_path / "out" / "loss_rank1.npy"), np.load(tmp_path / "out" / "e2e_loss_rank1.npy")
    assert a.dtype == np.float32 and a.shape == () and float(a) == 1.5
    assert b.dtype == np.float64 and float(b) == 2.5


def test_dump_outputs_refuses_other_dtypes_and_oversized_outputs(tmp_path):
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path), {"idx": np.arange(4)})
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path), {"big": np.zeros((64 << 20) // 8 + 1)})
    assert os.listdir(tmp_path) == []


@pytest.mark.gpu
def test_bench_dumps_the_loss_of_its_last_timed_step(tmp_path):
    """--steps 3 times batches 0, 1, 2: the dumped losses are those of batch 2, checked against the CPU oracle."""
    from oracle import kge_oracle as orc

    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                        "--no-configs", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    assert sorted(os.listdir(out)) == ["e2e_loss.npy", "loss.npy"]
    ent, rel = orc.make_tables(bench.MODEL, bench.E, bench.R, bench.D, sigma=1.0)
    tri = orc.make_triples(bench.E, bench.R, bench.N_BATCH, seed=2)
    ref = float(orc.train_1vsall_forward(bench.MODEL, ent.double(), rel.double(), tri, bench.LOSS))
    for name in ("loss.npy", "e2e_loss.npy"):
        got = np.load(out / name)
        assert got.shape == () and got.dtype in (np.float32, np.float64)
        assert float(got) == pytest.approx(ref, rel=1e-4), name
