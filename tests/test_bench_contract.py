"""CPU: the reference arm of bench.py (oracle port on the host cores) runs without a GPU and prints the contract's
JSON line; --dump-outputs writes bounded, comparable arrays.  GPU: the timed arm honours --steps and dumps the same
arrays from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--queries", "8", "--gallery", "32"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]:
        assert key in line, key
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["metric"] == "embed+top-k query images/sec" and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert line["value"] > 0


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_keeps_small_arrays_whole_and_samples_large_ones(tmp_path):
    import bench
    vals = torch.rand(100, 10)
    idx = torch.randint(0, 5000, (100, 10))
    feats = torch.randn(5000, 64, dtype=torch.float64)
    half = torch.randn(300, 8, dtype=torch.bfloat16)
    limit = 100 * 10 * 4 + 100 * 10 * 8 + 300 * 8 * 4 + 1000 * 64 * 8
    rows = bench.dump_outputs(str(tmp_path), {"values": vals, "indices": idx, "features": feats, "half": half},
                              limit=limit)
    assert rows == {"values": [100, 100], "indices": [100, 100], "half": [300, 300], "features": [1000, 5000]}
    v, i, h, f = (np.load(tmp_path / f"{n}.npy") for n in ("values", "indices", "half", "features"))
    assert v.dtype == np.float32 and np.array_equal(v, vals.numpy())
    assert i.dtype == np.float64 and np.array_equal(i, idx.numpy().astype(np.float64))
    assert h.dtype == np.float32 and np.array_equal(h, half.float().numpy())
    assert f.dtype == np.float64 and np.array_equal(f, feats.numpy()[np.arange(1000) * 5000 // 1000])
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= limit + 4 * 128


def test_dump_outputs_is_refused_by_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                          str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
    assert not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_timed_arm_honours_steps_and_dumps_the_same_outputs_every_run(tmp_path):
    """Two runs of the same small workload: the JSON line reports the requested step count, the dump holds the top-k of
    every query and the unit descriptors, and both runs write identical arrays."""
    nq, ng = 48, 320
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                              "--queries", str(nq), "--gallery", str(ng), "--batch", "64", "--no-e2e", "--parity-steps", "0",
                              "--cpu-embed-sample", "4", "--cpu-sim-sample", "8", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["check"]["indices_equal"]
        assert line["dump_outputs"]["rows_written_of"] == {"values": [nq, nq], "indices": [nq, nq],
                                                           "query_features": [nq, nq], "gallery_features": [ng, ng]}
        dumps.append({p.stem: np.load(p) for p in d.iterdir()})
    a, b = dumps
    assert sorted(a) == ["gallery_features", "indices", "query_features", "values"]
    assert a["values"].shape == a["indices"].shape == (nq, 10) and a["indices"].dtype == np.float64
    assert np.all(np.diff(a["values"], axis=1) <= 0) and a["indices"].min() >= 0 and a["indices"].max() < ng
    assert np.allclose(np.linalg.norm(a["query_features"], axis=1), 1.0, atol=1e-5)
    for name in a:
        assert a[name].dtype == b[name].dtype and np.array_equal(a[name], b[name]), name
