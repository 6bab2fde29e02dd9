"""bench.py on the CPU: the output dump of --dump-outputs and the step count of --impl reference."""
import json
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _outputs(n, rng):
    return {"obs": rng.standard_normal((n, 45)).astype(np.float32), "reward": rng.standard_normal(n).astype(np.float32),
            "done": rng.integers(0, 2, n).astype(np.uint8), "info": rng.standard_normal((n, 32)).astype(np.float32),
            "kin": rng.standard_normal((n, 4))}


def test_dump_writes_every_output_in_float(tmp_path):
    arrays = _outputs(300, np.random.default_rng(0))
    bench.dump_outputs(str(tmp_path / "new"), arrays, suffix="_rank1")
    assert sorted(os.listdir(tmp_path / "new")) == sorted(k + "_rank1.npy" for k in arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "new" / (k + "_rank1.npy"))
        assert got.dtype == (np.float64 if k == "kin" else np.float32)
        assert np.array_equal(got, v.astype(got.dtype))


def test_dump_samples_the_same_envs_of_every_output_beyond_the_limit(tmp_path):
    arrays = _outputs(5000, np.random.default_rng(1))
    limit = 100000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit=limit)
    rows = np.load(tmp_path / "a" / "env_index.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < 5000 and np.array_equal(rows, np.unique(rows))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit + 1024
    for k, v in arrays.items():
        got = np.load(tmp_path / "a" / (k + ".npy"))
        assert np.array_equal(got, v[rows.astype(np.int64)].astype(got.dtype)), k
        assert np.array_equal(got, np.load(tmp_path / "b" / (k + ".npy"))), k   # the sample is fixed


def test_reference_impl_runs_the_steps_asked_for():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scene", "human",
                          "--steps", "41", "--warmup", "1"], capture_output=True, text=True, check=True)
    line = json.loads(out.stdout)
    assert line["steps"] == 41 and " x 41 steps " in line["cpu_baseline"]["sample"]
