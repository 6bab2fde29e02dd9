"""bench.py --dump-outputs on the device: the files hold what the last of the K timed steps returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_holds_the_last_timed_step(tmp_path):
    from safemotionsrisk_b200 import human_backup_config
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    n, warmup, steps = 4096, 4, 5
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                          "--warmup", str(warmup), "--envs", str(n), "--scene", "human", "--no-scenes", "--no-e2e",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout)["steps"] == steps
    # the same env stepped as often here: bench seeds rank 0's env with 0 and runs the warm-up steps before the timed ones
    env = SafeMotionsVecEnv(num_envs=n, device="cuda:0", seed=0, auto_reset=True, config=human_backup_config())
    env.reset()
    for _ in range(warmup + steps):
        want = env.step_random()
    torch.cuda.synchronize()
    for name, t in zip(("obs", "reward", "done", "info"), want):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float32 and got.shape == tuple(t.shape), name
        assert np.array_equal(got, t.cpu().numpy().astype(np.float32)), name
    env.close()
