#!/usr/bin/env python
"""Cost of running the agent inside the step (smenv_step_agent), 65 536 envs by default, auto reset, per scene:

  step_random       the step with device-drawn random actions (no policy);
  python_loop       the policy from Python: env.step(env.mlp_forward(SM_NET_AGENT, env.obs, n_out=14)[:, :7]) -- one
                    network launch, the output allocation and the action copy around the step;
  agent_det         env.step_agent(explore=False);
  agent_sampled     env.step_agent(explore=True);
  rollout64         env.rollout(64) divided by 64 (the SampleBatch copies included).

Scenes: space_bm and human with the scene's shipped backup policy as the agent, and space_task_bm with the network gate
(shipped risk network, threshold 0.065) and a seeded random agent of input width 29 (29 -> 256 -> 128 -> 14, swish).
Every variant is warmed up, then its steps are timed one by one with CUDA events with the L2 flushed (256 MiB write)
between them (rollout64: once before the 64 steps); the variants run --repeats times, alternating.  Writes one JSON
record with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import scene_config  # noqa: E402
from safemotionsrisk_b200 import abi  # noqa: E402
from safemotionsrisk_b200.config import EnvConfig  # noqa: E402
from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv  # noqa: E402


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def random_agent(path, n_in, nj, seed=0):
    """Keras-fcnet-shaped random weights (Glorot-uniform kernels, zero biases) under agent/ keys."""
    rng = np.random.default_rng(seed)
    dims = [n_in, 256, 128, 2 * nj]
    w = {}
    for i, name in enumerate(("fc_1", "fc_2", "fc_out")):
        lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))
        w["agent/{}/kernel".format(name)] = rng.uniform(-lim, lim, (dims[i], dims[i + 1])).astype(np.float32)
        w["agent/{}/bias".format(name)] = np.zeros(dims[i + 1], np.float32)
    np.savez(path, **w)
    return path


def make_env(scene, envs, tmp):
    cfg = dict(scene_config(scene))
    if scene == "space_task_bm":
        cfg.update(risk_config_dir="risk_networks/state_action/space", risk_threshold=0.065)
    env = SafeMotionsVecEnv(num_envs=envs, config=EnvConfig(**cfg), seed=1, auto_reset=True)
    if scene == "space_task_bm":
        env.load_agent(random_agent(os.path.join(tmp, "agent.npz"), env.scene.obs_size, env.scene.n_joints))
    else:
        env.load_agent()
    env.reset()
    return env


def time_steps(step, steps, warmup, flush):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for i in range(steps):
        flush.fill_(i & 0xff)
        starts[i].record()
        step()
        ends[i].record()
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps


def main():
    p = argparse.ArgumentParser(description=__doc__)
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--steps", type=int, default=64)
    p.add_argument("--warmup", type=int, default=8)
    p.add_argument("--repeats", type=int, default=2)
    p.add_argument("--scenes", default="space_bm,human,space_task_bm")
    p.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                 "profiles", "r03_agent_step_time.json"))
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("agent_step_time.py needs a CUDA device")
    dev = torch.cuda.current_device()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    result = {"tool": "agent_step_time", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev),
              "envs": args.envs, "steps": args.steps, "warmup": args.warmup, "repeats": args.repeats,
              "l2": "flushed between timed steps (256 MiB write); rollout64 once per rollout", "unit": "ms per step",
              "scenes": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for scene in args.scenes.split(","):
            env = make_env(scene, args.envs, tmp)
            nj = env.scene.n_joints

            def loop():
                env.step(env.mlp_forward(abi.SM_NET_AGENT, env.obs, n_out=2 * nj)[:, :nj])

            variants = {"step_random": env.step_random, "python_loop": loop,
                        "agent_det": lambda: env.step_agent(explore=False),
                        "agent_sampled": lambda: env.step_agent(explore=True),
                        "rollout64": lambda: env.rollout(64)}
            rec = {k: [] for k in variants}
            for _ in range(args.repeats):
                for k, fn in variants.items():
                    if k == "rollout64":
                        rec[k].append(time_steps(fn, 2, 1, flush) / 64)
                    else:
                        rec[k].append(time_steps(fn, args.steps, args.warmup, flush))
            rec["agent_det_minus_python_loop"] = min(rec["agent_det"]) - min(rec["python_loop"])
            rec["spread_python_loop"] = max(rec["python_loop"]) - min(rec["python_loop"])
            rec["spread_agent_det"] = max(rec["agent_det"]) - min(rec["agent_det"])
            result["scenes"][scene] = rec
            print(scene, json.dumps(rec), flush=True)
            env.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
