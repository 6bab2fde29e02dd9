#!/usr/bin/env python
"""Cost of risk_check_initial_backup_trajectory, 65 536 envs by default, random actions with auto reset, the network gate
on (risk network + backup policy, the shipped networks of the scene at README.md's threshold):

  (a) flag_off         space_task_bm without the check;
  (b) pool_check       the same with the check on the start pool (smenv_set_initial_backup_check): resets draw from the
                       entries that passed, the step is the ungated-count step of (a);
  (c) host_loop        the check as the package ran it before, reproduced here through public methods on the same build:
                       the step without device auto reset, then, if an episode ended, reset(done) and up to 8 rounds of
                       initial_backup_trajectory_unsafe over all envs with a re-reset of the unsafe finished envs;
  (d) check_ms         the one-time pool check inside fill_pools (host clock around set_initial_backup_check, which ends
                       in a stream synchronise) for space_task_bm and human, with the entries checked and passed.

Every variant is warmed up, then its steps are timed one by one with CUDA events, the L2 flushed (256 MiB write) between
them as bench.py does; the events of (c) enclose the host round trips of the loop.  Prints one JSON line with the GPU's
name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import scene_config  # noqa: E402
from safemotionsrisk_b200.config import EnvConfig  # noqa: E402
from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv  # noqa: E402

NETWORKS = {"space_task_bm": "space", "human": "human"}
THRESHOLD = {"space_task_bm": 0.065, "human": 0.06}   # README.md:223-235, as bench.py --risk-gate


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def make_env(scene, envs, check, auto_reset=True):
    cfg = EnvConfig(**dict(scene_config(scene), risk_config_dir="risk_networks/state_action/" + NETWORKS[scene],
                           risk_threshold=THRESHOLD[scene], risk_check_initial_backup_trajectory=check))
    return SafeMotionsVecEnv(num_envs=envs, config=cfg, seed=1, auto_reset=auto_reset)


def host_loop_step(env, max_rounds=8):
    """One step of the former host-side check: device step without auto reset, then re-resets on the host."""
    env.step_random()
    done = env.done.clone()
    if bool(done.any().item()):
        out = (env.reward.clone(), env.term_reason.clone(), env.info.clone())
        env.reset(done)
        for _ in range(max_rounds):
            unsafe = env.initial_backup_trajectory_unsafe() & done.bool()
            if not bool(unsafe.any().item()):
                break
            env.reset(unsafe.to(torch.uint8))
        env.done.copy_(done)
        env.reward.copy_(out[0]); env.term_reason.copy_(out[1]); env.info.copy_(out[2])


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
    total = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    return {"ms_per_step": total / steps, "steps": steps}


def check_time(scene, envs, backup_steps):
    env = make_env(scene, envs, check=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    env.set_initial_backup_check(backup_steps)
    ms = (time.perf_counter() - t0) * 1e3
    checked, passed = env.initial_backup_check_counts()
    env.close()
    return {"check_ms": ms, "checked": checked, "passed": passed}


def main():
    p = argparse.ArgumentParser(description=__doc__)
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--host-loop-steps", type=int, default=40)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--repeats", type=int, default=2, help="(a) and (b) are timed this many times, alternating")
    p.add_argument("--backup-steps", type=int, default=20)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("initial_check_time.py needs a CUDA device")
    dev = torch.cuda.current_device()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    scene = "space_task_bm"
    result = {"tool": "initial_check_time", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev),
              "scene": scene, "envs": args.envs, "steps": args.steps, "warmup": args.warmup,
              "backup_steps": args.backup_steps, "threshold": THRESHOLD[scene], "actions": "random, auto reset",
              "l2": "flushed between timed steps (256 MiB write)"}
    envs = {"flag_off": make_env(scene, args.envs, check=False), "pool_check": make_env(scene, args.envs, check=True)}
    for k, env in envs.items():
        env.reset()
        result.setdefault(k, [])
    for _ in range(args.repeats):
        for k, env in envs.items():
            result[k].append(time_steps(env.step_random, args.steps, args.warmup, flush)["ms_per_step"])
    result["pool_check_counts"] = envs["pool_check"].initial_backup_check_counts()
    for env in envs.values():
        env.close()
    del envs
    loop = make_env(scene, args.envs, check=False, auto_reset=False)
    loop.reset()
    result["host_loop"] = time_steps(lambda: host_loop_step(loop), args.host_loop_steps, 2, flush)["ms_per_step"]
    loop.close()
    a, b = min(result["flag_off"]), min(result["pool_check"])
    result["pool_check_over_flag_off"] = b / a
    result["host_loop_over_flag_off"] = result["host_loop"] / a
    result["check_ms"] = {s: check_time(s, args.envs, args.backup_steps) for s in ("space_task_bm", "human")}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
