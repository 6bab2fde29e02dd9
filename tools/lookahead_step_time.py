#!/usr/bin/env python
"""Step time of the risk check inside the step, 65 536 envs by default: no gate, the network gate (risk network +
backup policy), the next-state check (risk_state_config 3: one simulated step and a state risk network,
smenv_set_risk_next_state) and the backup-trajectory look-ahead (risk_state_config 4, K backup steps,
smenv_set_risk_lookahead), on space_task_bm (the env of BASELINE.json configs[3]) and human.  The next-state check uses
the state network of `--state-risk-net` (an .npz written by risk_train) or, without it, a seeded random one with the
shipped risk network's hidden widths (512 / 256 / 128, selu, sigmoid), its threshold at the median of its risk over the
reset states unless `--state-risk-threshold` is given; `risky_fraction` matters there, because in exact mode the float32
backup work grows with it.  Random-action rollout with auto reset; every variant is warmed up, then `--steps` steps are
timed one by one with CUDA events, the L2 flushed (256 MiB write) between them as bench.py does.  Prints one JSON line:
ms per step and env-steps/s per variant, the ratios to the ungated step, and the GPU's name and power limit read in the
same run."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import scene_config  # noqa: E402
from safemotionsrisk_b200 import abi, risk_train  # noqa: E402
from safemotionsrisk_b200.config import EnvConfig  # noqa: E402
from safemotionsrisk_b200.scene import Scene  # noqa: E402
from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv  # noqa: E402

THRESHOLD = {"space_task_bm": 0.065, "human": 0.06}   # README.md:223-235, as bench.py --risk-gate


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def time_variant(env, steps, warmup, flush):
    for _ in range(warmup):
        env.step_random()
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    risky = torch.zeros((), dtype=torch.float64, device=env.device)
    for i in range(steps):
        flush.fill_(i & 0xff)
        starts[i].record()
        env.step_random()
        ends[i].record()
        risky += env.info[:, abi.INFO["risky_action"]].sum(dtype=torch.float64)   # after the timed region of the step
    torch.cuda.synchronize()
    total = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    return {"ms_per_step": total / steps, "env_steps_per_s": env.num_envs * steps / (total * 1e-3),
            "risky_fraction": float(risky.item()) / (env.num_envs * steps)}


def random_state_net(scene, path, seed=0):
    """A seeded random state risk network for `scene` (risk observation -> 512 -> 256 -> 128 -> 1) written to `path`."""
    sc = Scene(scene_config(scene))
    torch.manual_seed(seed)
    model = risk_train.build_model(sc.obs_size - sc.obs_target_size, [512, 256, 128], "selu")
    risk_train.export_weights(model, path, "selu", "sigmoid")
    return path


def time_next_state(scene, args, flush, tmp):
    net = args.state_risk_net or random_state_net(scene, os.path.join(tmp, "state_net_{}.npz".format(scene)))
    cfg = EnvConfig(**dict(scene_config(scene), risk_config_dir=net, risk_threshold=0.5, risk_state_config=3))
    env = SafeMotionsVecEnv(num_envs=args.envs, config=cfg, seed=1)
    env.reset()
    thr = args.state_risk_threshold
    if thr is None:
        thr = float(torch.quantile(env.mlp_forward(0, env.risk_observation())[:, 0], 0.5).item())
    env.set_risk_gate(thr)
    r = time_variant(env, args.steps, args.warmup, flush)
    r.update(threshold=thr, state_risk_net=args.state_risk_net or "random (seed 0, 512/256/128)")
    env.close()
    return r


def main():
    p = argparse.ArgumentParser(description=__doc__)
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--backup-steps", type=int, default=20)
    p.add_argument("--scenes", default="space_task_bm,human")
    p.add_argument("--state-risk-net", default=None, help="state risk network (.npz) of the next-state variant")
    p.add_argument("--state-risk-threshold", type=float, default=None)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lookahead_step_time.py needs a CUDA device")
    dev = torch.cuda.current_device()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    result = {"tool": "lookahead_step_time", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev),
              "envs": args.envs, "steps": args.steps, "warmup": args.warmup, "backup_steps": args.backup_steps,
              "l2": "flushed between timed steps (256 MiB write)", "scenes": {}}
    tmp = tempfile.mkdtemp(prefix="lookahead_step_time_")
    for scene in args.scenes.split(","):
        env = SafeMotionsVecEnv(num_envs=args.envs, config=scene_config(scene), seed=1)
        env.load_networks()
        env.reset()
        thr = THRESHOLD.get(scene, 0.065)
        r = {"threshold": thr}
        r["ungated"] = time_variant(env, args.steps, args.warmup, flush)
        env.set_risk_gate(thr)
        r["network_gate"] = time_variant(env, args.steps, args.warmup, flush)
        env.set_risk_lookahead(args.backup_steps)
        r["lookahead"] = time_variant(env, args.steps, args.warmup, flush)
        r["lookahead_over_ungated"] = r["lookahead"]["ms_per_step"] / r["ungated"]["ms_per_step"]
        env.close()
        del env
        r["next_state"] = time_next_state(scene, args, flush, tmp)
        r["next_state_over_ungated"] = r["next_state"]["ms_per_step"] / r["ungated"]["ms_per_step"]
        result["scenes"][scene] = r
    shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
