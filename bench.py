#!/usr/bin/env python
"""Benchmark of the env-step hot path (BASELINE.json: env-steps/sec, whole box, device-timed).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--scene ball|space] [--envs 65536] [--impl reference]
                    [--dump-outputs DIR]

Own arm (default): one process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE), each rank steps its own shard of
`--envs` environments with device-generated random actions (get_random_action, safe_motions_base.py:1327-1328) and
auto-reset; no collective on the step path.  K steps are timed with CUDA events on the launching stream, the L2 is
flushed between timed steps, the max over ranks is taken and rank 0 prints ONE JSON line.
`e2e` is the same metric through the public host-buffer API (SafeMotionsVecEnv.step_host): pinned host actions in,
observations / rewards / dones out, copies inside the timed region.
`--impl reference` times the CPU restatement of the reference path (oracle/, all host threads) on the same workload;
the real PyBullet/klimits env cannot be installed in this image (no network, SURVEY.md section 8c).
`--dump-outputs DIR` writes what the last timed step returned (obs, reward, done, info of the headline scene) as
DIR/<name>.npy, so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (whole box, device-timed)"
UNIT = "env-steps/s"
F_FIXED = 3300.0  # SURVEY.md 8d: safe range + FK + interpolation + reward flops per env step


def scene_config(name):
    from safemotionsrisk_b200 import ball_backup_config, space_backup_config
    if name == "ball":
        return ball_backup_config()
    if name == "space":
        return space_backup_config()
    if name == "space_task":
        from safemotionsrisk_b200 import space_task_config
        return space_task_config()
    if name == "space_task_bm":
        from safemotionsrisk_b200 import space_task_config
        return space_task_config(ball_machine_mode=True)
    if name == "space_bm":
        return space_backup_config(ball_machine_mode=True)
    if name == "ball_bm":
        return ball_backup_config(ball_machine_mode=True)
    if name == "human":
        from safemotionsrisk_b200 import human_backup_config
        return human_backup_config()
    if name == "human_bm":
        from safemotionsrisk_b200 import human_backup_config
        return human_backup_config(ball_machine_mode=True)
    raise SystemExit("unknown scene " + name)


WORKLOAD = {"ball": "Ball env (moving ball obstacles) batched random-action rollout, 65,536 envs per B200 "
                    "(BASELINE.json configs[1])",
            "space": "Space env (planet_mode, obstacle_scene=5) batched random-action rollout",
            "space_bm": "Space env, ball_machine_mode (shipped checkpoints' robot)",
            "ball_bm": "Ball env, ball_machine_mode (shipped checkpoints' robot)",
            "human": "Human env (human arms moved by the shipped human policy, braking-trajectory check of the nested "
                     "env) batched random-action rollout, 65,536 envs per B200 (BASELINE.json configs[2])",
            "human_bm": "Human env, ball_machine_mode (shipped checkpoints' robot)",
            "space_task": "Space reaching task (SafeMotionsEnv with target points, README.md:223)",
            "space_task_bm": "Space reaching task, ball_machine_mode (BASELINE.json configs[3] env)"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        self.nvml_rows, self.nvml_stop, self.nvml_thread = [], threading.Event(), None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        try:   # the same counters straight from NVML every 5 ms: one nvidia-smi query takes longer than a short timed region
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml_thread = threading.Thread(target=self._read_nvml, daemon=True)
            self.nvml_thread.start()
        except Exception:
            self.nvml_thread = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def _read_nvml(self):
        n = self.nvml
        bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        try:
            mx = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
        except Exception:
            mx = None
        while not self.nvml_stop.is_set():
            try:
                clk = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.nvml_rows.append((time.time(), clk, mx, [k for k, b in bits.items() if mask & b]))
            except Exception:
                break
            time.sleep(0.005)

    def stop(self, t0, t1):
        if self.proc is None and self.nvml_thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.nvml_stop.set()
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, mx = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            if t0 - 0.01 <= ts <= t1 + 0.03:
                sm.append(clk)
                for name, val in zip(names, parts[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        n_smi = len(sm)
        nv = [r for r in self.nvml_rows if t0 <= r[0] <= t1]
        for _, clk, nmx, rs in nv:
            sm.append(clk)
            mx = mx if mx is not None else nmx
            reasons.update(rs)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_nvidia_smi": n_smi, "samples_nvml": len(nv),
                "source": "nvidia-smi -lms 20 and NVML every 5 ms, samples inside the timed region"}


def pcie_bandwidth(dev, nbytes, reps=10):
    """GB/s of a pinned host <-> device copy of nbytes (the D2H block of one env range of the host-buffer step)."""
    import torch
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = {"bytes": int(nbytes)}
    for name, src, dst in (("d2h", d, h), ("h2d", h, d)):
        for _ in range(2):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            dst.copy_(src, non_blocking=True)
        e.record()
        torch.cuda.synchronize(dev)
        out[name] = nbytes * reps / (s.elapsed_time(e) * 1e-3) / 1e9
    return out


def cpu_reference_run(scene_name, envs_per_thread, steps, warmup, threads, target_seconds=None):
    """Times the CPU oracle on `threads` host threads (ctypes releases the GIL); returns env-steps/s and a note.
    With target_seconds the number of timed steps is chosen from the duration of the warm-up steps so that the
    sample is about that long (bounded sample of the same workload)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle
    from safemotionsrisk_b200.scene import Scene
    scene = Scene(scene_config(scene_name))
    rng = np.random.default_rng(0)
    lo, hi = np.array(scene.pos_lo), np.array(scene.pos_hi)
    shards = []
    for t in range(threads):
        env = oracle.OracleEnvs(scene, envs_per_thread)
        q = rng.uniform(0.5 * lo, 0.5 * hi, (envs_per_thread, scene.n_joints))
        ob = np.zeros((envs_per_thread, 16))
        if scene.struct.n_obstacles and scene.struct.obst_kind[0] == 1:
            ob[:, 0] = rng.integers(0, scene.struct.planet_steps, envs_per_thread)
        elif scene.struct.n_obstacles:
            ob[:, 2:5], ob[:, 5:8] = [2.4, 0.3, 1.0], [-5.5, -0.6, 1.5]
            ob[:, 13], ob[:, 14], ob[:, 15] = 1, 200, 150
        tgt = np.tile([0.3, 0.3, 0.5], (envs_per_thread, 1)) if scene.struct.use_target_points else None
        env.set_state(q, np.zeros_like(q), np.zeros_like(q), ob, tgt)
        env._q0, env._ob0, env._tgt = q, ob, tgt
        if scene.struct.human.enabled:   # the human starts with its arms lowered, at rest, first target in front of it
            hq = np.tile([0.3, -0.3, 0.2, -0.8, -0.3, -0.3, -0.2, -0.8], (envs_per_thread, 1)) + \
                rng.uniform(-0.1, 0.1, (envs_per_thread, 8))
            env._h0 = (hq, np.zeros_like(hq), np.zeros_like(hq), np.tile([0.4, -0.3, 0.3], (envs_per_thread, 1)),
                       np.zeros(envs_per_thread, dtype=np.int32))
            env.set_human_state(*env._h0)
        shards.append(env)
    acts = rng.uniform(-1, 1, (envs_per_thread, scene.n_joints)).astype(np.float32)
    nb = np.tile(np.array([2.4, 0.3, 1.0, -5.5, -0.6, 1.5, 0.3, 0.1, 0.0, 1.0, 200, 150.0]), (envs_per_thread, 1))

    hacts = rng.uniform(-1, 1, (envs_per_thread, 8)).astype(np.float32)
    htgt = np.tile([0.35, 0.3, 0.35], (envs_per_thread, 1))

    def one_step(env):
        if scene.struct.human.enabled:
            _, _, done, _, _ = env.step_human(acts, hacts, htgt)
        else:
            _, _, done, _, _ = env.step(acts, nb, env._tgt)
        if done.any():  # episodes restart from the same pool of start states
            env.set_state(env._q0, np.zeros_like(env._q0), np.zeros_like(env._q0), env._ob0, env._tgt)
            if scene.struct.human.enabled:
                env.set_human_state(*env._h0)
    with ThreadPoolExecutor(threads) as pool:
        tw = time.perf_counter()
        for _ in range(max(1, warmup)):
            list(pool.map(one_step, shards))
        tw = (time.perf_counter() - tw) / max(1, warmup)
        if target_seconds is not None:
            steps = int(min(max(2, target_seconds / max(tw, 1e-6)), 400))
        t0 = time.perf_counter()
        for _ in range(steps):
            list(pool.map(one_step, shards))
        dt = time.perf_counter() - t0
    total = threads * envs_per_thread * steps
    return total / dt, dt, total, steps


_STDOUT_FD = None


def _quiet_stdout():
    """Everything printed to stdout from here on (NCCL's version banner, library chatter) goes to stderr; the one JSON
    line of the contract is written to the real stdout by _emit."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    os.write(_STDOUT_FD if _STDOUT_FD is not None else 1, (line + "\n").encode())


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays, limit=DUMP_LIMIT_BYTES, suffix=""):
    """Writes each per-env array (first axis: env) as <path>/<name><suffix>.npy, float64 kept, everything else as
    float32.  When they exceed `limit` bytes together, every array keeps the same fixed, seeded sample of env rows and
    the sampled env indices go to env_index<suffix>.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64 if np.asarray(v).dtype == np.float64 else np.float32)
              for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v.nbytes for v in arrays.values()) // max(n, 1)
    if n * row_bytes > limit:
        rows = np.sort(np.random.default_rng(0).choice(n, limit // (row_bytes + 8), replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + suffix + ".npy"), v)


def bind_to_gpu_cpus(local_rank):
    """Pins this rank to the CPUs nearest to its GPU (NVML's ideal affinity) before any pinned host buffer exists, so
    that the staging buffers of the host-buffer step are first touched on the GPU's own NUMA node.  Returns what was
    done for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w in range(words) for b in range(64) if (mask[w] >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"bound": False, "why": "no overlap between the GPU's CPU set and this process' affinity"}
        os.sched_setaffinity(0, allowed)
        return {"bound": True, "cpus": "{}-{} ({})".format(allowed[0], allowed[-1], len(allowed))}
    except Exception as e:  # the bench runs unbound
        return {"bound": False, "why": repr(e)[:120]}


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--scene", default="human",
                    help="headline workload: human = BASELINE.json configs[2] (the config the 1/2/4/8 sweep is quoted on); the "
                         "scenes of --scenes are measured after it and reported in the same line")
    ap.add_argument("--envs", type=int, default=65536, help="environments per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--host-chunks", type=int, default=2,
                    help="env ranges of the host-buffer step whose copies and kernels overlap (smenv_step_host)")
    ap.add_argument("--risk-gate", action="store_true",
                    help="risk network + backup policy (tensor cores) in front of every step (BASELINE.json configs[3])")
    ap.add_argument("--risk-threshold", type=float, default=None)
    ap.add_argument("--scenes", default="space,space_bm,ball,human",
                    help="further scenes measured (device-timed, shorter) after the main one and reported under 'scenes'")
    ap.add_argument("--no-scenes", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write obs, reward, done and info of the last timed step of the headline scene as DIR/<name>.npy "
                         "(float32, at most 64 MiB in all: a fixed, seeded sample of envs beyond that; with several "
                         "ranks each rank writes <name>_rank<r>.npy)")
    args = ap.parse_args()
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the device step (--impl b200)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    threads = os.cpu_count() or 1
    config = {"workload": WORKLOAD[args.scene], "scene": args.scene, "envs_per_gpu": args.envs,
              "actions": "device Philox U(-1,1)", "auto_reset": True, "parallelism": "env-shards x{}".format(world),
              "l2": "flushed between timed steps (256 MiB write)"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # bounded sample: small shards so that `steps` finish within minutes on the host cores
        per_thread = 1024 if args.scene.startswith("ball") else 8 if args.scene.startswith("human") else 64
        # each of the K steps is one oracle step of the bounded sample
        val, dt, total, steps = cpu_reference_run(args.scene, per_thread, args.steps, min(max(args.warmup, 1), 2),
                                                  threads)
        sample = "{} host threads x {} envs x {} steps of the same scene ({} env-steps in {:.1f} s)".format(
            threads, per_thread, steps, total, dt)
        _emit(json.dumps({
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": min(args.warmup, 2), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "note": "oracle restatement -- NOT the PyBullet reference (pybullet/klimits cannot be "
                                     "installed in this image)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    args.all_cpus = sorted(os.sched_getaffinity(0))   # the CPU baseline leg runs on every host core again
    args.host_affinity = bind_to_gpu_cpus(local_rank)
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    fma_peaks = measure_fma_peaks(local_rank)
    main = measure_scene(args.scene, args, dev, rank, world, local_rank, fma_peaks, steps=args.steps,
                         full=True, with_cpu=(rank == 0 and world == 1 and not args.no_cpu_baseline),
                         dump=args.dump_outputs)
    # the other scenes of BASELINE.json on the same box, so that the driver's record carries the north-star scene (Space,
    # also with the robot of the shipped checkpoints) next to the headline workload: shorter runs, device-timed only
    extra = {}
    if not args.no_scenes:
        for name in [x for x in args.scenes.split(",") if x and x != args.scene]:
            r = measure_scene(name, args, dev, rank, world, local_rank, fma_peaks, steps=min(args.steps, 100),
                              full=False, with_cpu=False)
            if rank == 0:
                extra[name] = {k: r[k] for k in ("value", "ms_per_step", "workload", "gpu_launches", "roofline")}
                extra[name]["launch"] = r["config"]["launch"]
                extra[name]["e2e"] = r["e2e"]
    pin = None
    if rank == 0 and world == 1 and not args.no_scenes:
        pin = behavioural_pin(dev)
    if rank == 0:
        out = {"impl": "b200", "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world,
               "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": main["ms_per_step"],
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f64 joint space / f32 geometry", "data": "synthetic", "config": main["config"],
               "clocks": main["clocks"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
               "roofline": main["roofline"], "cpu_baseline": main["cpu_baseline"], "episode_stats": main["episode_stats"],
               "scenes": extra, "behavioural_pin": pin}
        _emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


def behavioural_pin(dev, envs=16384, steps=60):
    """The only reference-held artefacts that can pin the restated env are the shipped network weights (SURVEY 8c item 5):
    the backup policy, trained in the real PyBullet env, must keep far more 20-step episodes collision free in THIS env
    than random actions do.  Collision-termination rate per finished episode, scenes with the robot of the checkpoints."""
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    out = {"what": "collision terminations per finished episode over {} steps of {} envs from pool starts: shipped backup "
                   "policy (deterministic mean action, tensor cores) vs uniform random actions".format(steps, envs)}
    for name in ("space_bm", "ball_bm"):
        rates = {}
        for mode in ("backup_policy", "random_actions"):
            env = SafeMotionsVecEnv(num_envs=envs, device=dev, seed=11, auto_reset=True, config=scene_config(name))
            env.load_networks()
            env.reset()
            env.stats.zero_()
            for _ in range(steps):
                if mode == "backup_policy":
                    env.step(env.backup_policy_actions())
                else:
                    env.step_random()
            st = env.episode_statistics().cpu().numpy()
            rates[mode] = float((st[3 + 3] + st[3 + 4] + st[3 + 5]) / max(st[0], 1))
            env.close()
        out[name] = rates
    return out


def measure_fma_peaks(device_index):
    """FP32 / FP64 FMA throughput of this GPU measured by the library's micro-benchmark (TFLOP/s)."""
    import ctypes as C
    from safemotionsrisk_b200 import cabi
    f32, f64 = C.c_double(), C.c_double()
    cabi.check(cabi.load().smenv_measure_fma_peaks(int(device_index), C.byref(f32), C.byref(f64)), "smenv_measure_fma_peaks")
    return {"fp32": f32.value, "fp64": f64.value}


def measure_scene(scene_name, args, dev, rank, world, local_rank, fma_peaks, steps, full, with_cpu, dump=None):
    """One workload on this rank's GPU: K device-timed steps (max over ranks), roofline of the dominant kernel, and (full)
    the end-to-end number through the host-buffer API.  dump: directory for the outputs of the last timed step."""
    import torch
    import torch.distributed as dist
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    threads = os.cpu_count() or 1
    config = {"workload": WORKLOAD[scene_name], "scene": scene_name, "envs_per_gpu": args.envs,
              "actions": "device Philox U(-1,1)", "auto_reset": True, "parallelism": "env-shards x{}".format(world),
              "l2": "flushed between timed steps (256 MiB write)"}
    cfg = scene_config(scene_name)
    env = SafeMotionsVecEnv(num_envs=args.envs, device=dev, seed=1000 * rank, auto_reset=True, config=cfg)
    config["launch"] = env.launch_config()
    config["host_affinity"] = args.host_affinity
    gate_thr = None
    if args.risk_gate and full:
        env.load_networks()
        gate_thr = args.risk_threshold if args.risk_threshold is not None else \
            (0.105 if scene_name.startswith("ball") else 0.06 if scene_name.startswith("human") else 0.065)  # README.md:223-235
        env.set_risk_gate(gate_thr)
        config["risk_gate"] = {"threshold": gate_thr, "networks": "risk obs+7-512-256-128-1 selu + backup policy "
                               "obs-256-128-14 swish/tanh, fp16 x fp16 -> fp32 on tcgen05, inside the step"}
        config["workload"] += " + state-action risk network and backup policy in the step loop"

    def one_step():
        return env.step_random()
    sampler = ClockSampler(local_rank) if rank == 0 else None   # started early: nvidia-smi needs ~0.1 s to its first sample
    env.reset()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for _ in range(max(3, args.warmup)):
        one_step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    launches0 = env.launch_count()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    t_wall0 = time.time()
    for i in range(steps):
        flush.fill_(i & 0xff)  # evict the env state from L2 (outside the timed region of the step)
        starts[i].record()
        last = one_step()
        ends[i].record()
    torch.cuda.synchronize(dev)
    t_wall1 = time.time()
    if dump is not None:   # read before the counter and kernel-timing passes below step the env again
        dump_outputs(dump, {k: t.cpu().numpy() for k, t in zip(("obs", "reward", "done", "info"), last)},
                     limit=DUMP_LIMIT_BYTES // world, suffix="_rank{}".format(rank) if world > 1 else "")
    launches = env.launch_count() - launches0
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = float(sum(step_ms))
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tmax_ms = float(t.item())
    value = world * args.envs * steps / (tmax_ms * 1e-3)

    # end-of-iteration episode statistics: the only collective of the design (train.py:59-117 custom_metrics)
    stats = env.episode_statistics()
    t0 = time.perf_counter()
    if world > 1:
        dist.all_reduce(stats)
        torch.cuda.synchronize(dev)
    stats_ms = 1e3 * (time.perf_counter() - t0)
    stats = stats.cpu().numpy()

    # ---------------- roofline of the dominant kernel: algorithmic flops from device counters, kernel durations from
    # CUDA events around each launch (measurement mode of the library, separate pass after the timed region)
    if gate_thr is not None:
        env.set_risk_gate(None)
    env.enable_counters(True)
    env.counters(reset=True)
    for _ in range(3):
        env.step_random()
    c = env.counters()
    env.enable_counters(False)
    steps_counted = max(1, c["env_steps"])
    n_dot, n_iter = c["support_dots"] / steps_counted, c["gjk_iters"] / steps_counted
    sc_nj = env.scene.struct.n_joints
    env.kernel_timing(True)
    env.kernel_times(reset=True)
    for i in range(min(steps, 50)):
        flush.fill_(i & 0xff)
        env.step_random()
    ktimes, _ = env.kernel_times()
    env.kernel_timing(False)
    ksum = sum(ktimes.values())
    # algorithmic flops per env-step attributed to each kernel (SURVEY.md 8d: 300 flops per joint range + 60 per joint
    # interpolation; a position-bound solve costs what its braking-profile intervals cost, ~60 flops each, counted on
    # the device)
    hj, hs = c["heavy_joints"] / steps_counted, c["heavy_solves"] / steps_counted
    intervals = c["reserved"] / steps_counted      # braking-profile intervals evaluated by joint_solve_kernel
    brake_poses, brake_bounds = c["brake_poses"] / steps_counted, c["brake_pair_bounds"] / steps_counted
    kflops = {"joint_kernel": (sc_nj - hj) * 360.0, "joint_heavy_kernel": hj * 360.0 + intervals * 60.0,
              "contact_plan_kernel": 8 * 600.0, "distance_plan_kernel": 600.0,
              "gjk_kernel": 5.0 * n_dot + 100.0 * n_iter, "finish_kernel": 200.0,
              # Human scene: policy 2 x 44 544 MAC on the tensor cores; range + braking steps of 8 joints; the pose
              # checks from the device counters: per pose the FK of 8 joints (axis-angle matrix + two 3x3 products + the
              # translation: 140 flops each), 30 table points (18 flops) and 7 capsule tests (70), per evaluated convex
              # pair a sphere bound of 14 flops; culled group pairs are NOT counted.  GJK counted with the main GJK launch
              "human_policy": 2.0 * 44544.0, "human_joint_kernels": 8 * 360.0, "human_brake_traj_kernel": 8 * 3 * 360.0,
              "human_brake_plan_kernel": brake_poses * (8 * 140.0 + 30 * 18.0 + 7 * 70.0) + brake_bounds * 14.0,
              "human_brake_gjk": 0.0, "human_advance_outcome": 8 * 60.0 + 24 * 300.0}
    # the nested env's slots of a scene without a human hold only the event overhead (~3 us)
    ktimes = {k: v for k, v in ktimes.items() if v > 0.01 or not k.startswith("human")}
    kbound = {"joint_kernel": "fp64", "joint_heavy_kernel": "fp64", "human_joint_kernels": "fp64",
              "human_brake_traj_kernel": "fp64"}
    f_step = F_FIXED + 5.0 * n_dot + 100.0 * n_iter
    dom = max(ktimes, key=ktimes.get)
    kernel_ms = ktimes[dom]
    per_gpu_steps_s = args.envs / (statistics.mean(step_ms) * 1e-3)
    achieved_tflops = args.envs * kflops[dom] / (kernel_ms * 1e-3) / 1e12
    bound = kbound.get(dom, "fp32")
    dom_peak = fma_peaks[bound]
    sc = env.scene.struct
    bytes_step = 2 * (8 * 32 + 8 * 16 + 16 + 8) + 4 * sc.n_joints + 4 * sc.obs_size + 4 + 1 + 4 + 4 * 32
    if sc.human.enabled:   # + state of the nested env in and out, its observation and actions
        bytes_step += 2 * (8 * 32 + 8 * 32) + 4 * 40 + 4 * 8 + 2 * 8 * 8 * 3
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    uncull = {"space": 1.51e6, "space_bm": 1.71e6, "ball": 0.15e6, "ball_bm": 0.35e6, "space_task": 1.51e6,
              "space_task_bm": 1.71e6, "human": 3.6e6, "human_bm": 3.8e6}[scene_name]
    traffic = None  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
    for tf in ("r02c_traffic.json", "r02b_traffic.json", "r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", tf)) as f:
                traffic = json.load(f)["bytes_per_launch"].get(scene_name, {}).get(dom)
            if traffic is not None:
                break
        except Exception:
            pass
    roofline = {"bound": bound, "achieved": achieved_tflops, "peak": dom_peak, "unit": "TFLOP/s",
                "frac": achieved_tflops / dom_peak, "traffic": traffic,
                "traffic_unit": "DRAM bytes per launch (profiles/r0*_traffic.json, ncu --set full, 65536 envs)",
                "peak_source": "measured on this GPU before the run: dependent-free {} FMA chains on all SMs "
                               "(smenv_measure_fma_peaks); MEASURED_PEAKS.json holds no vector-pipe entry".format(bound),
                "measured_fma_peaks_tflops": fma_peaks,
                "kernel": dom, "kernel_ms": kernel_ms, "kernel_share_of_step": kernel_ms / ksum,
                "kernel_flops_per_env_step": kflops[dom],
                "kernels_ms": ktimes, "flops_per_env_step": f_step, "support_dots_per_env_step": n_dot,
                "gjk_iters_per_env_step": n_iter, "gjk_pairs_per_env_step": c["gjk_calls"] / steps_counted,
                "position_solve_intervals_per_env_step": intervals,
                "brake_poses_per_env_step": brake_poses, "brake_pair_bounds_per_env_step": brake_bounds,
                "whole_step": {"achieved": per_gpu_steps_s * f_step / 1e12,
                               "frac": per_gpu_steps_s * f_step / 1e12 / fma_peaks["fp32"],
                               "unculled_reference_flops_per_env_step": uncull},
                "hbm": {"achieved": per_gpu_steps_s * bytes_step / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": per_gpu_steps_s * bytes_step / 1e9 / hbm_peak, "bytes_per_env_step": bytes_step,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}
    if gate_thr is not None:
        env.set_risk_gate(gate_thr)

    if gate_thr is not None:  # the tensor-core part: time of the gate alone, dense flops against the bf16/fp16 peak
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        env.step_random()
        g0.record()
        for _ in range(10):
            env.risk_gate(gate_thr)
        g1.record()
        torch.cuda.synchronize(dev)
        gate_ms = g0.elapsed_time(g1) / 10
        ow = sc.obs_size
        n_tp = 3 * (sc.obs_add_tp_pos + sc.obs_add_tp_rel) if sc.use_target_points else 0
        risk_mac = (ow - n_tp + sc_nj) * 512 + 512 * 256 + 256 * 128 + 128
        backup_mac = (ow - n_tp) * 256 + 256 * 128 + 128 * sc_nj
        risky_frac = float(env.info[:, 16].mean().item())
        # tensor cores: the risk network on every row; float32 CUDA cores: the risk network on the rows within the band
        # of the threshold and the backup policy on the risky rows (smenv_set_gate_exact, the default)
        gflop = 2.0 * args.envs * risk_mac
        tpeak = peaks.get("bf16_tflops", 2250.0)
        roofline["risk_gate"] = {"bound": "tensor", "kernel": "mlp_kernel (risk network, all rows) + gate_band_kernel + "
                                 "mlp_exact_kernel (near-threshold rows) + risk_decide_kernel + mlp_exact_kernel (backup "
                                 "policy, risky rows)", "ms": gate_ms,
                                 "achieved": gflop / (gate_ms * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                                 "frac": gflop / (gate_ms * 1e-3) / 1e12 / tpeak,
                                 "flops_counted": "risk network on all rows only (2 x {} MAC per row); the float32 subset "
                                                  "passes add 2 x {} MAC per risky row".format(risk_mac, backup_mac),
                                 "peak_source": "MEASURED_PEAKS.json bf16_tflops" if peaks else "nominal",
                                 "risky_fraction": risky_frac}

    # ---------------- end to end through the host-buffer API
    e2e = None
    if not args.no_e2e:
        rng = np.random.default_rng(rank)
        acts = rng.uniform(-1, 1, (args.envs, sc.n_joints)).astype(np.float32)
        env.host_actions[...] = acts   # the step's inputs sit in the pinned host buffer the sampler writes into
        acts = None                    # step_host(None): no pageable -> pinned copy, the H2D copy happens every step
        for _ in range(3):
            env.step_host(acts, None, chunks=args.host_chunks)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        k_e2e = min(steps, 100 if full else 40)
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            env.step_host(acts, None, chunks=args.host_chunks)
        torch.cuda.synchronize(dev)
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": world * args.envs * k_e2e / float(te.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(env.host_actions.nbytes), "d2h_bytes_per_step": int(args.envs * (4 * sc.obs_size + 4 + 1)),
               "steps": k_e2e, "host_chunks": args.host_chunks,
               "api": "SafeMotionsVecEnv.step_host -> smenv_step_host (actions in the pinned host buffer, H2D, step, "
                      "D2H of obs / reward / done into pinned host buffers, all inside the timed region)"}
        try:   # the pinned-copy bandwidth of this box at the size the step moves: what bounds the part of e2e the step cannot hide
            e2e["pcie_gbs"] = pcie_bandwidth(dev, max(1 << 20, e2e["d2h_bytes_per_step"] // max(1, args.host_chunks)))
        except Exception as ex:   # a measurement aid, never a reason to lose the line
            e2e["pcie_gbs"] = {"error": str(ex)[:100]}

    # ---------------- CPU baseline beside it (rank 0, N = 1 only, bounded sample)
    cpu = None
    if with_cpu:
        os.sched_setaffinity(0, args.all_cpus)
        per_thread = 1024 if scene_name.startswith("ball") else 8 if scene_name.startswith("human") else 64
        val, dt, total, csteps = cpu_reference_run(scene_name, per_thread, 20, 1, threads, target_seconds=15.0)
        cpu = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "{} host threads x {} envs x {} steps of the same scene ({} env-steps in {:.1f} s)".format(
                   threads, per_thread, csteps, total, dt),
               "note": "oracle restatement (C, -O2) -- NOT the PyBullet reference (not installable here); its start states "
                       "are a fixed synthetic set (mid-range poses at rest, one ball launch), not the pool distribution "
                       "of the GPU run: same scene and step function, simpler state distribution"}
    out = {"value": value, "ms_per_step": tmax_ms / steps, "workload": config["workload"], "config": config,
           "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
           "episode_stats": {"episodes": float(stats[0]), "mean_return": float(stats[1] / max(stats[0], 1)),
                             "mean_length": float(stats[2] / max(stats[0], 1)),
                             "by_termination_reason": {str(r): float(stats[3 + r]) for r in range(1, 6)},
                             "allreduce_ms": stats_ms}}
    env.close()
    del env, flush
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    sys.exit(main())
