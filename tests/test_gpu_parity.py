"""Parity of the CUDA path (through the C ABI, libsmenv.so) against the CPU oracle and the golden vectors.

Tolerances are the north star's (BASELINE.json): safe-action clipping / joint trajectory bit-exact in float64,
termination and collision flags exact except for contacts within 1e-5 m of a threshold, distances within 1e-4 m,
rewards within 1e-4 relative.
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle  # noqa: E402
from safemotionsrisk_b200 import abi, ball_backup_config, cabi, human_backup_config, space_backup_config, space_task_config  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CONFIGS = {"space_task": lambda **k: space_task_config(**k), "human": lambda **k: human_backup_config(**k),
           "space": lambda **k: space_backup_config(**k), "ball": lambda **k: ball_backup_config(**k),
           "space_bm": lambda **k: space_backup_config(ball_machine_mode=True, **k),
           "ball_bm": lambda **k: ball_backup_config(ball_machine_mode=True, **k)}
I = abi.INFO


def _assets(name):
    return os.path.join(os.path.dirname(GOLDEN), "..", "safemotionsrisk_b200", "assets", "networks_{}.npz".format(name))


THRESH = 1e-3   # collision threshold of the reward (rewards.py:115-155)


def make_env(name, n, **kw):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=3, auto_reset=False)
    opts.update(kw)
    cfg_kw = opts.pop("cfg", {})
    return SafeMotionsVecEnv(num_envs=n, config=CONFIGS[name](**cfg_kw), **opts)


def reported(d):
    """Distances as the device reports them: a self-collision distance above the reward's relevant distance (0.05 m in
    every shipped config) cannot change reward or termination, such pairs are pruned and the class reports the cap."""
    d = np.array(d, dtype=np.float64, copy=True)
    col = d[..., 1]
    col[(col > 0.05) & (col <= 0.102)] = 0.102
    return d


def knife_edge(d_raw_oracle, caps):
    """True where an oracle distance sits within 1e-5 m of a decision threshold (flags may legitimately differ)."""
    edge = np.zeros(d_raw_oracle.shape[0], dtype=bool)
    for col in range(3):
        for th in (THRESH, caps[col]):
            edge |= np.abs(d_raw_oracle[:, col] - th) < 1e-5
    return edge


def test_extension_is_loaded_and_counts_launches():
    env = make_env("ball", 32, fill_pools=False)
    n0 = env.launch_count()
    q = np.zeros((32, 7))
    env.set_state(q, q, q, np.zeros((32, 16)))
    env.step(np.zeros((32, 7), dtype=np.float32))
    torch.cuda.synchronize()
    # set_state + observation, then the step: joint + joint first / solve / final + contact coarse + contact plan +
    # distance plan + gjk + finish kernels
    assert env.launch_count() - n0 == 11
    env.close()


def test_safe_range_bit_exact():
    env = make_env("space", 8, fill_pools=False)
    sc = env.scene
    rng = np.random.default_rng(0)
    n = 200000
    lo_p, hi_p, V, A = (np.array(x) for x in (sc.pos_lo, sc.pos_hi, sc.vel_max, sc.acc_max))
    q = rng.uniform(lo_p, hi_p, (n, 7))
    v = rng.uniform(-1, 1, (n, 7)) * V
    a = rng.uniform(-1, 1, (n, 7)) * A
    # a quarter of the states hug a position limit, a quarter a velocity limit
    q[: n // 4] = hi_p - rng.uniform(0, 0.05, (n // 4, 7)) ** 2
    v[n // 4: n // 2] = V * (1 - rng.uniform(0, 0.05, (n // 4, 7)) ** 2)
    # an eighth sits in the band where the conservative position filter of the light path switches (0 - 1.5 rad
    # below the limit, moving towards it), an eighth mirrors that at the lower limit
    q[n // 2: 5 * n // 8] = hi_p - rng.uniform(0, 1.5, (n // 8, 7))
    v[n // 2: 5 * n // 8] = np.abs(v[n // 2: 5 * n // 8])
    q[5 * n // 8: 3 * n // 4] = lo_p + rng.uniform(0, 1.5, (n // 8, 7))
    v[5 * n // 8: 3 * n // 4] = -np.abs(v[5 * n // 8: 3 * n // 4])
    kin = np.zeros((n, 32))
    kin[:, 0:7], kin[:, 8:15], kin[:, 16:23] = q, v, a
    lo, hi, code = env.safe_range(kin)
    o_lo, o_hi, o_code = oracle.safe_range(sc, q, v, a)
    assert np.array_equal(lo.cpu().numpy(), o_lo)
    assert np.array_equal(hi.cpu().numpy(), o_hi)
    assert np.array_equal(code.cpu().numpy(), o_code)
    env.close()


@pytest.mark.parametrize("name", ["space", "ball", "space_bm", "ball_bm"])
def test_distances_match_oracle(name):
    n = 1024 if name.startswith("ball") else 256
    env = make_env(name, n, fill_pools=False)
    sc = env.scene
    rng = np.random.default_rng(1)
    q = rng.uniform(sc.pos_lo, sc.pos_hi, (n, 7))
    ob = np.zeros((n, 16))
    if name.startswith("space"):
        ob[:, 0] = rng.integers(0, 1200, n)
    else:
        # balls placed near the arm so that many distances are below the 0.6 m query
        ob[:, 2:5] = rng.uniform([-0.8, -0.8, 0.1], [0.6, 0.8, 1.3], (n, 3))
        ob[:, 8:11] = rng.uniform(-1, 1, (n, 3))
        ob[:, 13] = 1
    kin = np.zeros((n, 32))
    kin[:, 0:7] = q
    ds, dse, dm = (x.cpu().numpy() for x in env.distances(kin, ob))
    ref = reported(np.array([oracle.distances(sc, q[e], ob[e]) for e in range(n)]))
    clamp = lambda d: np.where(d < THRESH, 0.0, d)    # below 1 mm everything counts as collision (rewards.py:115)
    for dev, col in ((ds, 0), (dse, 1), (dm, 2)):
        assert np.abs(clamp(dev) - clamp(ref[:, col])).max() < 1e-4, (name, col)
    assert (ref[:, 2] < 0.6).sum() > 10 and (ref[:, 0] < 0.102).sum() > 5
    env.close()


@pytest.mark.parametrize("name", ["space", "ball", "space_bm", "ball_bm"])
def test_golden_rollout(name):
    """Committed oracle vectors: same start states and actions through the CUDA step."""
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    n = g["q"].shape[0]
    env = make_env(name, n, fill_pools=False)
    caps = (env.scene.struct.static_cap, env.scene.struct.static_cap, env.scene.struct.moving_query)
    env.set_state(g["q"], g["v"], g["a"], g["obst"])
    torch.cuda.synchronize()
    assert np.array_equal(env.kin.cpu().numpy(), g["kin0"])
    assert np.array_equal(env.obs.cpu().numpy(), g["obs0"])
    alive = np.ones(n, dtype=bool)
    latch_flips = 0
    for s in range(g["actions"].shape[0]):
        if "balls" in g:   # the oracle takes the replacement launch as an input: inject the same one on the device
            ob = env.obst.cpu().numpy()
        obs, rew, done, info = env.step(g["actions"][s])
        torch.cuda.synchronize()
        kin, obst = env.kin.cpu().numpy(), env.obst.cpu().numpy()
        if "balls" in g:
            repl = obst[:, 13] == 0        # no device pool in this test: inactive balls are replaced by hand
            if repl.any():
                obst[repl, 2:12], obst[repl, 14:16] = g["balls"][s][repl, :10], g["balls"][s][repl, 10:12]
                obst[repl, 0], obst[repl, 12], obst[repl, 13], obst[repl, 1] = 0, 0, 1, 0
                env.obst.copy_(torch.from_numpy(obst))
                env._lib.smenv_observation(env._handle, __import__("ctypes").byref(env._buf), env._stream())
                torch.cuda.synchronize()
        o_info = g["out_info"][s]
        ok = alive.copy()
        assert np.array_equal(kin[ok], g["out_kin"][s][ok]), "joint trajectory must be bit-exact"
        d_dev, d_ref = info.cpu().numpy()[:, :3], reported(o_info[:, :3])
        assert np.abs(d_dev - d_ref)[ok].max() < 1e-4
        # a collision flag may flip only where the oracle's distance of its class sits on a knife edge; coll_moving also
        # where the oracle latched a contact in this step (the sub-step contact check, counted and bounded below);
        # done only where one of the flags may flip
        flips = info.cpu().numpy()[:, 3:6] != o_info[:, 3:6]
        edge = np.stack([(np.abs(o_info[:, c] - THRESH) < 1e-5) | (np.abs(o_info[:, c] - caps[c]) < 1e-5)
                         for c in range(3)], 1)
        latched = g["out_obst"][s][:, 1] != 0
        by_latch = flips[:, 2] & ~edge[:, 2] & latched
        assert (~flips[:, :2] | edge[:, :2]).all(1)[ok].all(), s
        assert (~flips[:, 2] | edge[:, 2] | latched)[ok].all(), s
        done_flip = done.cpu().numpy() != g["out_done"][s]
        assert (~done_flip | edge.any(1) | by_latch)[ok].all(), s
        latch_flips += int((by_latch & ok).sum())
        ok &= ~flips.any(1) & ~done_flip
        assert np.allclose(rew.cpu().numpy()[ok], g["out_reward"][s][ok], rtol=1e-4, atol=1e-4)
        assert np.array_equal(env.term_reason.cpu().numpy()[ok], g["out_term"][s][ok])
        assert np.array_equal(obst[ok], g["out_obst"][s][ok])
        assert np.array_equal(env.obs.cpu().numpy()[ok], g["out_obs"][s][ok])
        alive &= ok & (g["out_done"][s] == 0)
    assert latch_flips <= 1, latch_flips   # knife-edge contacts only
    env.close()


@pytest.mark.parametrize("name", ["space", "ball"])
def test_rollout_from_device_pools_matches_oracle(name):
    """Start states sampled on the device, full 20-step episodes against the live oracle."""
    n = 128
    env = make_env(name, n, seed=11)
    start, ball = env.pools()
    q, v, a, ob = start[:n, 0:7], start[:n, 8:15], start[:n, 16:23], start[:n, 32:48]
    env.set_state(q, v, a, ob)
    orc = oracle.OracleEnvs(env.scene, n)
    orc.set_state(q, v, a, ob)
    rng = np.random.default_rng(5)
    alive = np.ones(n, dtype=bool)
    mism = 0
    for s in range(20):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        obs, rew, done, info = env.step(act)
        torch.cuda.synchronize()
        dev_ob = env.obst.cpu().numpy()
        nb = np.concatenate([dev_ob[:, 2:12], dev_ob[:, 14:16]], axis=1)   # the launch the device drew from its pool
        o_obs, o_rew, o_done, o_term, o_info = orc.step(act, nb)
        assert np.array_equal(env.kin.cpu().numpy()[alive], orc.kin[alive])
        assert np.abs(info.cpu().numpy()[:, :3] - reported(o_info[:, :3]))[alive].max() < 1e-4
        same = (done.cpu().numpy() == o_done) & (info.cpu().numpy()[:, 3:6] == o_info[:, 3:6]).all(1)
        mism += int((~same & alive).sum())
        alive &= same
        assert np.allclose(rew.cpu().numpy()[alive], o_rew[alive], rtol=1e-4, atol=1e-4)
        assert np.array_equal(obs.cpu().numpy()[alive], o_obs[alive])
        assert np.array_equal(dev_ob[alive], orc.obst[alive])
        alive &= o_done == 0
    assert mism <= 1      # knife-edge contacts only
    env.close()


@pytest.mark.parametrize("name", ["space", "ball", "space_bm"])
def test_pools_hold_valid_start_states(name):
    """Device-side rejection sampling (ctlp.py:1461-1656, :4470-4501, :1723-1931) checked with the oracle."""
    env = make_env(name, 256, seed=5)
    sc = env.scene
    start, ball = env.pools()
    assert start.shape[0] >= 1024 and np.isfinite(start).all()
    q, v, a = start[:, 0:7], start[:, 8:15], start[:, 16:23]
    assert (q >= np.array(sc.pos_lo) - 1e-12).all() and (q <= np.array(sc.pos_hi) + 1e-12).all()
    _, _, code = oracle.safe_range(sc, q[:512], v[:512], a[:512])
    assert (code == 0).all()                                   # ctlp.py:1513-1523
    assert (np.abs(v).sum(1) > 0).mean() > 0.5                 # kinematic-state sampling is used (p = 0.7)
    # q_act = q + 0.87 dt v  (reset stepSimulation, safe_motions_base.py:973-978)
    assert np.allclose(start[:, 24:31], q + 0.87 * (0.1 / 24) * v, rtol=0, atol=1e-15)
    box_min, box_max = np.array(sc.struct.start_box_min[:]), np.array(sc.struct.start_box_max[:])
    for e in range(64):
        fr = oracle.fk(sc, q[e])
        r = fr[7][:9].reshape(3, 3)
        tgt = fr[7][9:] + r @ (np.array(sc.struct.target_t[:]) +
                               np.array(sc.struct.target_R[:]).reshape(3, 3) @ np.array(sc.struct.target_offset[:]))
        assert (tgt >= box_min - 1e-5).all() and (tgt <= box_max + 1e-5).all()
        ds, dse, dm = oracle.distances(sc, q[e], start[e, 32:48])
        assert ds >= 1e-3 - 1e-5 and dse >= 1e-3 - 1e-5        # collision-free start (ctlp.py:1468-1472)
        assert dm > 0                                           # obstacle phase without contact
    if name.startswith("space"):
        idx = start[:, 32]
        assert (idx == np.round(idx)).all() and idx.min() >= 0 and idx.max() < 1200 and len(np.unique(idx)) > 200
    if ball is not None:
        assert np.isfinite(ball).all()
        speed = np.linalg.norm(ball[:, 3:6], axis=1)
        assert np.allclose(speed, 6.0, atol=1e-9)              # moving_object_speed_meter_per_second
        rel = ball[:, 0:3] - np.array([0, 0, 0.5])
        assert np.allclose(np.linalg.norm(rel, axis=1), 2.5, atol=1e-9)   # release sphere (README.md:81)
        assert (ball[:, 10] > 0).all() and (ball[:, 11] > 0).all()
    env.close()


def test_auto_reset_loads_the_philox_indexed_pool_entry():
    n = 512
    env = make_env("space", n, seed=9, auto_reset=True)
    start, _ = env.pools()
    env.reset()
    torch.cuda.synchronize()
    first = env.kin.cpu().numpy().copy()
    key0, key1 = 9, 0
    for e in range(0, n, 37):      # reset #0 of env e picks entry philox(e, 0, 0x5E7, 1) % pool
        idx = oracle.philox(e, 0, 0x5E7, 1, key0, key1)[0] % start.shape[0]
        assert np.array_equal(first[e], start[idx, :32])
    # run until every env finished at least once; afterwards every env sits on some pool entry's trajectory
    finished = np.zeros(n, dtype=bool)
    lengths = []
    for s in range(21):
        obs, rew, done, info = env.step_random()
        torch.cuda.synchronize()
        d = done.cpu().numpy() > 0
        lengths.append(info.cpu().numpy()[d, I["episode_length"]])
        ep = env.episode.cpu().numpy()
        assert (ep[d, 0] == 0).all()                       # finished envs restart at episode_length 0
        finished |= d
    assert finished.all()
    lengths = np.concatenate(lengths)
    assert lengths.max() <= 20 and lengths.min() >= 1
    stats = env.episode_statistics().cpu().numpy()
    assert stats[0] == len(lengths) and abs(stats[2] - lengths.sum()) < 1e-9
    env.close()


def test_device_random_actions_are_uniform_and_deterministic():
    a = make_env("ball", 4096, seed=21, auto_reset=True)
    b = make_env("ball", 4096, seed=21, auto_reset=True)
    a.reset(); b.reset()
    for _ in range(5):
        a.step_random(); b.step_random()
    torch.cuda.synchronize()
    assert torch.equal(a.kin, b.kin) and torch.equal(a.obs, b.obs) and torch.equal(a.reward, b.reward)
    a.close(); b.close()


def test_envs_are_independent_of_batch_composition():
    """Multi-GPU sharding rests on this: an env's trajectory does not depend on which other envs share the launch."""
    n = 64
    env = make_env("space", n, seed=4)
    start, _ = env.pools()
    q, v, a, ob = start[:n, 0:7], start[:n, 8:15], start[:n, 16:23], start[:n, 32:48]
    rng = np.random.default_rng(2)
    acts = rng.uniform(-1, 1, (5, n, 7)).astype(np.float32)
    env.set_state(q, v, a, ob)
    for s in range(5):
        env.step(acts[s])
    torch.cuda.synchronize()
    full_kin, full_rew = env.kin.cpu().numpy().copy(), env.reward.cpu().numpy().copy()
    env.close()
    half = make_env("space", n // 2, seed=4, fill_pools=False)
    sel = np.arange(n // 2) * 2 + 1
    half.set_state(q[sel], v[sel], a[sel], ob[sel])
    for s in range(5):
        half.step(acts[s][sel])
    torch.cuda.synchronize()
    assert np.array_equal(half.kin.cpu().numpy(), full_kin[sel])
    assert np.array_equal(half.reward.cpu().numpy(), full_rew[sel])
    half.close()


@pytest.mark.parametrize("name", ["space", "ball"])
def test_full_size_invariants(name):
    """BASELINE.json size (65,536 envs): size-independent properties over several auto-reset steps."""
    n = 65536
    env = make_env(name, n, seed=1, auto_reset=True)
    sc = env.scene
    env.reset()
    lo_p, hi_p, V, A = (torch.tensor(x, device=env.device) for x in (sc.pos_lo, sc.pos_hi, sc.vel_max, sc.acc_max))
    total_done = 0
    for s in range(25):
        obs, rew, done, info = env.step_random()
        q, v, a = env.kin[:, 0:7], env.kin[:, 8:15], env.kin[:, 16:23]
        assert bool(((q >= lo_p - 1e-6) & (q <= hi_p + 1e-6)).all())
        assert bool((v.abs() <= V * (1 + 1e-9)).all()) and bool((a.abs() <= A * (1 + 1e-12)).all())
        assert bool((obs.abs() <= 1).all()) and bool(torch.isfinite(rew).all())
        assert float(info[:, I["max_jerk_rel"]].max()) <= 1.0 + 1e-6
        assert bool((info[:, I["episode_length"]] <= 20).all())
        d = done > 0
        total_done += int(d.sum())
        reasons = env.term_reason[d]
        assert bool(((reasons >= 2) & (reasons <= 5)).all())
        # reward algebra holds for every env (rewards.py:481-488)
        pun = info[:, I["action_punishment"]]
        base = 0.4 * (1 - pun) + info[:, I["r_self"]] + info[:, I["r_static"]] + 3 * info[:, I["r_moving"]]
        coll = (info[:, I["coll_static"]] + info[:, I["coll_self"]] + info[:, I["coll_moving"]]) > 0
        bonus = torch.where(coll, torch.full_like(base, -15.0),
                            torch.where(info[:, I["episode_length"]] >= 20, torch.full_like(base, 15.0),
                                        torch.zeros_like(base)))
        assert float((rew - base - bonus).abs().max()) < 1e-4
    assert total_done > n        # every env finished at least once on average
    stats = env.episode_statistics().cpu().numpy()
    assert stats[0] == total_done
    env.close()


def test_squeeze_mode_reproduces_the_scalar_gym_api():
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    env = SafeMotionsVecEnv(num_envs=1, squeeze=True, seed=2, auto_reset=False, config=space_backup_config())
    obs = env.reset()
    assert isinstance(obs, np.ndarray) and obs.shape == (23,) and obs.dtype == np.float32
    assert env.observation_space.shape == (23,) and env.action_space.shape == (7,)
    done, steps = False, 0
    while not done:
        obs, rew, done, info = env.step(env.action_space.sample())
        steps += 1
        assert isinstance(rew, float) and isinstance(done, bool) and "average" in info
    assert steps <= 20 and info["termination_reason"] in (2, 4, 5) and info["episode_length"] == steps
    env.close()


def test_bad_arguments_raise():
    from safemotionsrisk_b200 import cabi
    env = make_env("space", 8, fill_pools=False)
    with pytest.raises(cabi.SmEnvError):
        env.reset()                      # pools not filled
    env.close()


def test_item_buffer_overflow_is_reported_loudly(monkeypatch):
    """The GJK work-item buffer is finite; if a step needs more items than fit, the next call must fail instead of
    returning distances computed from a truncated list."""
    monkeypatch.setenv("SMENV_ITEM_CAPACITY", "4")
    env = make_env("space", 256, auto_reset=True)
    env.reset()
    env.step_random()
    torch.cuda.synchronize()
    with pytest.raises(cabi.SmEnvError, match="overflow"):
        for _ in range(3):
            env.step_random()
            torch.cuda.synchronize()
    env.close()


def test_kernel_timing_mode_reports_every_kernel():
    env = make_env("ball", 1024, auto_reset=True)
    env.reset()
    env.kernel_timing(True)
    for _ in range(3):
        env.step_random()
    times, steps = env.kernel_times(reset=True)
    env.kernel_timing(False)
    assert steps == 3 and set(times) == set(env.KERNELS)
    assert all(t > 0.0 for t in times.values())
    env.close()


def test_counters_account_for_the_planned_pairs():
    env = make_env("space", 2048, auto_reset=True)
    env.reset()
    env.enable_counters(True)
    env.counters(reset=True)
    for _ in range(4):
        env.step_random()
    c = env.counters()
    env.enable_counters(False)
    assert c["env_steps"] == 4 * 2048
    # every planned item is run exactly once by the GJK kernel
    assert c["gjk_calls"] == c["distance_items"] + c["contact_items"]
    assert c["gjk_iters"] >= c["gjk_calls"] and c["support_dots"] > 0
    assert 0 < c["heavy_joints"] <= 7 * c["env_steps"] and c["heavy_solves"] <= 2 * c["heavy_joints"]
    env.close()


# ---------------------------------------------------------------------------------------------- networks (risk gate)
@pytest.mark.parametrize("name", ["space_bm", "ball_bm"])
def test_networks_match_the_float32_reference(name):
    """tcgen05 fp16 x fp16 -> fp32 inference of the shipped risk network / backup policy against a NumPy float32
    forward pass (oracle/mlp.py).  Tolerance: fp16 operands carry 11 significant bits and the error passes through
    three layers with unbounded selu activations: 3e-2 absolute at most (rare rows where the sigmoid is steepest,
    risk around 0.5), 1e-3 on average, on outputs that live in [0, 1] / [-1, 1].  Near the gate thresholds of the
    reference (0.06 - 0.105) the sigmoid is flat and the error stays below 4e-3 (next test)."""
    from oracle import mlp
    env = make_env(name, 1000)   # not a multiple of the 128-row tile
    env.load_networks()
    w = np.load(os.path.join(os.path.dirname(GOLDEN), "..", "safemotionsrisk_b200", "assets",
                             "networks_{}.npz".format("ball" if name.startswith("ball") else "space")))
    rng = np.random.default_rng(5)
    obs = rng.uniform(-1, 1, (1000, env.scene.obs_size)).astype(np.float32)
    act = rng.uniform(-1, 1, (1000, 7)).astype(np.float32)
    risk = env.mlp_forward(0, obs, act, n_out=1).cpu().numpy()[:, 0]
    pol = env.mlp_forward(1, obs, None, n_out=7).cpu().numpy()
    e_risk, e_pol = np.abs(risk - mlp.risk_forward(w, obs, act)), np.abs(pol - mlp.backup_forward(w, obs))
    assert e_risk.max() < 3e-2 and e_risk.mean() < 1e-3
    assert e_pol.max() < 3e-2 and e_pol.mean() < 1e-3
    env.close()


def test_exact_network_path_matches_the_float32_reference():
    """The float32 CUDA-core path of the gate (mlp_exact_kernel) against the NumPy float32 forward pass: only the
    summation order differs (1e-5 absolute on outputs in [0, 1] / [-1, 1])."""
    from oracle import mlp
    env = make_env("space_bm", 777)
    env.load_networks()
    w = np.load(_assets("space"))
    rng = np.random.default_rng(6)
    obs = rng.uniform(-1, 1, (777, env.scene.obs_size)).astype(np.float32)
    act = rng.uniform(-1, 1, (777, 7)).astype(np.float32)
    risk = env.mlp_forward_exact(0, obs, act, n_out=1).cpu().numpy()[:, 0]
    pol = env.mlp_forward_exact(1, obs, None, n_out=7).cpu().numpy()
    assert np.abs(risk - mlp.risk_forward(w, obs, act)).max() < 1e-5
    assert np.abs(pol - mlp.backup_forward(w, obs)).max() < 1e-5
    env.close()


def test_risk_gate_replaces_exactly_the_risky_actions():
    """Gate decisions are those of a float32 evaluation of the shipped networks (exact gate: the tensor-core risk of
    the rows within 0.01 of the threshold is re-rated in float32, the backup action of the risky rows is computed in
    float32): decisions may differ only where the float32 risk itself lies within 1e-5 of the threshold."""
    from oracle import mlp
    n, thr = 4096, 0.065    # README.md:223 risk_threshold of the Space task
    env = make_env("space_bm", n, auto_reset=True)
    env.load_networks()
    env.reset()
    for _ in range(5):
        env.step_random()
    w = np.load(_assets("space"))
    obs = env.obs.cpu().numpy().copy()
    act = np.random.default_rng(9).uniform(-1, 1, (n, 7)).astype(np.float32)
    env.actions.copy_(torch.from_numpy(act))
    risk, risky = env.risk_gate(thr)
    torch.cuda.synchronize()
    o_act, o_risk, o_risky = mlp.gate(w, obs, act, thr)
    risk, risky, gated = risk.cpu().numpy(), risky.cpu().numpy().astype(bool), env.actions.cpu().numpy()
    assert np.abs(risk - o_risk).max() < 3e-2                       # far from the threshold: tensor-core value
    near = np.abs(o_risk - thr) < 5e-3
    assert np.abs(risk - o_risk)[near].max() < 1e-5                 # in the band: float32 value
    clear = np.abs(o_risk - thr) > 1e-5
    assert np.array_equal(risky[clear], o_risky[clear])
    assert 0 < risky.sum() < n                                      # the gate fires on some envs, not on all
    same = risky == o_risky
    assert np.abs(gated[same] - o_act[same]).max() < 1e-5           # backup actions in float32
    assert np.array_equal(gated[~risky], act[~risky])               # safe actions pass through untouched
    # tensor cores only (smenv_set_gate_exact(0)): decisions may differ on the fp16 knife edge
    env.set_gate_exact(False)
    env.actions.copy_(torch.from_numpy(act))
    risk2, risky2 = env.risk_gate(thr)
    torch.cuda.synchronize()
    risky2 = risky2.cpu().numpy().astype(bool)
    assert np.array_equal(risky2[np.abs(o_risk - thr) > 4e-3], o_risky[np.abs(o_risk - thr) > 4e-3])
    assert np.abs(env.actions.cpu().numpy()[risky2 & o_risky] - o_act[risky2 & o_risky]).max() < 3e-2
    env.set_gate_exact(True)
    # and the gated step runs end to end
    env.step_gated(threshold=thr)
    torch.cuda.synchronize()
    env.close()


# ---------------------------------------------------------------------------------------------- reaching task
def test_reaching_task_rollout_matches_oracle():
    """Space reaching task (README.md:223): target-point observation (29 entries), TargetPointReachingReward,
    reached points replaced from the device pool.  Start poses come from the device pool; the first target of some envs
    is placed 2-8 cm from the target link point so that points are reached (radius 6.5 cm) within the rollout."""
    n, steps = 256, 12
    env = make_env("space_task", n, auto_reset=False)
    assert env.scene.obs_size == 29
    start, _ = env.pools()
    q, v, a, ob = start[:n, 0:7], start[:n, 8:15], start[:n, 16:23], start[:n, 32:48]
    assert np.all(v == 0) and np.all(a == 0)          # not collision_avoidance_mode: start at rest
    rng = np.random.default_rng(11)
    link = np.array([oracle.target_link_point(env.scene, q[e]) for e in range(n)])
    ft = link + rng.uniform(-0.3, 0.3, (n, 3))
    near = rng.random(n) < 0.4
    direction = rng.normal(size=(n, 3))
    direction /= np.linalg.norm(direction, axis=1, keepdims=True)
    ft[near] = link[near] + direction[near] * rng.uniform(0.02, 0.08, (near.sum(), 1))
    env.set_state(q, v, a, ob, first_target=ft)
    orc = oracle.OracleEnvs(env.scene, n)
    orc.set_state(q, v, a, ob, first_target=ft)
    tp = env.target.cpu().numpy()
    assert np.abs(tp[:, abi.TP_LINK_POS:abi.TP_LINK_POS + 3] - orc.tp[:, abi.TP_LINK_POS:abi.TP_LINK_POS + 3]).max() < 1e-5
    assert np.abs(env.obs.cpu().numpy() - orc.obs).max() < 1e-5
    alive = np.ones(n, dtype=bool)
    reached_total = 0
    for s in range(steps):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        obs, rew, done, info = env.step(act)
        torch.cuda.synchronize()
        tp = env.target.cpu().numpy()
        o_obs, o_rew, o_done, _, o_info = orc.step(act, None, tp[:, 0:3])   # the targets the device drew
        edge = np.abs(np.linalg.norm(orc.tp[:, 7:10] - orc.tp[:, 0:3], axis=1) - env.scene.struct.tp_radius) < 1e-4
        ok = alive & ~edge
        assert np.array_equal(env.kin.cpu().numpy()[ok], orc.kin[ok])                       # joint state bit-exact
        assert np.array_equal(tp[ok, abi.TP_REACHED_N], orc.tp[ok, abi.TP_REACHED_N])       # same points reached
        assert np.array_equal(tp[ok, abi.TP_ACTIVE], orc.tp[ok, abi.TP_ACTIVE])
        assert np.abs(tp[ok, 7:10] - orc.tp[ok, 7:10]).max() < 1e-5                         # target link point
        assert np.abs(tp[ok, 3:5] - orc.tp[ok, 3:5]).max() < 1e-5                           # distances
        i_gpu = info.cpu().numpy()
        knife = knife_edge(np.stack([o_info[:, 0], o_info[:, 1], o_info[:, 2]], 1),
                           (env.scene.struct.static_cap, env.scene.struct.static_cap, env.scene.struct.moving_query))
        ok2 = ok & ~knife
        assert np.array_equal(done.cpu().numpy()[ok2], o_done[ok2])
        # reward: (last - current) / (ts * initial distance); float32 link point -> 1e-3 absolute at distances of cm
        assert np.allclose(rew.cpu().numpy()[ok2], o_rew[ok2], rtol=1e-3, atol=2e-3)
        d_obs = np.abs(obs.cpu().numpy() - o_obs)
        d_obs[~ok2] = 0
        assert d_obs.max() < 1e-5, (s, np.unravel_index(d_obs.argmax(), d_obs.shape), d_obs.max(),
                                    obs.cpu().numpy()[d_obs.max(1).argmax()], o_obs[d_obs.max(1).argmax()],
                                    tp[d_obs.max(1).argmax()], orc.tp[d_obs.max(1).argmax()])
        reached_total = int(orc.tp[:, abi.TP_REACHED_N].sum())
        alive &= (o_done == 0) & (done.cpu().numpy() == 0)
    assert reached_total > 10          # the rollout exercised the reached / replace path
    env.close()


def test_reaching_task_full_size_invariants():
    env = make_env("space_task", 65536, auto_reset=True)
    env.reset()
    for _ in range(30):
        obs, rew, done, info = env.step_random()
    torch.cuda.synchronize()
    tp = env.target.cpu().numpy()
    assert bool((obs.abs() <= 1).all()) and bool(torch.isfinite(rew).all())
    assert np.all(tp[:, abi.TP_ACTIVE] == 1.0)                       # a reached point is replaced at once
    lo, hi = np.array(env.scene.struct.tp_box_min), np.array(env.scene.struct.tp_box_max)
    assert np.all(tp[:, 0:3] >= lo - 1e-6) and np.all(tp[:, 0:3] <= hi + 1e-6)   # sampled inside the target box
    assert np.allclose(tp[:, abi.TP_LAST_DIST], np.linalg.norm(tp[:, 0:3] - tp[:, 7:10], axis=1), atol=1e-9)
    assert tp[:, abi.TP_REACHED_N].sum() > 0
    env.close()


def test_risk_gate_on_the_reaching_task_uses_the_risk_observation():
    """In the task env the networks see the observation WITHOUT the target-point entries (observations.py:419-431)."""
    from oracle import mlp
    n, thr = 2048, 0.065
    env = make_env("space_task", n, auto_reset=True, cfg=dict(ball_machine_mode=True))
    env.load_networks()
    env.reset()
    for _ in range(3):
        env.step_random()
    w = np.load(os.path.join(os.path.dirname(GOLDEN), "..", "safemotionsrisk_b200", "assets", "networks_space.npz"))
    obs = env.obs.cpu().numpy().copy()
    risk_obs = np.concatenate([obs[:, :21], obs[:, 27:]], axis=1)
    assert risk_obs.shape[1] == 23
    act = np.random.default_rng(2).uniform(-1, 1, (n, 7)).astype(np.float32)
    env.actions.copy_(torch.from_numpy(act))
    risk, risky = env.risk_gate(thr)
    torch.cuda.synchronize()
    assert np.abs(risk.cpu().numpy() - mlp.risk_forward(w, risk_obs, act)).max() < 3e-2
    env.step_gated(threshold=thr)
    torch.cuda.synchronize()
    env.close()


def test_backup_look_ahead_labels_and_restores_the_state():
    """Risk ground truth by rolling the backup policy in a copy of the state (safe_motions_base.py:1520-1592): the
    state is restored bit for bit, the labels are deterministic, and they agree with the same look-ahead done by the
    CPU oracle with the NumPy policy (the two policies differ by fp16 rounding, so a few borderline envs may flip)."""
    from oracle import mlp
    n, steps = 512, 20
    env = make_env("space_bm", n, auto_reset=True)
    env.load_networks()
    env.reset()
    for _ in range(4):
        env.step_random()
    before = {k: v.clone() for k, v in env.snapshot().items()}
    act = np.random.default_rng(4).uniform(-1, 1, (n, 7)).astype(np.float32)
    state, a, risk = env.risk_ground_truth(act, steps)
    after = env.snapshot()
    for k in before:
        assert torch.equal(before[k], after[k]), k
    state2, a2, risk2 = env.risk_ground_truth(act, steps)
    assert torch.equal(risk, risk2) and torch.equal(state, state2)
    risk = risk.cpu().numpy()
    assert 0.02 < risk.mean() < 0.98
    # the same look-ahead on the oracle
    w = np.load(os.path.join(os.path.dirname(GOLDEN), "..", "safemotionsrisk_b200", "assets", "networks_space.npz"))
    orc = oracle.OracleEnvs(env.scene, n)
    orc.kin[:], orc.obst[:] = env.kin.cpu().numpy(), env.obst.cpu().numpy()
    orc.episode[:], orc.ep_return[:] = env.episode.cpu().numpy(), env.ep_return.cpu().numpy()
    o_risky, alive, a_o = np.zeros(n, bool), np.ones(n, bool), act
    for i in range(1 + steps):
        o_obs, _, o_done, o_term, _ = orc.step(a_o)
        o_risky |= alive & (o_done != 0) & (o_term != abi.TERMINATION_TRAJECTORY_LENGTH)
        alive &= o_done == 0
        a_o = mlp.backup_forward(w, o_obs).astype(np.float32)
    assert (o_risky != (risk > 0.5)).mean() < 0.05
    env.close()


@pytest.mark.parametrize("scene", ["ball", "space_bm", "space_task", "human"])
def test_host_step_in_ranges_equals_the_device_step(scene):
    """smenv_step_host cuts the envs into ranges on separate streams (copies overlap kernels); every range count gives
    bit-identical states, observations and rewards to the one-launch device step, including auto-resets and ball /
    target replacements (their Philox counters use the global env index) and changes of the range count between steps."""
    n = 1000   # not a multiple of the range counts: ragged last range
    ref = make_env(scene, n, auto_reset=True)
    ref.reset()
    envs = {c: make_env(scene, n, auto_reset=True) for c in (1, 3, 4, 8)}
    for e in envs.values():
        e.reset()
    mixed = make_env(scene, n, auto_reset=True)
    mixed.reset()
    ref.set_step_ranges(1)
    envs[3].set_step_ranges(3)   # its device-side steps (none here) and ...
    mixed.set_step_ranges(3)     # ... the device steps in between run as three ranges side by side
    rng = np.random.default_rng(11)
    for step in range(45):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        ref.step(torch.from_numpy(act).cuda())
        torch.cuda.synchronize()
        want = (ref.obs.cpu().numpy(), ref.reward.cpu().numpy(), ref.done.cpu().numpy())
        for c, e in list(envs.items()) + [(1 + step % 5, mixed)]:
            if e is mixed and step % 7 == 3:
                e.step(torch.from_numpy(act).cuda())   # the device step in between: the list layout goes back to one range
                got = (e.obs.cpu().numpy(), e.reward.cpu().numpy(), e.done.cpu().numpy())
            else:
                got = e.step_host(act, chunks=c)
            for w, g in zip(want, got):
                assert np.array_equal(w, g), (scene, c, step)
            assert torch.equal(e.kin, ref.kin) and torch.equal(e.obst, ref.obst) and torch.equal(e.episode, ref.episode)
            if scene == "human":   # the nested env (its policy's Philox noise included) is independent of the ranges too
                assert torch.equal(e.hkin, ref.hkin) and torch.equal(e.hactions, ref.hactions)
    assert ref.stats[0].item() > 0   # episodes ended and were reset on the way
    for e in list(envs.values()) + [mixed, ref]:
        e.close()


@pytest.mark.parametrize("scene,threshold", [("space_bm", 0.065), ("human", 0.06)])
def test_gated_host_step_equals_the_gated_device_step(scene, threshold):
    """The risk gate inside the host-buffer step (CUDA graph replay, ranges on separate streams) decides and acts exactly
    like the gate inside the device step: same risky flags, executed actions, states and outputs."""
    n = 1000
    envs = [make_env(scene, n, auto_reset=True) for _ in range(3)]
    for e in envs:
        e.load_networks()
        e.set_risk_gate(threshold)
        e.reset()
    ref, host2, host3 = envs
    ref.set_step_ranges(1)
    rng = np.random.default_rng(17)
    risky_total = 0
    for step in range(25):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        ref.step(torch.from_numpy(act).cuda())
        torch.cuda.synchronize()
        want = (ref.obs.cpu().numpy(), ref.reward.cpu().numpy(), ref.done.cpu().numpy())
        for e, c in ((host2, 2), (host3, 3)):
            got = e.step_host(act, chunks=c)
            for w, g in zip(want, got):
                assert np.array_equal(w, g), (scene, c, step)
            assert torch.equal(e.kin, ref.kin) and torch.equal(e.info[:, 16], ref.info[:, 16]), (scene, c, step)
            if scene == "human":
                assert torch.equal(e.hkin, ref.hkin)
        risky_total += int(ref.info[:, 16].sum())
    assert 0 < risky_total < 25 * n
    for e in envs:
        e.close()


# ---------------------------------------------------------------------------------------------- round 2: gate wiring

def test_gate_inside_step_keeps_the_proposed_action_for_the_reward():
    """actions.py:303-340 / safe_motions_base.py:1066: the gate replaces the executed action only; the action
    punishment of the reward still rates what the policy proposed.  Env A steps with the gate switched on inside the
    step; env B gets the same proposal gated by hand (risk_gate in place) and steps ungated: the joint trajectories are
    identical, the rewards differ exactly by the punishment of the proposal vs the punishment of the backup action."""
    n, thr = 2048, 0.065
    cfg = dict(risk_config_dir="risk_networks/state_action/space", risk_threshold=thr)
    a_env = make_env("space_task", n, auto_reset=False, cfg=dict(ball_machine_mode=True, **cfg))
    b_env = make_env("space_task", n, auto_reset=False, cfg=dict(ball_machine_mode=True))
    b_env.load_networks()
    assert a_env._gate_threshold == thr and b_env._gate_threshold is None
    a_env.reset()
    b_env.restore(a_env.snapshot())
    rng = np.random.default_rng(2)
    prop = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
    prop[: n // 4] *= 0.5          # some proposals without punishment
    a_env.step(prop)
    b_env.actions.copy_(torch.from_numpy(prop))
    _, risky = b_env.risk_gate(thr)
    gated = b_env.actions.clone()
    b_env._step_device(gated)
    torch.cuda.synchronize()
    risky = risky.cpu().numpy().astype(bool)
    assert 0 < risky.sum() < n
    assert np.array_equal(a_env.kin.cpu().numpy(), b_env.kin.cpu().numpy())          # same executed actions
    assert np.array_equal(a_env.actions.cpu().numpy(), prop)                          # the proposal is kept
    ia, ib = a_env.info.cpu().numpy(), b_env.info.cpu().numpy()
    assert np.array_equal(ia[:, I["risky_action"]].astype(bool), risky)
    assert np.array_equal(ib[:, I["risky_action"]], np.zeros(n, dtype=np.float32))
    pun = lambda u: np.clip((np.abs(u).max(1) - 0.95) / 0.05, 0, 1) ** 2
    assert np.allclose(ia[:, I["action_punishment"]], pun(prop), atol=1e-5)
    assert np.allclose(ib[:, I["action_punishment"]], pun(gated.cpu().numpy()), atol=1e-5)
    dr = a_env.reward.cpu().numpy() - b_env.reward.cpu().numpy()
    assert np.allclose(dr, -0.4 * (pun(prop) - pun(gated.cpu().numpy())), atol=1e-4)
    first = ia[:, I["first_risky_step"]]
    assert np.array_equal(first >= 0, risky) and (first[risky] == 0).all()
    # host-buffer step with the gate: same decisions through the chunked graph path
    a_env.restore(b_env.snapshot())
    b_snap = b_env.snapshot()
    prop2 = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
    a_env.step_host(prop2, chunks=2)
    b_env.restore(b_snap)
    b_env.set_risk_gate(thr)
    b_env.step(prop2)
    torch.cuda.synchronize()
    assert np.array_equal(a_env.kin.cpu().numpy(), b_env.kin.cpu().numpy())
    assert np.array_equal(a_env.info.cpu().numpy()[:, I["risky_action"]], b_env.info.cpu().numpy()[:, I["risky_action"]])
    a_env.close()
    b_env.close()


def test_set_seed_reproduces_an_env_built_with_that_seed():
    a = make_env("ball", 512, seed=5, auto_reset=True)
    b = make_env("ball", 512, seed=9, auto_reset=True)
    b.reset()
    for _ in range(3):
        b.step_random()
    b.set_seed(5)
    a.reset()
    b.reset()
    for _ in range(25):       # past the first auto-resets and ball replacements
        a.step_random()
        b.step_random()
    torch.cuda.synchronize()
    assert np.array_equal(a.kin.cpu().numpy(), b.kin.cpu().numpy())
    assert np.array_equal(a.obst.cpu().numpy(), b.obst.cpu().numpy())
    a.close()
    b.close()


def test_two_envs_of_different_scenes_alternate_in_one_process():
    """The scene constants live in one per-device constant-memory block and the opt-in shared-memory limit is per
    function: a big scene created first must keep working after a small one is created, and alternating steps of two
    envs must give what each gives alone (ADVICE round 1)."""
    big = make_env("space_bm", 256, seed=1, auto_reset=True)
    small = make_env("ball", 256, seed=1, auto_reset=True)
    big_alone = make_env("space_bm", 256, seed=1, auto_reset=True)
    small_alone = make_env("ball", 256, seed=1, auto_reset=True)
    for e in (big, small, big_alone, small_alone):
        e.reset()
    side = torch.cuda.Stream()
    for i in range(6):
        big.step_random()
        with torch.cuda.stream(side):
            small.step_random()
    for i in range(6):
        big_alone.step_random()
    for i in range(6):
        small_alone.step_random()
    torch.cuda.synchronize()
    assert np.array_equal(big.kin.cpu().numpy(), big_alone.kin.cpu().numpy())
    assert np.array_equal(small.kin.cpu().numpy(), small_alone.kin.cpu().numpy())
    assert np.array_equal(big.reward.cpu().numpy(), big_alone.reward.cpu().numpy())
    for e in (big, small, big_alone, small_alone):
        e.close()


def test_reset_at_does_not_reset_an_auto_reset_env_twice():
    env = make_env("ball", 64, auto_reset=True)
    env.reset()
    done = None
    for _ in range(20):
        obs, rew, done, _ = env.vector_step(np.zeros((64, 7), dtype=np.float32))
    done = np.array(done)
    assert done.sum() > 32                             # most 20-step episodes end together (some ended early: ball hits)
    resets = env.episode.cpu().numpy()[:, 1].copy()
    first_obs = env.obs.cpu().numpy().copy()
    for i in np.where(done)[0]:
        assert np.array_equal(env.reset_at(int(i)), first_obs[i])
    assert np.array_equal(env.episode.cpu().numpy()[:, 1], resets)   # no second reset, no second episode counted
    env.step(np.zeros((64, 7), dtype=np.float32))
    i = int(np.where(env.done.cpu().numpy() == 0)[0][0])
    env.reset_at(i)                                    # not done in the last step: a real reset
    assert env.episode.cpu().numpy()[i, 1] == resets[i] + 1
    env.close()


def test_risk_ground_truth_window_ignores_the_end_of_the_real_episode():
    """The look-ahead runs on its own episode clock (safe_motions_base.py:1818-1822): an env three steps before its
    episode end is labelled like the same state at the start of an episode (ADVICE round 1)."""
    n = 1024
    env = make_env("space_bm", n, auto_reset=False)
    env.load_networks()
    env.reset()
    for _ in range(4):
        env.step_random()
    act = np.random.default_rng(4).uniform(-1, 1, (n, 7)).astype(np.float32)
    _, _, risk_early = env.risk_ground_truth(act, backup_steps=20)
    env.episode[:, 0] = 17                              # same state, three steps before the end of the real episode
    _, _, risk_late = env.risk_ground_truth(act, backup_steps=20)
    assert int(env.episode[0, 0].item()) == 17          # the state is restored
    assert torch.equal(risk_early, risk_late)
    assert 0 < float(risk_early.mean().item()) < 1
    env.close()


def test_initial_backup_trajectory_check_filters_start_states():
    """risk_check_initial_backup_trajectory (observations.py:155-185): after reset() no env starts from a state in
    which the backup policy itself collides within its 20 steps."""
    n = 2048
    env = make_env("space_bm", n, auto_reset=True,
                   cfg=dict(risk_config_dir="risk_networks/state_action/space", risk_threshold=0.065,
                            risk_check_initial_backup_trajectory=True))
    plain = make_env("space_bm", n, auto_reset=True)
    plain.load_networks()
    plain.reset()
    unsafe_plain = float(plain.initial_backup_trajectory_unsafe().float().mean().item())
    env.reset()
    unsafe = float(env.initial_backup_trajectory_unsafe().float().mean().item())
    assert unsafe == 0.0 and unsafe_plain >= 0.0
    env.close()
    plain.close()


@pytest.mark.parametrize("name", ["space_bm", "ball_bm"])
def test_behavioural_pin_shipped_backup_policy_avoids_collisions(name):
    """The only reference-held artefacts that can pin the restated env are the shipped network weights (SURVEY 8c item
    5): the backup policy, trained in the real PyBullet env, must keep most 20-step episodes collision free in THIS env,
    and far more of them than random actions do."""
    n = 16384
    rates = {}
    for mode in ("policy", "random"):
        env = make_env(name, n, seed=11, auto_reset=True)
        env.load_networks()
        env.reset()
        env.stats.zero_()
        for _ in range(60):
            if mode == "policy":
                env.step(env.backup_policy_actions())
            else:
                env.step_random()
        s = env.episode_statistics().cpu().numpy()
        rates[mode] = float((s[3 + 3] + s[3 + 4] + s[3 + 5]) / max(s[0], 1))
        env.close()
    print(name, "collision-termination rate: backup policy {:.4f}, random actions {:.4f}".format(
        rates["policy"], rates["random"]))
    assert rates["policy"] < 0.5 * rates["random"]
    assert rates["policy"] < 0.25


def test_episode_aggregates_match_host_accumulation():
    """SmBuffers.epinfo: sum / max / min of the step scalars over each finished episode, accumulated on the device,
    against the same aggregation done on the host from the per-step outputs (what train.py:59-117 does with the
    reference's per-step info dicts)."""
    n = 512
    env = make_env("ball", n, auto_reset=True)
    env.reset()
    keys = [("coll_self", 0), ("coll_static", 1), ("coll_moving", 2), ("action_punishment", 3), ("r_self", 4),
            ("r_static", 5), ("r_moving", 6)]
    s = np.zeros((n, 8)); mx = np.full((n, 8), -np.inf); mn = np.full((n, 8), np.inf)
    checked = 0
    rng = np.random.default_rng(0)
    for _ in range(45):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        _, rew, done, info = env.step(act)
        info, rew, done = info.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy().astype(bool)
        vals = np.stack([info[:, I[k]] for k, _ in keys] + [rew], 1)
        s += vals; mx = np.maximum(mx, vals); mn = np.minimum(mn, vals)
        if done.any():
            rec = env.epinfo.cpu().numpy()[done]
            for c in range(8):
                assert np.allclose(rec[:, c], s[done, c], rtol=1e-5, atol=1e-4)
                assert np.allclose(rec[:, 16 + c], mx[done, c], atol=1e-6) and np.allclose(rec[:, 32 + c], mn[done, c], atol=1e-6)
            assert np.array_equal(rec[:, abi.EPC["length"]], info[done, I["episode_length"]])
            assert np.allclose(rec[:, abi.EPC["ret"]], info[done, I["episode_return"]], rtol=1e-6)
            assert np.array_equal(rec[:, abi.EPC["reason"]], env.term_reason.cpu().numpy()[done])
            checked += int(done.sum())
            s[done] = 0; mx[done] = -np.inf; mn[done] = np.inf
    assert checked >= 2 * n
    d = [x for x in env.infos(only_done=True) if x]
    for x in d[:3]:
        assert x["episode_length"] <= 20 and "collision_rate_moving_obstacles_average" in x["episode"]
        assert x["trajectory_successful"] == 1.0 and "moving_object_hit_robot_total" in x
    env.close()


@pytest.mark.parametrize("variant", ["no_table", "planet_obs_1"])
def test_scene_variants_match_oracle(variant):
    """Config switches outside the two shipped scenes: obstacle_scene = 0 (no table, ctlp.py:2426-2434) and one
    observation entry per planet (observations.py:258-292).  (A single planet / independent planets raise in scene.py.)"""
    cfg = {"no_table": dict(obstacle_scene=0), "planet_obs_1": dict(obs_planet_size_per_planet=1)}[variant]
    n = 96
    env = make_env("space", n, seed=5, cfg=cfg)
    sc = env.scene.struct
    if variant == "no_table":
        assert sc.has_table == 0
    if variant == "planet_obs_1":
        assert sc.obs_planet_size == 1 and sc.obs_size == 22
    start, _ = env.pools()
    q, v, a, ob = start[:n, 0:7], start[:n, 8:15], start[:n, 16:23], start[:n, 32:48]
    env.set_state(q, v, a, ob)
    orc = oracle.OracleEnvs(env.scene, n)
    orc.set_state(q, v, a, ob)
    assert np.array_equal(env.obs.cpu().numpy(), orc.obs)
    rng = np.random.default_rng(9)
    alive = np.ones(n, dtype=bool)
    mism = 0
    for s in range(8):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        obs, rew, done, info = env.step(act)
        torch.cuda.synchronize()
        o_obs, o_rew, o_done, o_term, o_info = orc.step(act)
        assert np.array_equal(env.kin.cpu().numpy()[alive], orc.kin[alive])
        assert np.abs(info.cpu().numpy()[:, :3] - reported(o_info[:, :3]))[alive].max() < 1e-4
        same = (done.cpu().numpy() == o_done) & (info.cpu().numpy()[:, 3:6] == o_info[:, 3:6]).all(1)
        mism += int((~same & alive).sum())
        alive &= same
        assert np.allclose(rew.cpu().numpy()[alive], o_rew[alive], rtol=1e-4, atol=1e-4)
        assert np.array_equal(obs.cpu().numpy()[alive], o_obs[alive])
        alive &= o_done == 0
    assert mism <= 1
    env.close()


@pytest.mark.parametrize("hidden", [[512, 256, 128], [256, 128], [128, 64], [64, 64], [128, 64, 32], [32, 16], [192, 48]])
def test_tensor_core_mlp_layer_widths(hidden):
    """mlp_kernel for every supported layer shape (a network trained by risk_train.py need not have the shipped 512 /
    256 / 128 widths) against a NumPy float32 forward pass; unsupported widths are refused, not mis-computed."""
    from oracle import mlp
    env = make_env("space_bm", 1024, fill_pools=False)
    rng = np.random.default_rng(len(hidden) * 1000 + hidden[0])
    x = rng.uniform(-1, 1, (1024, 30)).astype(np.float32)
    dims = [30] + hidden + [1]
    layers = [(rng.normal(0, 1.0 / np.sqrt(dims[i]), (dims[i], dims[i + 1])).astype(np.float32),
               rng.normal(0, 0.1, dims[i + 1]).astype(np.float32)) for i in range(len(dims) - 1)]
    flat = np.concatenate([np.concatenate([k.ravel(), b.ravel()]) for k, b in layers])
    d = np.array(dims, dtype=np.int32)
    cabi.check(env._lib.smenv_mlp_load(env._handle, 0, len(hidden), d.ctypes.data, 0, 0, flat.ctypes.data), "smenv_mlp_load")
    h = x
    for k, b in layers[:-1]:
        h = mlp.selu(h @ k + b)
    want = (1 / (1 + np.exp(-(h @ layers[-1][0] + layers[-1][1]))))[:, 0]
    got = env.mlp_forward(0, x[:, :23], x[:, 23:])[:, 0].cpu().numpy()
    exact = env.mlp_forward_exact(0, x[:, :23], x[:, 23:])[:, 0].cpu().numpy()
    assert np.abs(got - want).max() < 2e-3 and np.abs(exact - want).max() < 2e-6
    bad = np.array([30, 96, 64, 1], dtype=np.int32)
    assert env._lib.smenv_mlp_load(env._handle, 0, 2, bad.ctypes.data, 0, 0, flat.ctypes.data) != 0
    env.close()


@pytest.mark.parametrize("scene", ["space_bm", "human"])
def test_restored_state_replays_bit_for_bit(scene):
    """The distance queries of a step start from the previous step's closest pairs (warm start, csrc/smenv_gjk.cuh), which
    only changes float rounding -- and snapshot / restore forget that history, so a replay from a restored state gives the
    same bits as the first run (parity with the oracle under warm starts is what the rollout tests above check)."""
    n, steps = 2048, 6
    env = make_env(scene, n, auto_reset=True)
    env.reset()
    for _ in range(5):
        env.step_random()
    snap = {k: v.clone() for k, v in env.snapshot().items()}
    acts = torch.from_numpy(np.random.default_rng(9).uniform(-1, 1, (steps, n, 7)).astype(np.float32)).cuda()
    if scene == "human":   # the human's policy noise depends on the library's step counter: drive it from outside
        env.set_human_actions_external(True)
        hact = torch.from_numpy(np.random.default_rng(10).uniform(-1, 1, (steps, n, 8)).astype(np.float32)).cuda()

    def run():
        out = []
        for i in range(steps):
            if scene == "human":
                env.hactions.copy_(hact[i])
            env.step(acts[i])
            out.append((env.obs.clone(), env.reward.clone(), env.done.clone(), env.info.clone()))
        return out

    first = run()
    env.restore(snap)
    second = run()
    for a, b in zip(first, second):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    env.close()
