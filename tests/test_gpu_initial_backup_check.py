"""risk_check_initial_backup_trajectory as a check of the start pool (smenv_set_initial_backup_check).

Every start-pool entry is checked once when the pool is filled, the pool is partitioned stably by the verdict and every
reset draws from the passing entries.  The kept set is checked against initial_backup_trajectory_unsafe entry by entry,
the episodes the step starts against the same function, and the step itself against an env without the check.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from safemotionsrisk_b200 import abi, human_backup_config, space_backup_config  # noqa: E402

K = 20
CONFIGS = {"space_bm": lambda **k: space_backup_config(ball_machine_mode=True, **k),
           "human": lambda **k: human_backup_config(**k)}
NETWORKS = {"space_bm": "space", "human": "human"}
THRESHOLD = {"space": 0.065, "human": 0.06}


def make_env(scene, n, check, seed=3, **kw):
    """The env as a user gets it with the network gate on, with or without risk_check_initial_backup_trajectory."""
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=seed, auto_reset=True)
    opts.update(kw)
    net = NETWORKS[scene]
    cfg = dict(risk_config_dir="risk_networks/state_action/" + net, risk_threshold=THRESHOLD[net],
               risk_check_initial_backup_trajectory=check, risk_state_initial_backup_trajectory_steps=K)
    return SafeMotionsVecEnv(num_envs=n, config=CONFIGS[scene](**cfg), **opts)


def label_entries(start, scene="space_bm"):
    """initial_backup_trajectory_unsafe of every pool entry, each in an env of its own (one env per entry)."""
    P = start.shape[0]
    lab = make_env(scene, P, check=False, auto_reset=False)
    lab.set_state(start[:, 0:7], start[:, 8:15], start[:, 16:23], start[:, 32:48])
    lab.kin.copy_(torch.from_numpy(start[:, 0:32]).to(lab.device))   # the entry's kin record exactly, as a reset copies it
    unsafe = lab.initial_backup_trajectory_unsafe(K).cpu().numpy()
    lab.close()
    return unsafe


def permutation(before, after):
    """Index of every row of `after` in `before` (rows are unique)."""
    where = {r.tobytes(): i for i, r in enumerate(before)}
    return np.array([where[r.tobytes()] for r in after])


@pytest.mark.parametrize("n", [2048, 256])
def test_kept_set_is_exactly_the_passing_entries_in_order(n):
    """space_bm is deterministic: the checked pool holds exactly the entries initial_backup_trajectory_unsafe passes,
    first and in their original order, then the failing ones.  At n = 256 the pool has 1024 entries: four batches."""
    plain = make_env("space_bm", n, check=False)
    start0, _ = plain.pools()
    plain.close()
    P = start0.shape[0]
    assert P == max(n, 1024)
    unsafe = label_entries(start0)
    keep = ~unsafe
    env = make_env("space_bm", n, check=True)
    start1, _ = env.pools()
    checked, passed = env.initial_backup_check_counts()
    assert checked == P and passed == int(keep.sum())
    assert 0 < passed < P
    assert np.array_equal(start1[:passed], start0[keep])
    assert np.array_equal(start1[passed:], start0[unsafe])
    env.close()


@pytest.mark.parametrize("mode", ["step", "step_random", "host1", "host2"])
def test_every_started_episode_passes(mode):
    """After reset() and after every auto reset of step / step_random / step_host the new episode starts from a state
    whose backup trajectory is free of collisions."""
    n = 512
    env = make_env("space_bm", n, check=True)
    env.reset()
    assert not bool(env.initial_backup_trajectory_unsafe(K).any())
    rng = np.random.default_rng(7)
    started = 0
    for _ in range(40):
        resets = env.episode[:, 1].clone()
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        if mode == "step":
            env.step(act)
        elif mode == "step_random":
            env.step_random()
        else:
            env.step_host(act, chunks=int(mode[-1]))
        done = env.done.bool()
        assert bool((env.episode[done, 0] == 0).all())
        assert torch.equal(env.episode[done, 1], resets[done] + 1)
        assert torch.equal(env.episode[~done, 1], resets[~done])
        if bool(done.any()):
            assert not bool((env.initial_backup_trajectory_unsafe(K) & done).any())
            started += int(done.sum())
    assert started > n
    env.close()


@pytest.mark.parametrize("ranges,chunks", [(1, 1), (2, 3)])
def test_step_host_resets_finished_envs_like_the_device_step(ranges, chunks):
    """Under the flag the host-buffer step auto-resets like the device step, bit for bit."""
    n = 1000
    dev = make_env("space_bm", n, check=True)
    host = make_env("space_bm", n, check=True)
    dev.set_step_ranges(ranges)
    dev.reset()
    host.reset()
    rng = np.random.default_rng(11)
    finished = 0
    for step in range(30):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        dev.step(act)
        obs, rew, done = host.step_host(act, chunks=chunks)
        torch.cuda.synchronize()
        for k in ("kin", "obst", "episode", "obs", "done", "reward", "term_reason", "info"):
            assert torch.equal(getattr(dev, k), getattr(host, k)), (step, k)
        assert np.array_equal(obs, dev.obs.cpu().numpy()) and np.array_equal(done, dev.done.cpu().numpy())
        finished += int(done.sum())
    assert finished > 0
    dev.close()
    host.close()


@pytest.mark.parametrize("gate", [True, False])
def test_no_extra_launches_per_step(gate):
    """The check costs nothing per step: the step issues as many kernels with the flag as without it."""
    deltas = {}
    for check in (True, False):
        env = make_env("space_bm", 512, check=check)
        if not gate:
            env.set_risk_gate(None)
        env.reset()
        for _ in range(3):
            env.step_random()
        c0 = env.launch_count()
        for _ in range(25):   # 20-step episodes: auto resets inside the window
            env.step_random()
        deltas[check] = env.launch_count() - c0
        env.close()
    assert deltas[True] == deltas[False]


def test_human_pairs_survive_compaction_and_resets_stay_valid():
    """Human scene: every kept robot entry still sits next to its own human start state and stored braking trajectory;
    episodes started by 30+ auto-reset steps are finite and inside the joint limits."""
    n = 1024
    plain = make_env("human", n, check=False)
    start0, _ = plain.pools()
    hstart0, _ = plain.human_pools()
    env = make_env("human", n, check=True)
    start1, _ = env.pools()
    hstart1, _ = env.human_pools()
    checked, passed = env.initial_backup_check_counts()
    assert checked == start0.shape[0] and 0 < passed <= checked
    perm = permutation(start0, start1)
    assert np.array_equal(np.sort(perm), np.arange(len(perm)))
    assert np.array_equal(hstart1, hstart0[perm])
    assert np.all(np.diff(perm[:passed]) > 0) and np.all(np.diff(perm[passed:]) > 0)   # stable
    # the stored braking trajectory moved with its entry: a reset copies it, set_human_state computes it from the state
    env.reset()
    entry = permutation(start1[:, 0:32], env.kin.cpu().numpy())
    assert np.all(entry < passed)
    h = hstart1[entry]
    plain.set_state(start1[entry, 0:7], start1[entry, 8:15], start1[entry, 16:23], start1[entry, 32:48])
    plain.set_human_state(h[:, 0:8], h[:, 8:16], h[:, 16:24], np.zeros((n, 3)), np.zeros(n, dtype=np.int32))
    torch.cuda.synchronize()
    assert torch.equal(env.hkin[:, 0:24], plain.hkin[:, 0:24])
    cnt = env.hstate[:, abi.HS_BRAKE_COUNT]
    assert torch.equal(cnt, plain.hstate[:, abi.HS_BRAKE_COUNT])
    steps = torch.arange(abi.SM_HBRAKE_STEPS, device=env.device).repeat_interleave(abi.SM_HUMAN_JOINTS)
    valid = steps[None, :] < cnt[:, None]
    assert torch.equal(env.hbrake[valid], plain.hbrake[valid])
    plain.close()
    sc = env.scene
    lo, hi = (torch.tensor(x, device=env.device) for x in (sc.pos_lo, sc.pos_hi))
    started = 0
    for _ in range(35):
        env.step_random()
        done = env.done.bool()
        started += int(done.sum())
        q = env.kin[done, 0:7]
        assert bool(torch.isfinite(env.kin).all()) and bool(torch.isfinite(env.hkin).all())
        assert bool(((q >= lo - 1e-6) & (q <= hi + 1e-6)).all())
    assert started > 0
    env.close()


def test_refill_and_off_switch():
    """Same seed, same checked pool; set_seed(s) gives the pool of a fresh env with seed s; 0 draws from the whole pool
    again; without a backup policy the check cannot be switched on."""
    from safemotionsrisk_b200 import cabi
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    a = make_env("space_bm", 256, check=True, seed=5)
    b = make_env("space_bm", 256, check=True, seed=5)
    assert np.array_equal(a.pools()[0], b.pools()[0])
    assert a.initial_backup_check_counts() == b.initial_backup_check_counts()
    b.close()
    a.set_seed(9)
    c = make_env("space_bm", 256, check=True, seed=9)
    assert np.array_equal(a.pools()[0], c.pools()[0])
    assert a.initial_backup_check_counts() == c.initial_backup_check_counts()
    c.close()
    P = a.pools()[0].shape[0]
    a.set_initial_backup_check(0)
    assert a.initial_backup_check_counts() == (0, P)
    a.set_seed(5)   # a refill restores the unchecked pool exactly
    d = make_env("space_bm", 256, check=False, seed=5)
    assert np.array_equal(a.pools()[0], d.pools()[0])
    d.close()
    a.close()
    bare = SafeMotionsVecEnv(num_envs=64, config=space_backup_config(ball_machine_mode=True), seed=1)
    with pytest.raises(cabi.SmEnvError):
        bare.set_initial_backup_check(K)
    bare.close()


def test_check_leaves_the_real_env_alone():
    """The pool check touches none of the real env's records, statistics or step counter."""
    n = 512
    env = make_env("space_bm", n, check=False, auto_reset=False)
    twin = make_env("space_bm", n, check=False, auto_reset=False)
    for e in (env, twin):
        e.reset()
        for _ in range(5):
            e.step_random()
    before = env.snapshot()
    env.set_initial_backup_check(K)
    assert env.initial_backup_check_counts()[0] > 0
    torch.cuda.synchronize()
    for k, v in before.items():
        assert torch.equal(getattr(env, k), v), k
    env.step_random()
    twin.step_random()
    torch.cuda.synchronize()
    for k in ("kin", "obst", "episode", "obs", "reward", "done", "term_reason", "info", "epinfo"):
        assert torch.equal(getattr(env, k), getattr(twin, k)), k
    # the statistics are float64 sums of per-block atomics, whose order varies from run to run
    assert torch.allclose(env.stats, twin.stats, rtol=1e-12, atol=0), "stats"
    env.close()
    twin.close()
