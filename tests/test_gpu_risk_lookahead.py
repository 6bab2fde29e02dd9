"""The backup-trajectory look-ahead as the risk check inside the step (risk_state_config 4, smenv_set_risk_lookahead).

The look-ahead restates risk_ground_truth on shadow copies of the state inside the step, so its decisions are checked
against risk_ground_truth bit for bit, and the real step that follows against a twin env that executes what the shield
decided.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from safemotionsrisk_b200 import abi, ball_backup_config, human_backup_config, space_backup_config, space_task_config  # noqa: E402

I = abi.INFO
K = 20
CONFIGS = {"space_bm": lambda **k: space_backup_config(ball_machine_mode=True, **k),
           "ball_bm": lambda **k: ball_backup_config(ball_machine_mode=True, **k),
           "space_task_bm": lambda **k: space_task_config(ball_machine_mode=True, **k),
           "human": lambda **k: human_backup_config(**k)}
NETWORKS = {"space_bm": "space", "ball_bm": "ball", "space_task_bm": "space", "human": "human"}
THRESHOLD = {"space": 0.065, "ball": 0.065, "human": 0.06}


def make_env(scene, n, shield, **kw):
    """shield: the env as a user gets it from risk_state_config=4; else an env without any gate."""
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=3, auto_reset=True)
    opts.update(kw)
    cfg = {}
    if shield:
        net = NETWORKS[scene]
        cfg = dict(risk_config_dir="risk_networks/state_action/" + net, risk_threshold=THRESHOLD[net],
                   risk_state_config=4, risk_state_backup_trajectory_steps=K)
    return SafeMotionsVecEnv(num_envs=n, config=CONFIGS[scene](**cfg), **opts)


def collided(env):
    return env.done.bool() & (env.term_reason != env.TERMINATION_TRAJECTORY_LENGTH)


def risky_of(env):
    return env.info[:, I["risky_action"]] > 0.5


@pytest.mark.parametrize("scene", ["space_bm", "ball_bm", "space_task_bm"])
def test_decisions_equal_risk_ground_truth(scene):
    """Every decision equals risk_ground_truth's label, and the real step equals a twin's step with the action the label
    asks for (the float32 backup action where risky).  No stochastic element enters the look-ahead of these scenes."""
    n = 1000   # ragged against the ranges of the step
    env = make_env(scene, n, shield=True)
    twin = make_env(scene, n, shield=False)
    twin.load_networks()
    env.reset()
    rng = np.random.default_rng(5)
    env.set_risk_gate(None)
    for _ in range(3):
        env.step(rng.uniform(-1, 1, (n, 7)).astype(np.float32))
    env.set_risk_gate(THRESHOLD[NETWORKS[scene]])
    twin.restore(env.snapshot())
    risky_total = 0
    for step in range(5):
        act = torch.from_numpy(rng.uniform(-1, 1, (n, 7)).astype(np.float32)).cuda()
        _, _, gt = twin.risk_ground_truth(act, K)
        want = gt > 0.5
        backup = twin.mlp_forward_exact(1, twin.risk_observation(), n_out=7)
        twin.step(torch.where(want[:, None], backup, act))
        env.step(act)
        torch.cuda.synchronize()
        risky = risky_of(env)
        assert torch.equal(risky, want), (scene, step, int((risky != want).sum()))
        for k in ("kin", "obst", "obs", "done"):
            assert torch.equal(getattr(env, k), getattr(twin, k)), (scene, step, k)
        assert torch.equal(env.episode[:, :3], twin.episode[:, :3]), (scene, step)   # [:, 3]: first risky step
        keep = ~risky
        assert torch.equal(env.reward[keep], twin.reward[keep]), (scene, step)
        assert torch.equal(env.info[:, I["risk"]], want.float())
        risky_total += int(risky.sum())
    assert 0 < risky_total < 5 * n
    env.close()
    twin.close()


@pytest.mark.parametrize("scene", ["space_bm", "human"])
def test_kept_actions_never_collide(scene):
    """Sub-step 0 of the look-ahead is the real step: an action the shield keeps cannot end the step in a collision."""
    n = 16384
    env = make_env(scene, n, shield=True)
    rand = make_env(scene, n, shield=False)
    env.reset()
    rand.reset()
    episodes = {"shield": n, "random": n}
    hits = {"shield": 0, "random": 0}
    kept = 0
    for step in range(10):
        env.step_random()     # the same device-drawn proposals as `rand` (same seed, same step counter)
        rand.step_random()
        torch.cuda.synchronize()
        risky = risky_of(env)
        assert not bool((collided(env) & ~risky).any()), (scene, step)
        kept += int((~risky).sum())
        for name, e in (("shield", env), ("random", rand)):
            hits[name] += int(collided(e).sum())
            episodes[name] += int(e.done.sum())
    frac = {k: hits[k] / episodes[k] for k in hits}
    print("{}: episodes ending in a collision: shield {:.4f}, random actions {:.4f}; {} of {} actions kept".format(
        scene, frac["shield"], frac["random"], kept, 10 * n))
    assert frac["shield"] < frac["random"]
    env.close()
    rand.close()


def test_human_scene_against_an_ungated_twin():
    """The nested env of the human does not see the robot: its state and actions equal an ungated twin's in every env at
    every step; the robot equals the twin's in the envs that were never risky."""
    n = 2048
    env = make_env("human", n, shield=True, auto_reset=False)
    twin = make_env("human", n, shield=False, auto_reset=False)
    env.reset()
    twin.reset()
    rng = np.random.default_rng(9)
    ever = torch.zeros(n, dtype=torch.bool, device=env.device)
    for step in range(8):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        env.step(act)
        twin.step(act)
        torch.cuda.synchronize()
        assert torch.equal(env.hkin, twin.hkin) and torch.equal(env.hactions, twin.hactions), step
        ever |= risky_of(env)
        calm = ~ever
        assert torch.equal(env.kin[calm], twin.kin[calm]) and torch.equal(env.obs[calm], twin.obs[calm]), step
    assert 0 < int(ever.sum()) < n
    env.close()
    twin.close()


@pytest.mark.parametrize("scene", ["space_bm", "human"])
def test_ranges_and_host_step_agree(scene):
    """One or two ranges of the device step and the host-buffer step (CUDA graph, 1 or 3 ranges) decide and step alike."""
    n = 1000
    envs = [make_env(scene, n, shield=True) for _ in range(4)]
    for e in envs:
        e.reset()
    one, two, host1, host3 = envs
    one.set_step_ranges(1)
    two.set_step_ranges(2)
    rng = np.random.default_rng(13)
    risky_total = 0
    for step in range(6):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        one.step(act)
        two.step(act)
        host1.step_host(act, chunks=1)
        host3.step_host(act, chunks=3)
        torch.cuda.synchronize()
        for e in (two, host1, host3):
            for k in ("info", "kin", "obs", "reward", "done"):
                assert torch.equal(getattr(e, k), getattr(one, k)), (scene, step, k)
        risky_total += int(risky_of(one).sum())
    assert risky_total > 0
    for e in envs:
        e.close()


def test_lookahead_leaves_the_real_records_alone():
    """The shadow steps write only shadow buffers.  The proposals are the backup policy's own float32 actions, so a
    shielded env executes the same action as an ungated twin whether or not the look-ahead flags it (from some start
    states the backup policy itself collides within the window).  Then the real statistics, episode records, states and
    rewards equal the twin's in every env, episode ends included; only the gate's own bookkeeping (risky_action_rate, the
    first risky step) differs.  And risk_ground_truth, called while the mode is on, still restores the state bit for bit
    and leaves the mode on."""
    n = 256
    env = make_env("space_bm", n, shield=True)
    twin = make_env("space_bm", n, shield=False)
    twin.load_networks()
    env.reset()
    env.episode[:, 0] = 17          # every episode reaches its length (20 steps) within the window
    twin.restore(env.snapshot())
    gate_cols = [abi.EP_SCALARS.index("risky_action_rate") + 16 * h for h in range(3)] + [abi.EPC["first_risky_step"]]
    rec_cols = [c for c in range(abi.SM_EP_STRIDE) if c not in gate_cols]
    risky_total = 0
    for step in range(4):
        act = twin.mlp_forward_exact(1, twin.risk_observation(), n_out=7)
        env.step(act)
        twin.step(act)
        torch.cuda.synchronize()
        risky_total += int(risky_of(env).sum())
        for k in ("kin", "obst", "obs", "reward", "done", "term_reason"):
            assert torch.equal(getattr(env, k), getattr(twin, k)), (step, k)
        assert torch.equal(env.episode[:, :3], twin.episode[:, :3]), step
        for k in ("epacc", "epinfo"):
            assert torch.equal(getattr(env, k)[:, rec_cols], getattr(twin, k)[:, rec_cols]), (step, k)
        # the statistics are summed with atomics: counts are exact, the sum of the returns is exact up to its order
        counts = [0] + list(range(2, 32))
        assert torch.equal(env.stats[counts], twin.stats[counts]), (step, env.stats, twin.stats)
        assert torch.allclose(env.stats[1], twin.stats[1], rtol=1e-12, atol=0), (step, env.stats[1], twin.stats[1])
    print("envs whose backup action the look-ahead flagged over 4 steps: {} of {}".format(risky_total, 4 * n))
    assert env.stats[0].item() >= n   # every first episode ended (by its length at the latest) and was counted once
    # risk_ground_truth while the look-ahead is on
    other = make_env("space_bm", n, shield=True)
    other.restore(env.snapshot())
    before = {k: v.clone() for k, v in env.snapshot().items()}
    act = torch.from_numpy(np.random.default_rng(4).uniform(-1, 1, (n, 7)).astype(np.float32)).cuda()
    env.risk_ground_truth(act, K)
    after = env.snapshot()
    for k in before:
        assert torch.equal(before[k], after[k]), k
    env.step(act)
    other.step(act)
    torch.cuda.synchronize()
    assert torch.equal(env.info, other.info) and torch.equal(env.kin, other.kin)
    for e in (env, twin, other):
        e.close()
