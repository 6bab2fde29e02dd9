"""The agent inside the step (smenv_step_agent): the policy that acts in the env, evaluated on the tensor cores and sampled
on the device, against twins stepped with the same actions from Python and against a float64 / NumPy-Philox rebuild.

The agent here is the scene's shipped backup policy with all 14 outputs (load_agent()), so its deterministic action is
exactly what the Python loop env.step(mlp_forward(...)[:, :7]) executes.
"""
import ctypes as C
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from agent_reference import agent_eps, diag_gaussian  # noqa: E402
from oracle import mlp  # noqa: E402
from safemotionsrisk_b200 import abi, ball_backup_config, cabi, human_backup_config, space_backup_config  # noqa: E402

ASSETS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "safemotionsrisk_b200", "assets")
SM_ERR_ARG, SM_ERR_STATE = -1, -4   # SmStatus (include/smenv.h)
LO, HI = -1.375, 0.0
CONFIGS = {"space_bm": lambda **k: space_backup_config(ball_machine_mode=True, **k),
           "ball_bm": lambda **k: ball_backup_config(ball_machine_mode=True, **k),
           "human": lambda **k: human_backup_config(**k)}
NETWORKS = {"space_bm": "space", "ball_bm": "ball", "human": "human"}
STATE = ("kin", "obst", "episode", "ep_return", "obs", "reward", "done", "term_reason", "info", "actions", "epacc",
         "epinfo", "hkin", "hstate", "hbrake", "hobs", "hactions")


def make_env(scene, n, agent=True, **kw):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=3, auto_reset=True)
    opts.update(kw)
    cfg = {k: opts.pop(k) for k in list(opts) if k.startswith("risk_")}
    env = SafeMotionsVecEnv(num_envs=n, config=CONFIGS[scene](**cfg), **opts)
    if agent:
        env.load_agent()
    return env


def assert_same(a, b, what, keys=STATE):
    for k in keys:
        x, y = getattr(a, k), getattr(b, k)
        if x is not None:
            assert torch.equal(x, y), (what, k)


def collided(env):
    return env.done.bool() & (env.term_reason != env.TERMINATION_TRAJECTORY_LENGTH)


@pytest.mark.parametrize("scene", ["space_bm", "ball_bm", "human"])
def test_deterministic_agent_equals_the_python_loop(scene):
    n = 4096
    env, twin = make_env(scene, n), make_env(scene, n)
    env.reset()
    twin.reset()
    nj = env.scene.n_joints
    for step in range(20):
        want = twin.mlp_forward(abi.SM_NET_AGENT, twin.obs, n_out=2 * nj)
        twin.step(want[:, :nj])
        env.step_agent(explore=False)
        torch.cuda.synchronize()
        assert_same(env, twin, (scene, step))
        assert not env.agent_logp.any()
        assert torch.equal(env.agent_dist_inputs[:, :nj], want[:, :nj]), (scene, step)
        assert torch.equal(env.agent_actions, want[:, :nj]), (scene, step)
        t = want[:, nj:].double()
        ls = (LO + 0.5 * (t + 1) * (HI - LO)).float()
        assert (env.agent_dist_inputs[:, nj:] - ls).abs().max().item() < 1e-6
    env.close()
    twin.close()


@pytest.mark.parametrize("scene", ["space_bm", "ball_bm", "human"])
def test_sampled_step_equals_a_step_with_its_own_actions(scene):
    """In the Human scene the twin's human draws its own policy noise: equal hactions mean the agent's noise stream does
    not disturb the human's."""
    n = 4096
    env, twin = make_env(scene, n), make_env(scene, n)
    env.reset()
    twin.reset()
    clipped = 0
    for step in range(10):
        env.step_agent(explore=True)
        twin.step(env.agent_actions.clamp(-1, 1))
        torch.cuda.synchronize()
        assert torch.equal(env.actions, env.agent_actions.clamp(-1, 1))
        assert_same(env, twin, (scene, step))
        clipped += int((env.agent_actions.abs() > 1).sum())
    assert clipped > 0
    env.close()
    twin.close()


@pytest.mark.parametrize("scene", ["space_bm", "human"])
def test_samples_rebuilt_on_the_host(scene):
    """65 536 envs: the samples of one step from forward_tc and NumPy Philox (tag 0xA6E7, the step's counter) within
    the bound of test_human_policy_actions_at_full_size, logp against the float64 head, z against N(0, 1)."""
    stats = pytest.importorskip("scipy.stats")
    n, steps = 65536, 3
    env = make_env(scene, n)
    env.reset()
    for _ in range(steps):                # the first step of the env uses step counter 0
        env.step_random()
    obs = env.obs.cpu().numpy().copy()
    env.step_agent(explore=True)
    torch.cuda.synchronize()
    nj = env.scene.n_joints
    sample = env.agent_actions.cpu().numpy().astype(np.float64)
    dist = env.agent_dist_inputs.cpu().numpy().astype(np.float64)
    logp = env.agent_logp.cpu().numpy().astype(np.float64)
    w = np.load(os.path.join(ASSETS, "networks_{}.npz".format(NETWORKS[scene])))
    out = mlp.forward_tc(mlp.shipped_layers(w, "backup"), obs, "swish", "tanh")
    eps = agent_eps(n, nj, steps, env._seed)
    want, want_clipped, _, _ = diag_gaussian(out, nj, LO, HI, eps)
    d = np.abs(sample - want)
    print("{}: agent samples max |difference| {:.2e}, max / (1 + |eps|) {:.2e}".format(
        scene, d.max(), (d / (1 + np.abs(eps))).max()))
    assert (d <= 2e-3 * (1 + np.abs(eps))).all()
    assert np.array_equal(env.actions.cpu().numpy(), np.clip(sample, -1, 1).astype(np.float32))
    # logp of the device's own distribution inputs and the noise
    t = 2.0 * (dist[:, nj:] - LO) / (HI - LO) - 1.0
    _, _, ref_logp, ref_dist = diag_gaussian(np.concatenate([dist[:, :nj], t], 1), nj, LO, HI, eps)
    assert np.abs(ref_dist - dist).max() < 1e-12
    print("{}: logp max |difference| {:.2e}".format(scene, np.abs(logp - ref_logp).max()))
    assert np.abs(logp - ref_logp).max() < 1e-4
    z = (sample - dist[:, :nj]) / np.exp(dist[:, nj:])
    p = stats.kstest(z.ravel(), "norm").pvalue
    print("{}: KS p-value of z {:.3g}".format(scene, p))
    assert p > 1e-3
    assert (np.abs(want_clipped - env.actions.cpu().numpy()) <= 2e-3 * (1 + np.abs(eps))).all()
    env.close()


def test_reproducible_across_ranges_runs_and_seeds():
    n = 5000
    envs = []
    for ranges in (1, 2, 3, 2):
        e = make_env("space_bm", n)
        e.set_step_ranges(ranges)
        e.reset()
        envs.append(e)
    for step in range(6):
        for e in envs:
            e.step_agent(explore=True)
        torch.cuda.synchronize()
        for e in envs[1:]:
            assert_same(envs[0], e, step)
            for k in ("agent_actions", "agent_logp", "agent_dist_inputs"):
                assert torch.equal(getattr(envs[0], k), getattr(e, k)), (step, k)
    # same state, same step counter, other seed: the same means, other samples
    a, b = envs[0], envs[1]
    snap = a.snapshot()
    a.set_seed(3)
    b.set_seed(4)
    a.restore(snap)
    b.restore(snap)
    a.step_agent(explore=True)
    b.step_agent(explore=True)
    torch.cuda.synchronize()
    assert torch.equal(a.agent_dist_inputs, b.agent_dist_inputs)
    assert (a.agent_actions != b.agent_actions).float().mean().item() > 0.99
    for e in envs:
        e.close()


def test_with_the_network_gate():
    """buf->actions keeps the agent's clipped proposal; decisions and the executed actions (through the state they lead
    to) equal those of step_gated on a twin; rollout records the proposal and risky."""
    n, thr = 4096, 0.065
    env = make_env("space_bm", n, risk_config_dir="risk_networks/state_action/space", risk_threshold=thr)
    twin = make_env("space_bm", n)
    twin.load_networks()
    env.reset()
    twin.reset()
    risky_total = 0
    for step in range(8):
        env.step_agent(explore=True)
        proposal = env.agent_actions.clamp(-1, 1)
        twin.step_gated(proposal, threshold=thr)
        torch.cuda.synchronize()
        assert torch.equal(env.actions, proposal)
        assert_same(env, twin, step)
        risky_total += int(env.info[:, abi.INFO["risky_action"]].sum().item())
    assert risky_total > 0
    ro = env.rollout(4)
    assert ro["risky"].shape == (4, n) and ro["risky"].dtype == torch.bool
    for t in range(4):
        assert torch.equal(twin.obs, ro["obs"][t])
        twin.step_gated(ro["actions"][t].clamp(-1, 1), threshold=thr)
        assert torch.equal(twin.info[:, abi.INFO["risky_action"]] > 0.5, ro["risky"][t]), t
        assert torch.equal(twin.reward, ro["rewards"][t])
    assert torch.equal(twin.obs, ro["last_obs"])
    env.close()
    twin.close()


def test_with_the_lookahead():
    n, k = 512, 5
    cfg = dict(risk_config_dir="risk_networks/state_action/space", risk_threshold=0.065, risk_state_config=4,
               risk_state_backup_trajectory_steps=k)
    env, twin = make_env("space_bm", n, **cfg), make_env("space_bm", n, **cfg)
    env.reset()
    twin.reset()
    risky_total = 0
    for step in range(8):
        env.step_agent(explore=True)
        proposal = env.agent_actions.clamp(-1, 1)
        twin.step(proposal)
        torch.cuda.synchronize()
        assert torch.equal(env.actions, proposal)
        assert_same(env, twin, step)
        risky_total += int(env.info[:, abi.INFO["risky_action"]].sum().item())
    ro = env.rollout(3)
    for t in range(3):
        twin.step(ro["actions"][t].clamp(-1, 1))
        assert torch.equal(twin.info[:, abi.INFO["risky_action"]] > 0.5, ro["risky"][t]), t
    print("look-ahead K = {}: {} risky proposals in 8 steps of {} envs".format(k, risky_total, n))
    env.close()
    twin.close()


def test_rollout_equals_step_agent_by_hand():
    n, T = 4096, 16
    env, ref = make_env("space_bm", n), make_env("space_bm", n)
    env.reset()
    ref.reset()
    ro = env.rollout(T)
    assert "risky" not in ro
    for t in range(T):
        assert torch.equal(ref.obs, ro["obs"][t]), t
        ref.step_agent(explore=True)
        assert torch.equal(ref.agent_actions, ro["actions"][t]), t
        assert torch.equal(ref.agent_logp, ro["action_logp"][t]), t
        assert torch.equal(ref.agent_dist_inputs, ro["action_dist_inputs"][t]), t
        assert torch.equal(ref.reward, ro["rewards"][t]), t
        assert torch.equal(ref.done.bool(), ro["dones"][t]), t
    assert torch.equal(ref.obs, ro["last_obs"])
    assert_same(env, ref, "after the rollout")
    # launches: the step's own plus the agent's network and head, per env range
    ranges = env.launch_config()["step_ranges"]
    c0 = env.launch_count()
    env.step(env.actions)
    c1 = env.launch_count()
    env.step_agent()
    c2 = env.launch_count()
    assert c2 - c1 == (c1 - c0) + 2 * ranges
    env.close()
    ref.close()


def test_refusals(tmp_path):
    env = make_env("ball_bm", 256, agent=False)
    lib, h, s = env._lib, env._handle, env._stream()
    step = lambda buf: lib.smenv_step_agent(h, C.byref(buf), 0, 1, None, None, None, s)   # noqa: E731
    assert step(env._buf) == SM_ERR_STATE                                    # no agent loaded
    layers = lambda f: [(f["backup/{}/kernel".format(k)], f["backup/{}/bias".format(k)])   # noqa: E731
                        for k in ("fc_1", "fc_2", "fc_out")]
    space = layers(np.load(os.path.join(ASSETS, "networks_space.npz")))      # 23 inputs, the Ball env has 27
    ball = layers(np.load(os.path.join(ASSETS, "networks_ball.npz")))
    narrow = ball[:2] + [(ball[2][0][:, :7], ball[2][1][:7])]                 # 7 outputs, the head needs 14

    def save(name, net):
        path = str(tmp_path / name)
        np.savez(path, **{"agent/{}/{}".format(k, part): v for k, (kern, bias) in zip(("fc_1", "fc_2", "fc_out"), net)
                          for part, v in (("kernel", kern), ("bias", bias))})
        return path

    def raw_load(net):
        dims = np.array([net[0][0].shape[0]] + [k.shape[1] for k, _ in net], dtype=np.int32)
        flat = np.concatenate([np.concatenate([k.astype(np.float32).ravel(), b.astype(np.float32).ravel()])
                               for k, b in net])
        cabi.check(lib.smenv_mlp_load(h, abi.SM_NET_AGENT, len(net) - 1, dims.ctypes.data, 1, 1, flat.ctypes.data),
                   "smenv_mlp_load")

    with pytest.raises(ValueError):
        env.load_agent(save("space.npz", space))
    with pytest.raises(ValueError):
        env.load_agent(save("narrow.npz", narrow))
    raw_load(space)
    assert step(env._buf) == SM_ERR_STATE                                    # input width
    raw_load(narrow)
    assert step(env._buf) == SM_ERR_STATE                                    # output count
    env.load_agent(save("ball.npz", ball))                                    # the same network from an agent/ file
    no_obs = abi.SmBuffers.from_buffer_copy(env._buf)
    no_obs.obs = None
    assert step(no_obs) == SM_ERR_ARG
    no_act = abi.SmBuffers.from_buffer_copy(env._buf)
    no_act.actions = None
    assert step(no_act) == SM_ERR_ARG
    assert lib.smenv_set_agent_head(h, 0.5, -0.5) == SM_ERR_ARG
    assert lib.smenv_set_agent_head(h, -0.5, -0.5) == 0
    with pytest.raises(ValueError):
        env.load_agent(log_std_range=(0.5, -0.5))
    env.reset()
    env.step_agent()                                                          # still usable
    torch.cuda.synchronize()
    assert (env.agent_actions.abs() <= 10).all()
    env.close()


def test_sampled_backup_policy_collides_less_than_random_actions():
    """space_bm, 16 384 envs, 60 steps: the share of episodes that end in a collision."""
    n, T = 16384, 60
    envs = {k: make_env("space_bm", n) for k in ("deterministic", "sampled", "random")}
    for e in envs.values():
        e.reset()
    hits = {k: 0 for k in envs}
    episodes = {k: n for k in envs}
    for _ in range(T):
        envs["deterministic"].step_agent(explore=False)
        envs["sampled"].step_agent(explore=True)
        envs["random"].step_random()
        for k, e in envs.items():
            hits[k] += int(collided(e).sum())
            episodes[k] += int(e.done.sum())
    rate = {k: hits[k] / episodes[k] for k in envs}
    print("space_bm, {} envs, {} steps: episodes ending in a collision: deterministic {:.4f}, sampled {:.4f}, "
          "random {:.4f}".format(n, T, rate["deterministic"], rate["sampled"], rate["random"]))
    assert rate["sampled"] < 0.5 * rate["random"]
    for e in envs.values():
        e.close()
