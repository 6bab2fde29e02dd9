"""Rating the simulated next state with a state risk network as the risk check inside the step (risk_state_config 3,
smenv_set_risk_next_state).

The state networks are built here: seeded random MLPs with the shipped risk network's hidden widths, written with
risk_train.export_weights, the threshold at a quantile of their risk so that both decisions occur.  The decisions are
checked bit for bit against a Python twin that restates the check with the env's own hooks: snapshot, one step of the
proposal without auto reset and with the gate off, risk = 1 where that step ended in a collision, else the float32 state
network on the risk observation it leads to, restore.
"""
import argparse
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from safemotionsrisk_b200 import (abi, ball_backup_config, cabi, human_backup_config, risk_data, risk_train,  # noqa: E402
                                  space_backup_config, space_task_config)
from safemotionsrisk_b200.scene import Scene  # noqa: E402

I = abi.INFO
CONFIGS = {"space_bm": lambda **k: space_backup_config(ball_machine_mode=True, **k),
           "ball_bm": lambda **k: ball_backup_config(ball_machine_mode=True, **k),
           "space_task_bm": lambda **k: space_task_config(ball_machine_mode=True, **k),
           "human": lambda **k: human_backup_config(**k)}
SEEDS = {"space_bm": 11, "ball_bm": 12, "space_task_bm": 13, "human": 14}


@pytest.fixture(scope="module")
def state_nets(tmp_path_factory):
    """scene -> .npz of a seeded random state risk network: risk observation -> 512 -> 256 -> 128 -> 1, selu / sigmoid."""
    root = tmp_path_factory.mktemp("state_nets")
    out = {}
    for scene, seed in SEEDS.items():
        sc = Scene(CONFIGS[scene]())
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(seed)
            model = risk_train.build_model(sc.obs_size - sc.obs_target_size, [512, 256, 128], "selu")
        out[scene] = str(root / "{}.npz".format(scene))
        risk_train.export_weights(model, out[scene], "selu", "sigmoid")
    return out


def make_env(scene, n, net, threshold=0.5, **kw):
    """The env as a user gets it from risk_state_config=3 with the state network `net`."""
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=3, auto_reset=True)
    opts.update(kw)
    cfg = CONFIGS[scene](risk_config_dir=net, risk_threshold=threshold, risk_state_config=3)
    return SafeMotionsVecEnv(num_envs=n, config=cfg, **opts)


def make_twin(scene, n, net, **kw):
    """The same env with the gate off: it steps what it is given, and its networks serve the Python restatement."""
    twin = make_env(scene, n, net, **kw)
    twin.set_risk_gate(None)
    return twin


def collided(env):
    return env.done.bool() & (env.term_reason != env.TERMINATION_TRAJECTORY_LENGTH)


def risky_of(env):
    return env.info[:, I["risky_action"]] > 0.5


def state_risk(env):
    return env.mlp_forward_exact(0, env.risk_observation())[:, 0]


def quantile_threshold(env, q):
    return float(torch.quantile(state_risk(env), q).item())


def twin_next_state_risk(twin, act):
    """The check restated: one step of `act` from a copy of the state, without auto reset and with the gate off; risk 1
    where it ended the episode for a reason other than the trajectory length, else the float32 state network's rating
    of the risk observation it leads to.  The state is restored."""
    snap = twin.snapshot()
    auto = twin.auto_reset
    twin.auto_reset = False
    try:
        twin.step(act)
        risk = torch.where(collided(twin), torch.ones_like(twin.reward), state_risk(twin))
    finally:
        twin.restore(snap)
        twin.auto_reset = auto
    return risk


@pytest.mark.parametrize("scene", ["space_bm", "ball_bm", "space_task_bm"])
def test_decisions_equal_the_python_twin(scene, state_nets):
    """Every decision and every reported risk equals the twin's, and the real step equals the twin's step with the decided
    actions (the float32 backup action where risky).  The band covers every row, so that the reported risk is the float32
    rating everywhere (outside the band the info slot holds the tensor-core rating)."""
    n = 1000   # ragged against the ranges of the step
    env = make_env(scene, n, state_nets[scene])
    twin = make_twin(scene, n, state_nets[scene])
    env.set_gate_exact(True, band=1.0)
    env.reset()
    rng = np.random.default_rng(5)
    env.set_risk_gate(None)
    for _ in range(3):
        env.step(rng.uniform(-1, 1, (n, 7)).astype(np.float32))
    thr = quantile_threshold(env, 0.7)
    env.set_risk_gate(thr)
    twin.restore(env.snapshot())
    risky_total = 0
    for step in range(5):
        act = torch.from_numpy(rng.uniform(-1, 1, (n, 7)).astype(np.float32)).cuda()
        risk = twin_next_state_risk(twin, act)
        want = risk >= thr
        backup = twin.mlp_forward_exact(1, twin.risk_observation(), n_out=7)
        twin.step(torch.where(want[:, None], backup, act))
        env.step(act)
        torch.cuda.synchronize()
        risky = risky_of(env)
        assert torch.equal(risky, want), (scene, step, int((risky != want).sum()))
        assert torch.equal(env.info[:, I["risk"]], risk), (scene, step)
        for k in ("kin", "obst", "obs", "done"):
            assert torch.equal(getattr(env, k), getattr(twin, k)), (scene, step, k)
        assert torch.equal(env.episode[:, :3], twin.episode[:, :3]), (scene, step)   # [:, 3]: first risky step
        keep = ~risky
        assert torch.equal(env.reward[keep], twin.reward[keep]), (scene, step)
        risky_total += int(risky.sum())
    assert 0 < risky_total < 5 * n
    env.close()
    twin.close()


@pytest.mark.parametrize("scene", ["space_bm", "human"])
def test_kept_actions_never_collide(scene, state_nets):
    """The simulated step is the real step: an action the check keeps cannot end the step in a collision."""
    n = 16384
    env = make_env(scene, n, state_nets[scene])
    env.reset()
    env.set_risk_gate(quantile_threshold(env, 0.8))
    kept = hits = 0
    for step in range(10):
        env.step_random()
        torch.cuda.synchronize()
        risky = risky_of(env)
        assert not bool((collided(env) & ~risky).any()), (scene, step)
        kept += int((~risky).sum())
        hits += int(collided(env).sum())
    print("{}: {} of {} actions kept, {} steps ended in a collision (all with the backup action)".format(
        scene, kept, 10 * n, hits))
    assert 0 < kept < 10 * n
    env.close()


def test_human_scene_against_an_ungated_twin(state_nets):
    """The nested env of the human does not see the robot, and the simulated step draws the human's policy noise of the
    real step: the human's state and actions equal an ungated twin's in every env at every step; the robot equals the
    twin's in the envs that were never risky."""
    n = 2048
    env = make_env("human", n, state_nets["human"], auto_reset=False)
    twin = make_twin("human", n, state_nets["human"], auto_reset=False)
    env.reset()
    twin.reset()
    env.set_risk_gate(quantile_threshold(env, 0.8))
    rng = np.random.default_rng(9)
    ever = torch.zeros(n, dtype=torch.bool, device=env.device)
    for step in range(8):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        env.step(act)
        twin.step(act)
        torch.cuda.synchronize()
        for k in ("hkin", "hstate", "hobs", "hactions"):
            assert torch.equal(getattr(env, k), getattr(twin, k)), (step, k)
        ever |= risky_of(env)
        calm = ~ever
        assert torch.equal(env.kin[calm], twin.kin[calm]) and torch.equal(env.obs[calm], twin.obs[calm]), step
    assert 0 < int(ever.sum()) < n
    env.close()
    twin.close()


@pytest.mark.parametrize("scene", ["space_bm", "human"])
def test_ranges_and_host_step_agree(scene, state_nets):
    """One or two ranges of the device step and the host-buffer step (CUDA graph, 1 or 3 ranges) decide and step alike."""
    n = 1000
    envs = [make_env(scene, n, state_nets[scene]) for _ in range(4)]
    for e in envs:
        e.reset()
    one, two, host1, host3 = envs
    thr = quantile_threshold(one, 0.7)
    for e in envs:
        e.set_risk_gate(thr)
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
    assert 0 < risky_total < 6 * n
    for e in envs:
        e.close()


def test_simulated_step_leaves_the_real_records_alone(state_nets):
    """The simulated step writes only shadow buffers.  The proposals are the backup policy's own float32 actions, so the
    checked env executes the same action as an ungated twin whether or not the check flags it.  Then the real statistics,
    episode records, states and rewards equal the twin's in every env, episode ends included; only the gate's own
    bookkeeping (risky_action_rate, the first risky step) differs."""
    n = 256
    net = state_nets["space_bm"]
    env = make_env("space_bm", n, net)
    twin = make_twin("space_bm", n, net)
    env.reset()
    env.set_risk_gate(quantile_threshold(env, 0.5))
    env.episode[:, 0] = 17          # every episode reaches its length (20 steps) within the run
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
    assert 0 < risky_total < 4 * n
    assert env.stats[0].item() >= n   # every first episode ended (by its length at the latest) and was counted once
    env.close()
    twin.close()


def test_state_risk_ground_truth(state_nets):
    """state_risk_ground_truth labels the current states with initial_backup_trajectory_unsafe's rule, returns their risk
    observation and restores the state bit for bit, also while the check is on."""
    n = 2048
    env = make_env("space_bm", n, state_nets["space_bm"])
    env.reset()
    rng = np.random.default_rng(2)
    for _ in range(4):
        env.step(rng.uniform(-1, 1, (n, 7)).astype(np.float32))
    torch.cuda.synchronize()
    before = {k: v.clone() for k, v in env.snapshot().items()}
    obs = env.risk_observation().clone()
    state, risk = env.state_risk_ground_truth(20)
    after = env.snapshot()
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert torch.equal(state, obs) and state.shape == (n, env.scene.obs_size - env.scene.obs_target_size)
    assert risk.dtype == torch.float32 and risk.shape == (n,)
    assert torch.equal(risk, env.initial_backup_trajectory_unsafe(20).float())
    print("states whose backup trajectory ends in a collision: {} of {}".format(int(risk.sum()), n))
    env.close()


def test_state_risk_round_trip(tmp_path):
    """state_risk_ground_truth rows -> write_risk_csv (state_risk files) -> risk_train -> an env with
    risk_state_config=3 and the trained directory as risk_config_dir, whose gate then flags some actions, not all."""
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    n = 4096
    env = SafeMotionsVecEnv(num_envs=n, config=space_backup_config(ball_machine_mode=True), seed=21, auto_reset=True)
    env.load_networks()                    # the backup policy of the labelling roll-outs
    env.reset()
    rows = []
    gen = torch.Generator(device=env.device).manual_seed(4)
    for step in range(6):
        state, risk = env.state_risk_ground_truth(backup_steps=20)
        rows.append((state.cpu().numpy(), risk.cpu().numpy()))
        env.step(torch.rand((n, 7), device=env.device, generator=gen) * 2 - 1)
    env.close()
    state, risk = (np.concatenate([r[i] for r in rows]) for i in range(2))
    rate = float(risk.mean())
    print("state risk rate {:.4f} over {} rows".format(rate, len(risk)))
    assert 0.0 < rate < 1.0
    data = tmp_path / "set" / "data"
    n_train = 16384
    risk_data.write_risk_csv(str(data), state[:n_train], risk[:n_train], pid=1)
    os.rename(data / "state_risk", data / "train")
    risk_data.write_risk_csv(str(data), state[n_train:], risk[n_train:], pid=2)
    os.rename(data / "state_risk", data / "test")
    args = risk_train.add_arguments(argparse.ArgumentParser()).parse_args([
        "--risk_data_dir", str(data), "--experiment_name", "gpu", "--hidden_layer_activation", "selu",
        "--fcnet_hiddens", "[128, 64]", "--batch_size", "512", "--shuffle", "--epochs", "10", "--lr", "0.002",
        "--logdir", str(tmp_path / "results"), "--seed", "1", "--device", "cuda"])
    log_dir = risk_train.run(args, log=lambda *_: None)
    assert os.sep + "state_risk" + os.sep in log_dir
    env2 = SafeMotionsVecEnv(num_envs=n, config=space_backup_config(
        ball_machine_mode=True, risk_config_dir=log_dir, risk_threshold=0.5, risk_state_config=3), seed=21, auto_reset=True)
    assert env2.risk_network_kind == "state"
    env2.reset()
    env2.set_risk_gate(quantile_threshold(env2, 0.5))
    risky = 0
    for step in range(3):
        env2.step(torch.rand((n, 7), device=env2.device, generator=gen) * 2 - 1)
        torch.cuda.synchronize()
        risky += int(risky_of(env2).sum())
    print("trained state network: {} of {} actions risky".format(risky, 3 * n))
    assert 0 < risky < 3 * n
    env2.close()


def test_refusals(state_nets):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    net = state_nets["space_bm"]
    # a state network under the network gate
    with pytest.raises(ValueError):
        SafeMotionsVecEnv(num_envs=64, config=space_backup_config(ball_machine_mode=True, risk_config_dir=net,
                                                                  risk_threshold=0.5), seed=1)
    # a state-action network under risk_state_config 3
    shipped = os.path.join(os.path.dirname(os.path.abspath(abi.__file__)), "assets", "networks_space.npz")
    with pytest.raises(NotImplementedError):
        make_env("space_bm", 64, shipped)
    env = make_env("space_bm", 64, net)
    env.reset()
    with pytest.raises(cabi.SmEnvError):   # smenv_risk_gate rates (state, action) pairs
        env.risk_gate(0.5)
    with pytest.raises(cabi.SmEnvError):   # the look-ahead and the next-state check exclude each other
        env.set_risk_lookahead(20)
    with pytest.raises(cabi.SmEnvError):   # the gate is on: the network gate cannot take over a state network
        env.set_risk_next_state(False)
    env.set_risk_gate(None)
    env.set_risk_next_state(False)
    with pytest.raises(cabi.SmEnvError):   # the network gate with a state network
        env.set_risk_gate(0.5)
    env.set_risk_next_state(True)
    env.set_risk_gate(0.5)
    env.step_random()
    env.close()
    # risk_state_config 4 accepts a state network (the look-ahead does not consult it); the next-state check is refused
    la = SafeMotionsVecEnv(num_envs=64, config=space_backup_config(ball_machine_mode=True, risk_config_dir=net,
                                                                   risk_threshold=0.5, risk_state_config=4), seed=1)
    with pytest.raises(cabi.SmEnvError):
        la.set_risk_next_state(True)
    la.close()


# The gate's mode against the loaded risk network (smenv.h): every row starts in the network mode with the gate off and
# the network S (state) or SA (state-action, the shipped one) loaded, runs its setup, then the call under test.  Columns:
# setup, call, refused, and whether a following step_random() runs.  Under risk_state_config 4 both kinds load.
MODE_TABLE = [
    # set_risk_gate(t >= 0): refused in the network mode with S and in the next-state mode without S
    (["SA"], "gate", False, True),
    (["S"], "gate", True, True),
    (["S", "next_state", "SA"], "gate", True, True),
    (["S", "next_state"], "gate", False, True),
    (["S", "lookahead"], "gate", False, True),
    (["SA", "lookahead"], "gate", False, True),
    # set_risk_gate(None): never refused
    (["SA", "gate", "S"], "gate_off", False, True),
    (["S", "next_state", "gate", "SA"], "gate_off", False, True),
    # set_risk_lookahead(K > 0): refused in the next-state mode
    (["S", "next_state"], "lookahead", True, True),
    (["S", "next_state", "gate"], "lookahead", True, True),
    (["SA"], "lookahead", False, True),
    (["SA", "gate", "S"], "lookahead", False, True),
    (["S", "lookahead", "gate"], "lookahead", False, True),
    # set_risk_lookahead(0): refused when it leaves the gate on in the network mode with S
    (["S", "lookahead", "gate"], "lookahead_off", True, True),
    (["SA", "lookahead", "gate", "S"], "lookahead_off", True, True),
    (["SA", "gate", "S"], "lookahead_off", True, False),
    (["SA", "lookahead", "gate"], "lookahead_off", False, True),
    (["S", "lookahead"], "lookahead_off", False, True),
    (["S", "next_state", "gate"], "lookahead_off", False, True),
    (["S", "next_state", "gate", "SA"], "lookahead_off", False, False),
    # set_risk_next_state(1): refused without S and in the look-ahead mode
    (["SA"], "next_state", True, True),
    (["S", "lookahead"], "next_state", True, True),
    (["S", "lookahead", "gate"], "next_state", True, True),
    (["S"], "next_state", False, True),
    (["SA", "gate", "S"], "next_state", False, True),
    # set_risk_next_state(0): refused when it leaves the gate on in the network mode with S
    (["S", "next_state", "gate"], "next_state_off", True, True),
    (["SA", "gate", "S"], "next_state_off", True, False),
    (["S", "next_state", "gate", "SA"], "next_state_off", False, True),
    (["S", "lookahead", "gate"], "next_state_off", False, True),
    (["S", "next_state"], "next_state_off", False, True),
    # risk_gate: refused with S, whatever the mode
    (["S"], "risk_gate", True, True),
    (["S", "next_state"], "risk_gate", True, True),
    (["SA"], "risk_gate", False, True),
    (["SA", "lookahead"], "risk_gate", False, True),
    # the step with the gate on: refused in the network mode with S and in the next-state mode without S
    (["SA", "gate", "S"], None, False, False),
    (["S", "next_state", "gate", "SA"], None, False, False),
    (["SA", "lookahead", "gate", "S"], None, False, True),
]


def test_mode_and_network_table(state_nets):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    shipped = os.path.join(os.path.dirname(os.path.abspath(abi.__file__)), "assets", "networks_space.npz")
    nets = {"S": state_nets["space_bm"], "SA": shipped}
    env = SafeMotionsVecEnv(num_envs=64, config=space_backup_config(ball_machine_mode=True, risk_config_dir=nets["S"],
                                                                    risk_threshold=0.5, risk_state_config=4), seed=1)
    env.reset()
    calls = {"gate": lambda: env.set_risk_gate(0.5), "gate_off": lambda: env.set_risk_gate(None),
             "lookahead": lambda: env.set_risk_lookahead(5), "lookahead_off": lambda: env.set_risk_lookahead(0),
             "next_state": lambda: env.set_risk_next_state(True), "next_state_off": lambda: env.set_risk_next_state(False),
             "S": lambda: env.load_networks(nets["S"]), "SA": lambda: env.load_networks(nets["SA"]),
             "risk_gate": lambda: env.risk_gate(0.5)}

    def refuses(fn):
        try:
            fn()
        except cabi.SmEnvError:
            return True
        torch.cuda.synchronize()
        return False

    for setup, call, refused, steps in MODE_TABLE:
        row = "{} then {}".format(setup, call)
        env.set_risk_gate(None)            # with the gate off, both off-switches are accepted in every mode
        env.set_risk_next_state(False)
        env.set_risk_lookahead(0)
        for op in setup:
            calls[op]()
        if call is not None:
            assert refuses(calls[call]) == refused, row
        assert refuses(env.step_random) != steps, row
    env.close()
    # without the networks the gate and both modes are refused
    bare = SafeMotionsVecEnv(num_envs=64, config=space_backup_config(ball_machine_mode=True), seed=1)
    for call in (lambda: bare.set_risk_gate(0.5), lambda: bare.set_risk_lookahead(5),
                 lambda: bare.set_risk_next_state(True)):
        assert refuses(call)
    for call in (lambda: bare.set_risk_gate(None), lambda: bare.set_risk_lookahead(0),
                 lambda: bare.set_risk_next_state(False)):
        assert not refuses(call)
    bare.close()
