"""Parity of the Human scene (BASELINE.json configs[2]; Human, ctlp.py:4647-4959) on the GPU against the CPU oracle,
through the C ABI.  The nested env's joint trajectory is float64 on both sides: bit-exact.  Geometry (distances,
contacts, the braking-trajectory collision predicate) is float32 on the device: decisions may differ within 1e-5 m of a
threshold; such envs are dropped from the comparison and counted.  A braking decision may differ only where the oracle's
check visited a pose whose smallest pair distance lies within 1e-5 m of the safety distance."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle  # noqa: E402
from safemotionsrisk_b200 import abi, human_backup_config  # noqa: E402

I = abi.INFO


def make_env(n, **kw):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=3, auto_reset=False)
    opts.update(kw)
    cfg_kw = opts.pop("cfg", {})
    return SafeMotionsVecEnv(num_envs=n, config=human_backup_config(**cfg_kw), **opts)


def _inject(env, orc, n, rng):
    start, _ = env.pools()
    hstart, htarget = env.human_pools()
    q, v, a, ob = start[:n, 0:7], start[:n, 8:15], start[:n, 16:23], start[:n, 32:48]
    hq, hv, ha = hstart[:n, 0:8], hstart[:n, 8:16], hstart[:n, 16:24]
    arm = rng.integers(0, 2, n)
    ft = htarget[arm, rng.integers(0, htarget.shape[1], n), :3]
    env.set_state(q, v, a, ob)
    env.set_human_state(hq, hv, ha, ft, arm)
    orc.set_state(q, v, a, ob)
    orc.set_human_state(hq, hv, ha, ft, arm)
    return hstart, htarget


def test_human_pools_are_valid_start_states():
    env = make_env(256)
    hstart, htarget = env.human_pools()
    sc = env.scene
    assert (hstart[:, 0:8] >= sc.human_pos_lo).all() and (hstart[:, 0:8] <= sc.human_pos_hi).all()
    assert (np.abs(hstart[:, 8:16]) <= sc.human_vel_max).all() and (np.abs(hstart[:, 16:24]) <= sc.human_acc_max).all()
    assert (hstart[:, 8:16] != 0).any(axis=1).mean() > 0.5       # most start states move (kinematic sampling / walk)
    box = np.array([[0.0, 0.6], [-0.8, 0.8], [0.075, 0.75]])
    for r in range(2):
        assert (htarget[r, :, :3] >= box[:, 0] - 1e-6).all() and (htarget[r, :, :3] <= box[:, 1] + 1e-6).all()
    # the sampled poses are free of collisions for the oracle as well (clearance 0.05 / 0.1 > safety distance 0.01);
    # rest poses only: moving ones have left the sampled pose
    rest = np.where((hstart[:, 8:16] == 0).all(1))[0][:40]
    for e in rest:
        assert not oracle.human_pose_collides(sc, hstart[e, 0:8])
    env.close()


def test_human_rollout_matches_oracle():
    n, steps = 192, 14
    env = make_env(n)
    env.set_human_actions_external(True)
    sc = env.scene
    assert sc.obs_size == 45
    orc = oracle.OracleEnvs(sc, n)
    rng = np.random.default_rng(7)
    _inject(env, orc, n, rng)
    assert np.array_equal(env.hkin.cpu().numpy(), orc.hkin)
    assert np.abs(env.hobs.cpu().numpy() - orc.hobs).max() < 1e-5
    assert np.abs(env.obs.cpu().numpy() - orc.obs).max() < 1e-5
    alive = np.ones(n, dtype=bool)        # robot side still comparable
    same_h = np.ones(n, dtype=bool)       # nested env still on the same trajectory
    dropped = 0
    for s in range(steps):
        act = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        hact = rng.uniform(-1, 1, (n, 8)).astype(np.float32)
        env.hactions.copy_(torch.from_numpy(hact))
        obs, rew, done, info = env.step(act)
        torch.cuda.synchronize()
        hs = env.hstate.cpu().numpy()
        # the target point the device drew for an arm that became active is what the oracle gets as "next target"
        act_arm = (hs[:, 12 + abi.TP_ACTIVE] != 0).astype(int)
        nt = np.stack([hs[np.arange(n), 12 * act_arm + abi.TP_POS + i] for i in range(3)], 1)
        o_obs, o_rew, o_done, _, o_info = orc.step_human(act, hact, nt)
        # ---- nested env: braking decision, joint trajectory, bookkeeping, observation
        braked_d, braked_o = hs[:, abi.HS_BRAKED] != 0, orc.hinfo[:, 0] != 0
        flip = same_h & (braked_d != braked_o)
        assert (orc.hmargin[flip] < 1e-5).all(), "braking decisions differ away from a knife edge at step {}: margins {}".format(
            s, orc.hmargin[flip & (orc.hmargin >= 1e-5)])
        same_h &= ~flip
        hk = env.hkin.cpu().numpy()
        assert np.array_equal(hk[same_h], orc.hkin[same_h]), "human joint trajectory differs at step {}".format(s)
        reach_flip = same_h & ((hs[:, [abi.TP_ACTIVE, 12 + abi.TP_ACTIVE]] != orc.hstate[:, [abi.TP_ACTIVE, 12 + abi.TP_ACTIVE]]).any(1))
        dropped += int(reach_flip.sum())
        same_h &= ~reach_flip
        assert np.array_equal(hs[same_h, abi.HS_BRAKE_COUNT], orc.hstate[same_h, abi.HS_BRAKE_COUNT])
        assert np.abs(env.hobs.cpu().numpy()[same_h] - orc.hobs[same_h]).max() < 1e-5
        # ---- main env
        ok = alive & same_h
        assert np.array_equal(env.kin.cpu().numpy()[alive], orc.kin[alive]), "robot joint trajectory"
        d_dev, d_ref = info.cpu().numpy()[:, :3], o_info[:, :3].copy()
        d_ref[(d_ref[:, 1] > 0.05) & (d_ref[:, 1] <= 0.102), 1] = 0.102   # reporting rule of the self class (test_gpu_parity.reported)
        edge = np.zeros(n, dtype=bool)
        for col, caps in ((0, (1e-3, 0.102)), (1, (1e-3, 0.102)), (2, (1e-3, 0.6))):
            for th in caps:
                edge |= np.abs(d_ref[:, col] - th) < 1e-5
        flags_equal = (info.cpu().numpy()[:, 3:6] == o_info[:, 3:6]).all(1) & (done.cpu().numpy() == o_done)
        bad = ok & ~flags_equal & ~edge
        # a contact latched within 1e-5 m of its manifold threshold may differ too: allow a handful
        assert bad.sum() <= max(1, n // 100), "flags differ in {} envs at step {}".format(bad.sum(), s)
        dropped += int((ok & ~flags_equal).sum())
        alive &= flags_equal | ~ok
        ok = alive & same_h
        assert np.abs(d_dev - d_ref)[ok].max() < 1e-4, "distances"
        assert np.allclose(rew.cpu().numpy()[ok], o_rew[ok], rtol=1e-4, atol=1e-4), "reward"
        assert np.abs(obs.cpu().numpy()[ok] - o_obs[ok]).max() < 1e-5, "observation"
        alive &= o_done == 0
        same_h &= o_done == 0
        if not alive.any():
            break
    assert dropped <= n // 8, "too many knife-edge drops: {}".format(dropped)
    env.close()


def test_human_policy_head_and_auto_reset():
    """The human's policy on the tensor cores + Philox noise: the actions land in [-1, 1], differ between envs and
    steps, the mean of many draws follows the network's mean output; episodes restart (30 steps) with a fresh nested env."""
    from oracle import mlp
    n = 2048
    env = make_env(n, auto_reset=True)
    env.reset()
    w = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "safemotionsrisk_b200", "assets",
                             "networks_human.npz"))
    hobs = env.hobs.cpu().numpy().copy()
    x = hobs[:, :38]
    for name in ("fc_1", "fc_2"):
        x = mlp.swish(x @ w["human/{}/kernel".format(name)] + w["human/{}/bias".format(name)])
    out = np.tanh(x @ w["human/fc_out/kernel"] + w["human/fc_out/bias"])
    mean, log_std = out[:, :8], -1.375 + 0.5 * (out[:, 8:] + 1) * 1.375
    env.step_random()
    torch.cuda.synchronize()
    ha = env.hactions.cpu().numpy()
    assert (np.abs(ha) <= 1).all()
    z = (ha - mean) / np.exp(log_std)
    inside = np.abs(ha) < 0.999                      # clipped draws carry no information about eps
    assert abs(z[inside].mean()) < 0.05 and 0.8 < z[inside].std() < 1.1
    first = env.hstate.cpu().numpy()[:, abi.HS_STEPS].copy()
    for _ in range(31):
        env.step_random()
    torch.cuda.synchronize()
    hs = env.hstate.cpu().numpy()
    assert (env.episode.cpu().numpy()[:, 1] >= 2).all()              # every env was reset at least once (30-step episodes)
    assert (hs[:, abi.HS_STEPS] <= 30).all() and (first <= 1).all()   # 0: the env collided in its first step and restarted
    active = hs[:, [abi.TP_ACTIVE, 12 + abi.TP_ACTIVE]]
    assert (active.sum(1) == 1).all()
    hk = env.hkin.cpu().numpy()
    sc = env.scene
    assert (hk[:, 0:8] >= sc.human_pos_lo - 1e-9).all() and (hk[:, 0:8] <= sc.human_pos_hi + 1e-9).all()
    assert np.array_equal(env.obs.cpu().numpy()[:, 21:], env.hobs.cpu().numpy()[:, :24])
    s = env.episode_statistics().cpu().numpy()
    assert s[0] >= n
    env.close()


def test_human_golden_rollout():
    """Committed oracle vectors of the Human scene (tests/golden/human.npz): same start states, robot actions and human
    actions through the CUDA step.  Joint space bit-exact; an env whose braking decision or collision flag sits on a
    float32 knife edge leaves the comparison (counted)."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "human.npz"))
    n = g["q"].shape[0]
    env = make_env(n)
    env.set_human_actions_external(True)
    env.set_state(g["q"], g["v"], g["a"], np.zeros((n, 16)))
    env.set_human_state(g["hq"], g["hv"], g["ha"], g["first_target"], g["arm"])
    torch.cuda.synchronize()
    assert np.array_equal(env.kin.cpu().numpy(), g["kin0"]) and np.array_equal(env.hkin.cpu().numpy(), g["hkin0"])
    assert np.abs(env.obs.cpu().numpy() - g["obs0"]).max() < 1e-6 and np.abs(env.hobs.cpu().numpy() - g["hobs0"]).max() < 1e-6
    k0 = env.hstate.cpu().numpy()[:, abi.HS_BRAKE_COUNT].astype(int)
    assert np.array_equal(k0, g["hstate0"][:, abi.HS_BRAKE_COUNT].astype(int))
    for e in range(n):
        assert np.array_equal(env.hbrake.cpu().numpy().reshape(n, -1, 8)[e, :k0[e]], g["hbrake0"].reshape(n, -1, 8)[e, :k0[e]])
    alive = np.ones(n, dtype=bool)
    same_h = np.ones(n, dtype=bool)
    dropped = 0
    for s in range(g["actions"].shape[0]):
        env.hactions.copy_(torch.from_numpy(g["hactions"][s]))
        obs, rew, done, info = env.step(g["actions"][s])
        torch.cuda.synchronize()
        hs, hk = env.hstate.cpu().numpy(), env.hkin.cpu().numpy()
        flip = same_h & ((hs[:, abi.HS_BRAKED] != 0) != (g["out_hinfo"][s][:, 0] != 0))
        flip |= same_h & (hs[:, [abi.TP_ACTIVE, 12 + abi.TP_ACTIVE]] != g["out_hstate"][s][:, [abi.TP_ACTIVE, 12 + abi.TP_ACTIVE]]).any(1)
        dropped += int(flip.sum())
        same_h &= ~flip
        assert np.array_equal(hk[same_h], g["out_hkin"][s][same_h]), "human joint trajectory, step {}".format(s)
        assert np.array_equal(hs[same_h, abi.HS_BRAKE_COUNT], g["out_hstate"][s][same_h, abi.HS_BRAKE_COUNT])
        hb, hb_ref = env.hbrake.cpu().numpy().reshape(n, -1, 8), g["out_hbrake"][s].reshape(n, -1, 8)
        for e in np.where(same_h)[0]:    # only the first `count` rows of the stored braking trajectory are defined
            k = int(hs[e, abi.HS_BRAKE_COUNT])
            assert np.array_equal(hb[e, :k], hb_ref[e, :k]), "stored braking trajectory, env {} step {}".format(e, s)
        assert np.abs(env.hobs.cpu().numpy()[same_h] - g["out_hobs"][s][same_h]).max() < 1e-5
        assert np.array_equal(env.kin.cpu().numpy()[alive], g["out_kin"][s][alive]), "robot joint trajectory"
        ok = alive & same_h
        o_info = g["out_info"][s]
        d_dev, d_ref = info.cpu().numpy()[:, :3], o_info[:, :3].copy()
        d_ref[(d_ref[:, 1] > 0.05) & (d_ref[:, 1] <= 0.102), 1] = 0.102   # reporting rule of the self class
        flags_equal = (info.cpu().numpy()[:, 3:6] == o_info[:, 3:6]).all(1) & (done.cpu().numpy() == g["out_done"][s])
        dropped += int((ok & ~flags_equal).sum())
        alive &= flags_equal | ~ok
        ok = alive & same_h
        if ok.any():
            assert np.abs(d_dev - d_ref)[ok].max() < 1e-4, "distances"
            assert np.allclose(rew.cpu().numpy()[ok], g["out_reward"][s][ok], rtol=1e-4, atol=1e-4), "reward"
            assert np.abs(obs.cpu().numpy()[ok] - g["out_obs"][s][ok]).max() < 1e-5, "observation"
            assert np.array_equal(env.term_reason.cpu().numpy()[ok], g["out_term"][s][ok])
        alive &= g["out_done"][s] == 0
        same_h &= g["out_done"][s] == 0
    assert dropped <= 2, "knife-edge drops: {}".format(dropped)
    env.close()


def test_human_full_size_invariants():
    """BASELINE.json configs[2] at its full size (65 536 envs): size-independent properties of the nested env and of the
    main env over auto-reset steps with the human's policy in the loop."""
    n = 65536
    env = make_env(n, seed=1, auto_reset=True)
    sc = env.scene
    env.reset()
    hlo, hhi, hV, hA = (torch.tensor(x, device=env.device) for x in (sc.human_pos_lo, sc.human_pos_hi, sc.human_vel_max,
                                                                     sc.human_acc_max))
    lo, hi, V = (torch.tensor(x, device=env.device) for x in (sc.pos_lo, sc.pos_hi, sc.vel_max))
    total_done, braked = 0, 0
    for s in range(35):
        obs, rew, done, info = env.step_random()
        hq, hv, ha = env.hkin[:, 0:8], env.hkin[:, 8:16], env.hkin[:, 16:24]
        # position limits: kept by the safe range, except while an env executes the INITIAL braking trajectory of its
        # reset -- the reference computes that one without advancing the position along it (ctlp.py:1120-1139, restated
        # as is), so a start state close to a limit overshoots it by a few mrad (measured: 2 - 4 of 65 536 envs, <= 7 mrad)
        over = (torch.clamp(hq - hhi, min=0) + torch.clamp(hlo - hq, min=0)).max(1).values
        assert int((over > 1e-6).sum()) <= n // 4096 and float(over.max()) < 0.02, "human joint positions inside their limits"
        assert bool((hv.abs() <= hV * (1 + 1e-9)).all()) and bool((ha.abs() <= hA * (1 + 1e-12)).all())
        q, v = env.kin[:, 0:7], env.kin[:, 8:15]
        assert bool(((q >= lo - 1e-6) & (q <= hi + 1e-6)).all()) and bool((v.abs() <= V * (1 + 1e-9)).all())
        assert bool((obs.abs() <= 1).all()) and bool((env.hobs.abs() <= 1).all()) and bool(torch.isfinite(rew).all())
        assert bool((env.hactions.abs() <= 1).all())
        hs = env.hstate
        assert bool(((hs[:, abi.TP_ACTIVE] != 0).int() + (hs[:, 12 + abi.TP_ACTIVE] != 0).int() == 1).all())   # one active target
        assert bool((hs[:, abi.HS_BRAKE_COUNT] >= 0).all()) and bool((hs[:, abi.HS_BRAKE_COUNT] <= abi.SM_HBRAKE_STEPS).all())
        assert bool(torch.equal(obs[:, 21:], env.hobs[:, :24]))       # the human's kinematic observation inside the main obs
        assert bool((info[:, I["episode_length"]] <= 30).all())
        braked += int((hs[:, abi.HS_BRAKED] != 0).sum())
        total_done += int((done > 0).sum())
    assert total_done > n                         # 30-step episodes: every env finished at least once
    assert 0 < braked < 35 * n // 2               # the braking-trajectory method intervenes, but not most of the time
    stats = env.episode_statistics().cpu().numpy()
    assert stats[0] == total_done
    env.close()


def test_human_backup_look_ahead_restores_the_nested_env():
    """risk_ground_truth in the Human scene: the look-ahead (robot under its backup policy, human under its own policy)
    runs on a copy; afterwards both envs are bit for bit where they were, and the labels separate risky from safe rows."""
    n = 2048
    env = make_env(n, auto_reset=True)
    env.load_networks()
    env.reset()
    for _ in range(3):
        env.step_random()
    before = {k: v.clone() for k, v in env.snapshot().items()}
    assert {"hkin", "hstate", "hbrake", "hobs"} <= set(before)
    act = np.random.default_rng(4).uniform(-1, 1, (n, 7)).astype(np.float32)
    state, a, risk = env.risk_ground_truth(act, 20)
    after = env.snapshot()
    for k in before:
        assert torch.equal(before[k], after[k]) or (before[k].isnan() == after[k].isnan()).all(), k
    assert state.shape == (n, 45) and 0.02 < float(risk.mean()) < 0.98
    shipped = env.mlp_forward_exact(0, state, a)[:, 0].cpu().numpy()
    r = risk.cpu().numpy() > 0.5
    assert shipped[r].mean() > shipped[~r].mean()      # the shipped risk network rates the risky rows higher on average
    env.close()
