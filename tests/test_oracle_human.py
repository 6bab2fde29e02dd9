"""The Human scene in the oracle (ctlp.py:4647-4959; trained_networks/human_network/params.json): kinematic tree,
limits, pair sets, braking-trajectory method, target points, observation.  PARITY UNPINNED like the rest of the oracle:
what is checked here are closed forms, invariants and the constants the reference's files hold."""
import numpy as np
import pytest

from oracle import oracle
from safemotionsrisk_b200 import abi, human_backup_config
from safemotionsrisk_b200.scene import Scene


@pytest.fixture(scope="module")
def scene():
    return Scene(human_backup_config())


def test_human_scene_constants(scene):
    sc, h = scene.struct, scene.struct.human
    assert sc.obs_size == 45 and h.obs_size == 38                    # risk_config.json / checkpoint input widths
    assert sc.episode_steps == 30 and sc.n_obstacles == 1 and sc.obst_kind[0] == abi.SM_OBST_HUMAN
    assert h.n_arm_shapes == 22 and h.n_shapes == 40                 # SURVEY 8a: 2 x (4 + 3 + 4) parts, 18 body parts
    assert sc.n_mov_reward * sc.obst_shape_cnt[0] == 132             # SURVEY 2.1: 6 links x 22 convex parts
    assert h.n_brake_pairs == 203 and h.brake_checks == 3            # round(0.1 / 0.033) (ctlp.py:99-103)
    # human.urdf:140-416 limits without a safety buffer; robot_scene_base.py:24-25
    assert np.allclose(list(h.pos_lo), [-0.5, -1.4, -0.2, -2.6179938316345, -1.2, -1.4, -1.5708, -2.6179938316345])
    assert np.allclose(list(h.pos_hi), [1.2, 0.1, 1.5708, 0.087266445159912, 0.5, 0.1, 0.2, 0.087266445159912])
    assert np.allclose(list(h.vel_max), 1.710422666954443) and np.allclose(list(h.acc_max), 15.0)
    assert np.allclose(list(h.jerk_max), 300.0)
    assert list(h.joint_parent) == [0, 1, 2, 3, 0, 5, 6, 7]


def test_human_fk_closed_form(scene):
    """At q = 0 the shoulders sit where the URDF origins put them: base (0.7, 0, -0.94) turned by pi about z, root joint
    at z = 0.052 with rpy (0, -pi/2, 0), ... (human.urdf:3-145).  The elbow follows the shoulder rotation."""
    fr = oracle.human_fk(scene, np.zeros(8))
    assert np.allclose(fr[0, 9:], [0.7, 0, -0.94])
    for r, j in ((0, 1), (1, 5)):
        shoulder = fr[j, 9:]
        assert 1.25 < shoulder[2] + 0.94 < 1.4 and abs(abs(shoulder[1]) - 0.21) < 0.01    # shoulder height / width
        assert np.allclose(fr[j, 9:], fr[j + 1, 9:]) and np.allclose(fr[j, 9:], fr[j + 2, 9:])   # dummy links
        elbow = fr[j + 3, 9:]
        assert abs(np.linalg.norm(elbow - shoulder) - np.linalg.norm([0.001, 0.004, 0.276004])) < 2e-3
    # moving only the forearm joint keeps the shoulder frames and turns the hand about the elbow
    q = np.zeros(8)
    q[3] = -1.0
    fr2 = oracle.human_fk(scene, q)
    assert np.allclose(fr2[:4], fr[:4]) and np.allclose(fr2[4, 9:], fr[4, 9:])
    lp, lp2 = oracle.human_link_points(scene, np.zeros(8)), oracle.human_link_points(scene, q)
    assert abs(np.linalg.norm(lp[0] - fr[4, 9:]) - 0.375) < 1e-9      # hand 0.19 below the elbow + offset 0.185
    assert abs(np.linalg.norm(lp2[0] - fr[4, 9:]) - 0.375) < 1e-9 and np.linalg.norm(lp2[0] - lp[0]) > 0.3
    assert np.allclose(lp2[1], lp[1])


def test_braking_target_brings_a_joint_to_rest(scene):
    """The braking accelerations of the nested env end with velocity and acceleration at zero, inside the limits."""
    rng = np.random.default_rng(0)
    h = scene.struct.human
    for _ in range(50):
        q = rng.uniform(0.6 * scene.human_pos_lo + 0.4 * scene.human_pos_hi, 0.4 * scene.human_pos_lo + 0.6 * scene.human_pos_hi)
        v = rng.uniform(-1, 1, 8) * scene.human_vel_max * 0.7
        a = rng.uniform(-1, 1, 8) * 3.0
        lo, hi, code = oracle.human_safe_range(scene, q, v, a)
        if code.any():
            continue
        at = rng.uniform(lo, hi)
        # a pose far from everything would be needed for "no collision"; here only the joint-space part is looked at
        _, acc, poses, coll = oracle.human_check_braking(scene, q, v, a, at)
        if coll != 0:
            continue
        assert 0 < len(acc) <= 21
        # integrate: (q, v, a) -> at -> acc[0] -> ... ends at rest
        qq, vv, aa = q.copy(), v.copy(), a.copy()
        for a1 in [at] + list(acc):
            qq = qq + vv * 0.1 + (aa / 3 + a1 / 6) * 0.01
            vv = vv + (aa + a1) * 0.05
            aa = a1
            assert (np.abs(vv) <= scene.human_vel_max * (1 + 1e-9)).all()
            assert (qq >= scene.human_pos_lo - 1e-9).all() and (qq <= scene.human_pos_hi + 1e-9).all()
        # after the last stored acceleration the next braking step finds the arm at rest
        assert (np.abs(vv) < 0.5).all()


def _start(scene, n, rng):
    hq = []
    while len(hq) < n:
        c = rng.uniform(scene.human_pos_lo, scene.human_pos_hi)
        if not oracle.human_pose_collides(scene, c):
            hq.append(c)
    hq = np.array(hq)
    lp = np.array([oracle.human_link_points(scene, hq[e]) for e in range(n)])
    arm = rng.integers(0, 2, n)
    ft = lp[np.arange(n), arm] + rng.uniform(-0.25, 0.25, (n, 3))
    return hq, ft, arm


def test_human_rollout_invariants(scene):
    n, steps = 12, 30
    rng = np.random.default_rng(1)
    env = oracle.OracleEnvs(scene, n)
    q = rng.uniform(0.3 * np.array(scene.pos_lo), 0.3 * np.array(scene.pos_hi), (n, 7))
    env.set_state(q, np.zeros((n, 7)), np.zeros((n, 7)), np.zeros((n, 16)))
    hq, ft, arm = _start(scene, n, rng)
    env.set_human_state(hq, np.zeros((n, 8)), np.zeros((n, 8)), ft, arm)
    assert env.obs.shape == (n, 45) and np.array_equal(env.obs[:, 21:], env.hobs[:, :24])
    assert (env.hobs[np.arange(n), 36 + arm] == 1).all() and (env.hobs[np.arange(n), 37 - arm] == 0).all()
    braked = 0
    for s in range(steps):
        a = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        ha = rng.uniform(-1, 1, (n, 8)).astype(np.float32)
        nt = rng.uniform([0, -0.8, 0.075], [0.6, 0.8, 0.75], (n, 3))
        env.step_human(a, ha, nt)
        braked += int(env.hinfo[:, 0].sum())
        hk = env.hkin
        assert (hk[:, 0:8] >= scene.human_pos_lo - 1e-9).all() and (hk[:, 0:8] <= scene.human_pos_hi + 1e-9).all()
        assert (np.abs(hk[:, 8:16]) <= scene.human_vel_max * (1 + 1e-9)).all()
        assert (np.abs(hk[:, 16:24]) <= scene.human_acc_max * (1 + 1e-9)).all()
        assert (env.hinfo[:, 2] >= 0).all(), "braking timeout"
        assert np.array_equal(env.obs[:, 21:], env.hobs[:, :24])           # Human.kinematic_observation
        active = env.hstate[:, [abi.TP_ACTIVE, 12 + abi.TP_ACTIVE]]
        assert (active.sum(1) == 1).all()                                  # alternating target points: one arm at a time
        assert (np.abs(env.hobs) <= 1).all()
    assert 0 < braked < n * steps                                          # the braking method intervenes, not always


def test_human_contact_terminates_the_episode(scene):
    """A robot pose reaching into the human's arm: moving-obstacle collision in the first step (ctlp.py:3246-3249)."""
    rng = np.random.default_rng(2)
    env = oracle.OracleEnvs(scene, 1)
    hq = np.array([[0.8, -0.2, 0.0, -1.2, -0.8, -0.2, 0.0, -1.2]])
    lp = oracle.human_link_points(scene, hq[0])
    # search a robot pose whose link 7 comes close to the human's right hand point
    best, bq = 1e9, None
    for _ in range(4000):
        q = rng.uniform(scene.pos_lo, scene.pos_hi)
        p = oracle.target_link_point(scene, q)
        d = np.linalg.norm(p - lp[0])
        if d < best:
            best, bq = d, q
    env.set_state(bq[None], np.zeros((1, 7)), np.zeros((1, 7)), np.zeros((1, 16)))
    env.set_human_state(hq, np.zeros((1, 8)), np.zeros((1, 8)), lp[0][None] + 0.3, [0])
    ds, dse, dm = None, None, None
    env.step_human(np.zeros((1, 7), dtype=np.float32), np.zeros((1, 8), dtype=np.float32), None)
    assert env.info[0, abi.INFO["d_moving"]] < 0.2


def test_oracle_reproduces_human_golden_vectors(scene):
    """tests/golden/human.npz (make_golden.py record_human): regression vectors of the oracle for BASELINE.json configs[2]."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "human.npz"))
    n = g["q"].shape[0]
    env = oracle.OracleEnvs(scene, n)
    env.set_state(g["q"], g["v"], g["a"], np.zeros((n, 16)))
    env.set_human_state(g["hq"], g["hv"], g["ha"], g["first_target"], g["arm"])
    assert np.array_equal(env.kin, g["kin0"]) and np.array_equal(env.hkin, g["hkin0"])
    assert np.array_equal(env.obs, g["obs0"]) and np.array_equal(env.hobs, g["hobs0"])
    assert np.array_equal(env.hstate, g["hstate0"], equal_nan=True) and np.array_equal(env.hbrake, g["hbrake0"])
    for s in range(g["actions"].shape[0]):
        env.step_human(g["actions"][s], g["hactions"][s], g["next_targets"][s])
        for key, arr in (("kin", env.kin), ("hkin", env.hkin), ("hbrake", env.hbrake), ("obs", env.obs), ("hobs", env.hobs),
                         ("reward", env.reward), ("done", env.done), ("term", env.term), ("hinfo", env.hinfo)):
            assert np.array_equal(arr, g["out_" + key][s]), (key, s)
        assert np.array_equal(env.hstate, g["out_hstate"][s], equal_nan=True)
    assert (g["out_hinfo"][:, :, 0] != 0).any() and (g["out_done"] != 0).any()   # the vectors hold braking steps and terminations


def test_brake_pair_distances_and_check_margin(scene):
    """The pair-distance hook agrees with the collision predicate of the braking check, and the check's margin is the
    distance of its deciding pose from the safety distance (a pose at rest: every visited pose is the start pose)."""
    rng = np.random.default_rng(3)
    h = scene.struct.human
    seen = set()
    for _ in range(300):
        hq = rng.uniform(scene.human_pos_lo, scene.human_pos_hi)
        d = oracle.human_brake_pair_distances(scene, hq)
        assert d.shape == (h.n_brake_pairs,)
        dmin = d.min()
        assert (dmin < h.brake_safety) == oracle.human_pose_collides(scene, hq)
        seen.add(bool(dmin < h.brake_safety))
        z = np.zeros(8)
        ex, _, poses, coll = oracle.human_check_braking(scene, hq, z, z, z)
        margin = oracle.human_check_braking_margin(scene, hq, z, z, z)
        assert ex == (dmin < h.brake_safety) and poses >= 1 and coll == (1 if ex else 0)
        if abs(dmin - h.brake_safety) < 1e-3:
            assert abs(margin - abs(dmin - h.brake_safety)) < 1e-12
        else:
            assert margin >= 1e-3 - 1e-12
    assert seen == {True, False}
