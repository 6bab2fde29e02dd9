"""The span pass of the human's braking-trajectory check (human_brake_plan_kernel<true>) against the CPU oracle at the
threshold, with moving states.

The span pass runs one forward kinematics per run of consecutive poses, at the middle pose, and grows the volumes by the
joint motion inside the run.  It can only go wrong where the pose that decides lies away from the middle of its run and
the motion inside the run is not zero.  So the states here move, and their first pose closer than the safety distance is
not the middle pose of its run: from a free and a colliding pose at rest, the start pose of a moving state is slid along
the joint-space segment between them until the oracle's decision flips (its first colliding pose p*), then placed so
that p* lies at clearances of +-1e-4, +-1e-3 and +-5e-3 m from the safety distance.  Decisions, stored braking
trajectories and joint states of the nested env must match the oracle in every env."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle  # noqa: E402
from safemotionsrisk_b200 import abi, human_backup_config  # noqa: E402
from safemotionsrisk_b200.scene import Scene  # noqa: E402

EDGE = 1e-5                      # float32 geometry on the device: decisions within this of the threshold may differ
CLEARANCES = (1e-4, 1e-3, 5e-3)  # |d_min - safety| of the deciding pose, on both sides
SPAN = 3                         # default run length of the span pass (HBP_SPAN): middle pose = first + 1
ROOTS = 48                       # decision flips kept, each gives one state per clearance and side
BISECT = 26


def _oracle_step(scene, robot, hq, hv, ha, hact):
    """(braked, first colliding pose (1-based, 0 none, -1 timeout), margin, oracle) of one oracle step of the Human scene."""
    q, v, a, ob, ft, arm = (x[:len(hq)] for x in robot)
    orc = oracle.OracleEnvs(scene, len(hq))
    orc.set_state(q, v, a, ob)
    orc.set_human_state(hq, hv, ha, ft, arm)
    orc.step_human(np.zeros((len(hq), 7), dtype=np.float32), hact, ft)
    return orc.hinfo[:, 0] != 0, orc.hinfo[:, 2].copy(), orc.hmargin.copy(), orc


def _signed(braked, margin):
    return np.where(braked, -margin, margin)


def _span_states(scene, robot, rng):
    """Moving states whose deciding pose is off the middle of its run: (hq, hv, ha, hact, target clearance, p*)."""
    h = scene.struct.human
    lo, hi = np.array(scene.human_pos_lo), np.array(scene.human_pos_hi)
    V = np.array(scene.human_vel_max)
    colliding, free = [], []
    while len(colliding) < 4 * ROOTS or len(free) < 64:
        q = rng.uniform(lo, hi)
        c = (oracle.human_brake_pair_distances(scene, q) - h.brake_safety).min()
        if c < -0.01 and len(colliding) < 4 * ROOTS:
            colliding.append(q)
        elif c > 0.03 and len(free) < 64:
            free.append(q)
    qc = np.array(colliding)
    qf = np.array([min(free, key=lambda x: np.abs(x - c).sum()) for c in qc])
    n = len(qc)
    hv = rng.uniform(-0.5, 0.5, (n, 8)) * V
    ha = np.zeros((n, 8))
    hact = rng.uniform(-1, 1, (n, 8)).astype(np.float32)
    at = lambda t, rows: np.clip(qf[rows] + t[:, None] * (qc[rows] - qf[rows]), lo, hi)
    rows = np.arange(n)
    b0 = _oracle_step(scene, robot, at(np.zeros(n), rows), hv, ha, hact)[0]
    b1 = _oracle_step(scene, robot, at(np.ones(n), rows), hv, ha, hact)[0]
    rows = np.where(~b0 & b1)[0]   # free at the free pose, braking at the colliding one
    t_pos, t_neg = np.zeros(len(rows)), np.ones(len(rows))
    for _ in range(BISECT):        # the flip of the decision
        t = 0.5 * (t_pos + t_neg)
        br = _oracle_step(scene, robot, at(t, rows), hv[rows], ha[rows], hact[rows])[0]
        t_pos, t_neg = np.where(br, t_pos, t), np.where(br, t, t_neg)
    br, first, _, _ = _oracle_step(scene, robot, at(t_neg, rows), hv[rows], ha[rows], hact[rows])
    off_middle = br & (first > 0) & ((first - 1) % SPAN != 1)
    rows, t_pos, t_neg, first = rows[off_middle], t_pos[off_middle], t_neg[off_middle], first[off_middle]
    rows, t_pos, t_neg, first = rows[:ROOTS], t_pos[:ROOTS], t_neg[:ROOTS], first[:ROOTS]
    # every target clearance at once: bisection on the signed margin of the decision along the same segment
    targets = np.array([s * c for c in CLEARANCES for s in (1.0, -1.0)])
    R = np.repeat(rows, len(targets))
    T = np.tile(targets, len(rows))
    lo_t, hi_t = np.zeros(len(R)), np.ones(len(R))   # signed(lo_t) > target > signed(hi_t)
    for _ in range(BISECT):
        t = 0.5 * (lo_t + hi_t)
        br, _, mg, _ = _oracle_step(scene, robot, at(t, R), hv[R], ha[R], hact[R])
        above = _signed(br, mg) > T
        lo_t, hi_t = np.where(above, t, lo_t), np.where(above, hi_t, t)
    t = np.where(T > 0, lo_t, hi_t)   # stay on the side of the threshold the target is on
    hq = at(t, R)
    br, fst, mg, _ = _oracle_step(scene, robot, hq, hv[R], ha[R], hact[R])
    p_star = np.where(br, fst, np.repeat(first, len(targets)))
    keep = (np.abs(_signed(br, mg) - T) < 0.1 * np.abs(T)) & (br == (T < 0)) & ((p_star - 1) % SPAN != 1)
    return hq[keep], hv[R][keep], ha[R][keep], hact[R][keep], T[keep], p_star[keep]


def test_span_pass_at_the_threshold_off_the_middle_pose():
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    scene = Scene(human_backup_config())
    rng = np.random.default_rng(31)
    n_max = 4 * ROOTS * 2 * len(CLEARANCES)
    env = SafeMotionsVecEnv(num_envs=n_max, config=human_backup_config(), seed=3, auto_reset=False)
    start, _ = env.pools()
    _, htarget = env.human_pools()
    rows = np.arange(n_max) % start.shape[0]
    arm = rng.integers(0, 2, n_max)
    robot = (start[rows, 0:7], start[rows, 8:15], start[rows, 16:23], start[rows, 32:48],
             htarget[arm, rng.integers(0, htarget.shape[1], n_max), :3], arm)
    env.close()
    hq, hv, ha, hact, target, p_star = _span_states(scene, robot, rng)
    n = len(hq)
    print("span states: {} envs, first colliding pose (1-based) {}".format(n, np.bincount(p_star).nonzero()[0].tolist()))
    for c in CLEARANCES:
        assert (np.isclose(target, c)).sum() >= 12 and (np.isclose(target, -c)).sum() >= 12, c
    # the device step from the same states
    env = SafeMotionsVecEnv(num_envs=n, config=human_backup_config(), seed=3, auto_reset=False)
    env.set_human_actions_external(True)
    q, v, a, ob, ft, arm = (x[:n] for x in robot)
    env.set_state(q, v, a, ob)
    env.set_human_state(hq, hv, ha, ft, arm)
    env.hactions.copy_(torch.from_numpy(hact))
    env.enable_counters(True)
    env.counters(reset=True)
    env.step(np.zeros((n, 7), dtype=np.float32))
    torch.cuda.synchronize()
    cnt = env.counters()
    hs, hkin = env.hstate.cpu().numpy(), env.hkin.cpu().numpy()
    hbrake = env.hbrake.cpu().numpy().reshape(n, -1, 8)
    env.close()
    braked, _, margin, orc = _oracle_step(scene, robot, hq, hv, ha, hact)
    assert (margin >= EDGE).all(), "knife-edge envs: {}".format(int((margin < EDGE).sum()))
    assert np.array_equal(braked, target < 0)
    assert np.array_equal(hs[:, abi.HS_BRAKED] != 0, braked), "braking decisions differ: envs {}".format(
        np.where((hs[:, abi.HS_BRAKED] != 0) != braked)[0])
    assert np.array_equal(hs[:, abi.HS_BRAKE_COUNT], orc.hstate[:, abi.HS_BRAKE_COUNT])
    hb_ref = orc.hbrake.reshape(n, -1, 8)
    for e in range(n):
        k = int(hs[e, abi.HS_BRAKE_COUNT])
        assert np.array_equal(hbrake[e, :k], hb_ref[e, :k]), "stored braking trajectory, env {}".format(e)
    assert np.array_equal(hkin, orc.hkin), "human joint state"
    # both passes ran: every pose of the trajectories in a run, the deciding runs went on to the per-pose pass
    assert cnt["brake_spans"] >= cnt["brake_poses"] / SPAN and 0 < cnt["brake_fine_poses"] <= cnt["brake_poses"], cnt
