"""The Human scene's braking-trajectory check (human_brake_traj_kernel -> human_brake_plan_kernel -> gjk_kernel ->
human_advance_kernel) and the robot-versus-human distance query, pose by pose against the CPU oracle.

The culling layers of human_brake_plan_kernel (link-group capsules, the two-sphere test against the table, sphere bounds,
the separating-axis bound) must all be conservative: a bound that is too tight drops a pair, and the human does not brake
where the reference would.  Rollouts rarely bring a pose near the 0.01 m safety distance of a given link-group pair, so
the threshold batches put poses there on purpose: for every link-group pair, poses at rest whose deciding pair belongs
to it, at clearances of +-1e-4, +-1e-3 and +-5e-3 m from the safety distance (bisection along joint-space segments
between a colliding and a free pose, with the oracle's pair distances).  Nothing there is on a float32 knife edge, so the
decisions must match in every env.  The moving batches start near those poses or from the start pool, with velocities,
and include states that run into the 2 s braking timeout; there a decision may differ only where the oracle's smallest
|d_min - safety| over the poses the check visited is below 1e-5 m."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle  # noqa: E402
from safemotionsrisk_b200 import abi, human_backup_config  # noqa: E402
from safemotionsrisk_b200.scene import Scene  # noqa: E402

EDGE = 1e-5                      # float32 geometry on the device: decisions within this of the threshold may differ
CLEARANCES = (1e-4, 1e-3, 5e-3)  # |d_min - safety| of the threshold poses, on both sides
ROOTS = 6                        # crossings per link-group pair, each gives one pose per clearance: 36 envs per pair


def make_env(n):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    return SafeMotionsVecEnv(num_envs=n, config=human_backup_config(), seed=3, auto_reset=False)


def _group_of_pair(scene):
    """Link-group pair (frame of A, frame of B) of every pair of the check, as an index into the sorted list of them."""
    sc, h = scene.struct, scene.struct.human
    keys = [(sc.shapes[h.brake_pairs[i][0]].frame, sc.shapes[h.brake_pairs[i][1]].frame) for i in range(h.n_brake_pairs)]
    groups = sorted(set(keys))
    return groups, np.array([groups.index(k) for k in keys])


def _clearance(scene, gid, hq):
    """(d_min - safety, link-group pair of the deciding pair, smallest clearance of the other link-group pairs)."""
    d = oracle.human_brake_pair_distances(scene, hq) - scene.struct.human.brake_safety
    i = int(np.argmin(d))
    other = d[gid != gid[i]]
    return d[i], int(gid[i]), float(other.min()) if other.size else np.inf


def _bisect(f, t_pos, t_neg, target, iters=48):
    """t on [t_pos, t_neg] with f(t) close to target, f(t_pos) > target > f(t_neg)."""
    for _ in range(iters):
        t = 0.5 * (t_pos + t_neg)
        if f(t) > target:
            t_pos = t
        else:
            t_neg = t
        if abs(t_pos - t_neg) < 1e-12:
            break
    return t_pos if target > 0 else t_neg   # stay on the side of the threshold the target is on


@pytest.fixture(scope="module")
def threshold_poses():
    """Poses at rest on both sides of the safety distance, per link-group pair: (hq [N, 8], group [N], clearance [N])."""
    scene = Scene(human_backup_config())
    groups, gid = _group_of_pair(scene)
    lo, hi = np.array(scene.human_pos_lo), np.array(scene.human_pos_hi)
    rng = np.random.default_rng(20)
    colliding = {g: [] for g in range(len(groups))}
    free = []
    for _ in range(4000):   # colliding poses whose deciding pair is in each link-group pair, and free poses
        q = rng.uniform(lo, hi)
        c, g, _ = _clearance(scene, gid, q)
        if c < -2 * CLEARANCES[-1] and len(colliding[g]) < 4 * ROOTS:
            colliding[g].append(q)
        elif c > 4 * CLEARANCES[-1] and len(free) < 64:
            free.append(q)
    safety = scene.struct.human.brake_safety
    for g in range(len(groups)):   # rare link-group pairs (an upper arm against the other arm): random descent
        for _ in range(200):
            if len(colliding[g]) >= 8 * ROOTS:
                break
            q = rng.uniform(lo, hi)
            dg = (oracle.human_brake_pair_distances(scene, q) - safety)[gid == g].min()
            for _ in range(300):
                q2 = np.clip(q + rng.normal(0, 0.08, 8), lo, hi)
                d2 = (oracle.human_brake_pair_distances(scene, q2) - safety)[gid == g].min()
                if d2 < dg:
                    q, dg = q2, d2
                if dg < -2 * CLEARANCES[-1]:
                    break
            c, gd, _ = _clearance(scene, gid, q)
            if gd == g and c < -2 * CLEARANCES[-1]:
                colliding[g].append(q)
    hq, grp, clr = [], [], []
    for g in range(len(groups)):
        assert len(colliding[g]) >= ROOTS, "no colliding poses found for link-group pair {}".format(groups[g])
        roots = 0
        for qc in colliding[g]:
            if roots == ROOTS:
                break
            # the free poses nearest in joint space first: their segments meet other link-group pairs less often
            for qf in sorted(free, key=lambda x: np.abs(x - qc).sum())[:8]:
                f = lambda t: _clearance(scene, gid, qf + t * (qc - qf))[0]
                t0 = _bisect(f, 0.0, 1.0, 0.0)
                if _clearance(scene, gid, qf + t0 * (qc - qf))[1] == g:
                    break
            else:
                continue   # every segment meets another link-group pair first
            landed = []
            for c in CLEARANCES:
                for target in (c, -c):
                    t = _bisect(f, 0.0, 1.0, target) if target > 0 else _bisect(f, t0, 1.0, target)
                    q = qf + t * (qc - qf)
                    cl, gd, other = _clearance(scene, gid, q)
                    if gd == g and abs(cl - target) < 0.1 * c and other > cl + EDGE:
                        landed.append((q, cl))
            if len(landed) == 2 * len(CLEARANCES):
                roots += 1
                for q, cl in landed:
                    hq.append(q); grp.append(g); clr.append(cl)
    return scene, groups, np.array(hq), np.array(grp), np.array(clr)


def _robot_and_targets(env, n, rng):
    start, _ = env.pools()
    _, htarget = env.human_pools()
    rows = np.arange(n) % start.shape[0]
    q, v, a, ob = start[rows, 0:7], start[rows, 8:15], start[rows, 16:23], start[rows, 32:48]
    arm = rng.integers(0, 2, n)
    ft = htarget[arm, rng.integers(0, htarget.shape[1], n), :3]
    return q, v, a, ob, ft, arm


def _action_at_rest(scene, hq, hv, ha):
    """Human action that maps to an end acceleration of 0 (the safe range need not be symmetric near a limit)."""
    u = np.zeros((len(hq), 8))
    for e in range(len(hq)):
        lo, hi, _ = oracle.human_safe_range(scene, hq[e], hv[e], ha[e])
        u[e] = np.where(hi > lo, 2.0 * (0.0 - lo) / np.where(hi > lo, hi - lo, 1.0) - 1.0, 0.0)
    return np.clip(u, -1, 1).astype(np.float32)


def _one_step(hq, hv, ha, hact, seed):
    """One step of the Human scene on the device and in the oracle from the same injected state."""
    n = len(hq)
    env = make_env(n)
    env.set_human_actions_external(True)
    rng = np.random.default_rng(seed)
    q, v, a, ob, ft, arm = _robot_and_targets(env, n, rng)
    orc = oracle.OracleEnvs(env.scene, n)
    for side in (env, orc):
        side.set_state(q, v, a, ob)
        side.set_human_state(hq, hv, ha, ft, arm)
    torch.cuda.synchronize()
    assert np.array_equal(env.hkin.cpu().numpy(), orc.hkin)
    assert np.array_equal(env.hstate.cpu().numpy()[:, abi.HS_BRAKE_COUNT], orc.hstate[:, abi.HS_BRAKE_COUNT])
    act = np.zeros((n, 7), dtype=np.float32)
    env.hactions.copy_(torch.from_numpy(hact))
    env.step(act)
    torch.cuda.synchronize()
    hs = env.hstate.cpu().numpy()
    act_arm = (hs[:, 12 + abi.TP_ACTIVE] != 0).astype(int)
    nt = np.stack([hs[np.arange(n), 12 * act_arm + abi.TP_POS + i] for i in range(3)], 1)
    orc.step_human(act, hact, nt)
    dev = dict(hs=hs, hkin=env.hkin.cpu().numpy(), hbrake=env.hbrake.cpu().numpy().reshape(n, -1, 8))
    env.close()
    return dev, orc


def _nested_env_equal(dev, orc, envs):
    """Braking decision, stored braking trajectory and joint state of the nested env, exactly."""
    hs = dev["hs"]
    assert np.array_equal(hs[envs, abi.HS_BRAKED], orc.hstate[envs, abi.HS_BRAKED]), "braking decision"
    assert np.array_equal(hs[envs, abi.HS_BRAKE_COUNT], orc.hstate[envs, abi.HS_BRAKE_COUNT]), "HS_BRAKE_COUNT"
    hb_ref = orc.hbrake.reshape(len(hs), -1, 8)
    for e in envs:
        k = int(hs[e, abi.HS_BRAKE_COUNT])
        assert np.array_equal(dev["hbrake"][e, :k], hb_ref[e, :k]), "stored braking trajectory, env {}".format(e)
    assert np.array_equal(dev["hkin"][envs], orc.hkin[envs]), "human joint state"


def test_braking_decision_at_the_threshold_of_every_link_group_pair(threshold_poses):
    scene, groups, hq, grp, clr = threshold_poses
    per_group = np.bincount(grp, minlength=len(groups))
    print("threshold envs per link-group pair:", dict(zip(groups, per_group.tolist())))
    assert (per_group >= 32).all(), dict(zip(groups, per_group.tolist()))
    table_arms = {fa for (fa, fb) in groups if fb == 0}   # world-frame side B: the table
    assert table_arms == {104, 108}, groups                # forearm + hand of both arms against the table
    n = len(hq)
    zero = np.zeros((n, 8))
    hact = _action_at_rest(scene, hq, zero, zero)
    dev, orc = _one_step(hq, zero, zero, hact, seed=5)
    # the action maps to (nearly) zero acceleration: the check visits the start pose within rounding, and none of these
    # envs is on a knife edge
    assert (orc.hmargin >= EDGE).all(), "knife-edge envs in the threshold batch: {}".format(int((orc.hmargin < EDGE).sum()))
    assert np.array_equal(orc.hinfo[:, 0] != 0, clr < 0), "the oracle brakes exactly below the safety distance"
    _nested_env_equal(dev, orc, np.arange(n))
    for g in range(len(groups)):   # both decisions occur in every link-group pair
        sel = grp == g
        assert (dev["hs"][sel, abi.HS_BRAKED] != 0).any() and (dev["hs"][sel, abi.HS_BRAKED] == 0).any()


def test_braking_decision_of_moving_states(threshold_poses):
    """Moving states near the threshold poses, start-pool states drawn towards them, and states with one joint at five
    times its velocity limit (the only states that run into the 2 s braking timeout: within the limits the human stops
    in well under a second)."""
    scene, groups, hq0, grp, clr = threshold_poses
    rng = np.random.default_rng(9)
    lo, hi = np.array(scene.human_pos_lo), np.array(scene.human_pos_hi)
    V, A = np.array(scene.human_vel_max), np.array(scene.human_acc_max)
    m = len(hq0)
    # near the threshold poses, moving
    hq_a = hq0
    hv_a = rng.uniform(-0.4, 0.4, (m, 8)) * V
    ha_a = rng.uniform(-0.4, 0.4, (m, 8)) * A
    # start-pool states pulled halfway towards a threshold pose
    env = make_env(8)
    hstart, _ = env.human_pools()
    env.close()
    rows = rng.integers(0, hstart.shape[0], m)
    hq_b = np.clip(0.5 * (hstart[rows, 0:8] + hq0[rng.permutation(m)]), lo, hi)
    hv_b, ha_b = hstart[rows, 8:16], hstart[rows, 16:24]
    # one joint far beyond its velocity limit: braking takes longer than the timeout
    k = 96
    hq_c = np.clip(0.5 * (lo + hi) + rng.uniform(-0.3, 0.3, (k, 8)), lo, hi)
    hv_c, ha_c = np.zeros((k, 8)), np.zeros((k, 8))
    hv_c[np.arange(k), rng.integers(0, 8, k)] = 5.0 * V[0] * rng.choice([-1.0, 1.0], k)
    hq, hv, ha = (np.concatenate(x) for x in ((hq_a, hq_b, hq_c), (hv_a, hv_b, hv_c), (ha_a, ha_b, ha_c)))
    hact = rng.uniform(-1, 1, (len(hq), 8)).astype(np.float32)
    dev, orc = _one_step(hq, hv, ha, hact, seed=6)
    clear = orc.hmargin >= EDGE
    flips = (dev["hs"][:, abi.HS_BRAKED] != 0) != (orc.hinfo[:, 0] != 0)
    print("moving batches: {} envs, {} knife edges excluded, {} braked, {} timeouts, {} decisions differ".format(
        len(hq), int((~clear).sum()), int((orc.hinfo[:, 0] != 0).sum()), int((orc.hinfo[:, 2] == -1).sum()), int(flips.sum())))
    assert not (flips & clear).any(), "braking decisions differ away from a knife edge: envs {}".format(np.where(flips & clear)[0])
    assert (~clear).sum() <= len(hq) // 50, "too many knife edges: {}".format(int((~clear).sum()))
    _nested_env_equal(dev, orc, np.where(clear)[0])
    assert (orc.hinfo[:, 2] == -1).sum() >= 10, "the batch holds braking timeouts"
    braked = orc.hinfo[:, 0] != 0
    assert 0.1 < braked[:2 * m].mean() < 0.9, "near the threshold poses both decisions occur"


def test_robot_human_distances_match_oracle():
    """smenv_distances with the human's joint angles against the oracle's smo_distances_h.  From random robot and human
    poses the batch keeps every touching one (below 1 mm), every one within 5 cm, and fills up with the rest, most of
    which lie below the 0.6 m query."""
    n = 256
    env = make_env(n)
    sc = env.scene
    rng = np.random.default_rng(4)
    ob = np.zeros(16)
    q = rng.uniform(sc.pos_lo, sc.pos_hi, (4000, 7))
    hq = rng.uniform(sc.human_pos_lo, sc.human_pos_hi, (4000, 8))
    d = np.array([oracle.distances_h(sc, q[i], ob, hq[i]) for i in range(len(q))])
    close = np.where(d[:, 2] < 0.05)[0][:n // 4]
    rest = np.setdiff1d(np.arange(len(q)), close)[:n - len(close)]
    pick = np.concatenate([close, rest])
    kin, hkin = np.zeros((n, 32)), np.zeros((n, 32))
    kin[:, 0:7], hkin[:, 0:8] = q[pick], hq[pick]
    ref = d[pick].copy()
    ref[(ref[:, 1] > 0.05) & (ref[:, 1] <= 0.102), 1] = 0.102   # reporting rule of the self class (test_gpu_parity.reported)
    ds, dse, dm = (x.cpu().numpy() for x in env.distances(kin, np.zeros((n, 16)), hkin))
    clamp = lambda x: np.where(x < 1e-3, 0.0, x)    # below 1 mm everything counts as collision (rewards.py:115)
    for dev, col in ((ds, 0), (dse, 1), (dm, 2)):
        assert np.abs(clamp(dev) - clamp(ref[:, col])).max() < 1e-4, col
    print("robot-human distances: {} below 0.6 m, {} below 5 cm, {} below 1 mm".format(
        int((ref[:, 2] < 0.6).sum()), int((ref[:, 2] < 0.05).sum()), int((ref[:, 2] < 1e-3).sum())))
    assert (ref[:, 2] < 0.6).sum() >= n // 2 and (ref[:, 2] < 1e-3).sum() >= 16
    assert ((ref[:, 2] >= 1e-3) & (ref[:, 2] < 0.05)).sum() >= 16   # the near range above the clamp as well
    env.close()
