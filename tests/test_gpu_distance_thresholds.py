"""The robot's static, self and moving distance classes (distance_plan_kernel -> gjk_kernel -> distances_out_kernel)
pose by pose at their thresholds, against the CPU oracle.

Every culling step of the distance planning (centroid upper bound, sphere and box lower bounds, the separating-axis bound
from the support-width tables, the two-point bound of the moving class, the pruning of self pairs at self_query) and of
the GJK kernel (separating-plane test, pruning between the lanes of one env and class, the iteration cap, atomicMin on a
pre-seeded slot) drops pairs.  A bound that is slightly too tight drops the pair that holds a class minimum: the class
reports a larger distance or its cap, and a collision (distance below collision_dist, 1 mm) is missed.  Random poses
rarely come near a threshold, so the threshold poses put one pair at a time there on purpose: for every static and self
pair, and every (robot shape, obstacle), poses where that pair holds the class minimum, every other pair of the class is
more than 1e-5 m farther away, and the minimum is collision_dist +- {1e-4, 1e-3} or one of the class's own edges +-
{1e-4, 1e-3} (bisection with the oracle's pair distances along segments between a pose below and a pose above).  Then
poses where the pair penetrates: just past the first touch, and 1 cm and 5 cm deeper.  The robot moves in joint space
(at a fixed planet index for the moving class of the Space scenes); in the Ball scenes the ball moves along a line
towards a robot shape instead."""
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle  # noqa: E402
from safemotionsrisk_b200 import abi  # noqa: E402
from safemotionsrisk_b200.config import ball_backup_config, space_backup_config, space_task_config  # noqa: E402
from safemotionsrisk_b200.scene import Scene  # noqa: E402

CONFIGS = {"space": space_backup_config, "space_bm": lambda: space_backup_config(ball_machine_mode=True),
           "ball": ball_backup_config, "ball_bm": lambda: ball_backup_config(ball_machine_mode=True),
           "space_task_bm": lambda: space_task_config(ball_machine_mode=True)}
EDGE = 1e-5                 # float32 geometry on the device: nothing in the threshold batches is this close to a threshold
OFFSETS = (1e-4, 1e-3)      # distance of the class minimum from each threshold, on both sides
DEPTHS = (0.0, 0.01, 0.05)  # penetrating poses: just past the first touch, then this much deeper
BATCH = 2048                # envs per device batch; every pose appears at least twice
CLS = ("static", "self", "moving")


def make_env(name, n):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    return SafeMotionsVecEnv(num_envs=n, config=CONFIGS[name](), seed=3, auto_reset=False, fill_pools=False)


def self_query(sc):
    return min(sc.static_cap, max(sc.collision_dist, sc.d_self if sc.w_self != 0 else 0.0))


def class_edges(sc, c):
    """(thresholds of class c, the largest distance the class reports exactly, the value it reports above that)."""
    if c == 0:
        top, cap = sc.static_cap, sc.static_cap
        edges = [sc.collision_dist, sc.d_static, sc.static_cap]
    elif c == 1:
        top, cap = self_query(sc), sc.static_cap
        edges = [sc.collision_dist, top]
    else:
        top, cap = sc.moving_query, float(np.float32(sc.moving_query) + np.float32(0.002))
        edges = [sc.collision_dist, top]
    return sorted({e for e in edges if e <= top}), top, cap


class Setup:
    def __init__(self, name):
        self.name, self.scene = name, Scene(CONFIGS[name]())
        sc = self.sc = self.scene.struct
        self.cls = oracle.pair_classes(self.scene)
        self.members = {c: np.where(self.cls[:, 0] == c)[0] for c in range(3)}
        self.margin = np.array([sc.shapes[a].margin + sc.shapes[b].margin for _, a, b in self.cls])
        self.ball = name.startswith("ball")

    def ob_far(self, idx=0):
        ob = np.zeros(16)
        ob[0] = idx
        if self.ball:   # an active ball far above the robot: the moving class reports its cap
            ob[2:5], ob[13] = (0.0, 0.0, 5.0), 1.0
        return ob

    def d(self, q, ob):
        return oracle.pair_distances(self.scene, q, ob)


def _targets(sc, c):
    edges, _, _ = class_edges(sc, c)
    return {round(e + s * off, 9) for e in edges for off in OFFSETS for s in (-1, 1)} | {"pen"}


def _land(S, c, group, at, poses, key, want):
    """Poses on the segment at(t), t in [0, 1] (group distance above the targets at 0, lowest at 1), for the targets in
    want: the class-c minimum held by a pair of group at the target distance, every other pair of the class more than
    EDGE farther away; 'pen': penetrating poses.  Appends (q, ob, class, key, target) to poses and returns the targets
    it placed."""
    g = lambda t: S.d(*at(t))
    lo_v, hi_v = g(1.0)[group].min(), g(0.0)[group].min()
    edges, _, _ = class_edges(S.sc, c)
    landed = set()
    for target in sorted(x for x in want if x != "pen" and lo_v < x < hi_v):
        off = min(abs(target - e) for e in edges)
        a, b, tol = 0.0, 1.0, 0.05 * off
        for _ in range(60):
            t = 0.5 * (a + b)
            d = g(t)
            v = d[group].min()
            if abs(v - target) < tol:
                break
            a, b = (t, b) if v > target else (a, t)
        cd = np.sort(d[S.members[c]])
        if abs(v - target) < tol and cd[0] == v and cd[1] > v + EDGE:
            poses.append((at(t)[0], at(t)[1], c, key, target))
            landed.add(target)
    m = S.margin[group].min()
    if "pen" in want and lo_v <= -m + 1e-12:   # the core distance reaches 0: the oracle reports -(sum of the margins)
        a, b = 0.0, 1.0
        for _ in range(44):
            t = 0.5 * (a + b)
            a, b = (t, b) if g(t)[group].min() > -m + 1e-12 else (a, t)
        h = min(1e-3, b)
        slope = (g(b - h)[group].min() + m) / h   # metres of pair distance per unit of t just before the touch
        for depth in DEPTHS:
            t = min(1.0, b + depth / max(slope, 1e-9))
            if g(t)[group].min() <= -m + 1e-12:
                poses.append((at(t)[0], at(t)[1], c, key, "pen"))
                landed.add("pen")
    return landed


def _robot_segments(S, rng, c, n_pool=1500):
    """Threshold poses of class c with the robot moving in joint space: one pose set per static / self pair, per (robot
    shape, planet) for the moving class."""
    sc = S.sc
    q = rng.uniform(S.scene.pos_lo, S.scene.pos_hi, (n_pool, S.scene.n_joints))
    obs = [S.ob_far(int(rng.integers(0, max(sc.planet_steps, 1)))) for _ in range(n_pool)]
    D = np.array([S.d(q[i], obs[i]) for i in range(n_pool)])
    _, top, _ = class_edges(sc, c)
    if c < 2:
        groups = {(int(S.cls[p, 1]), int(S.cls[p, 2])): np.array([p]) for p in S.members[c]}
    else:
        groups = {}
        for p in S.members[2]:
            o = next(o for o in range(sc.n_obstacles) if sc.obst_shape_off[o] <= S.cls[p, 2] < sc.obst_shape_off[o] + sc.obst_shape_cnt[o])
            groups.setdefault((int(S.cls[p, 1]), o), []).append(p)
        groups = {k: np.array(v) for k, v in groups.items()}
    poses = []
    for key, grp in groups.items():
        gv = D[:, grp].min(1)
        want = {x for x in _targets(sc, c) if x == "pen" or x > gv.min()}
        for lo in np.argsort(gv)[:8]:     # the lowest poses of the pool, each with the nearest poses above the targets
            if not want or gv[lo] > top - 1e-3:
                break
            ob = obs[lo]
            tried = 0
            for hi in [i for i in np.argsort(np.abs(q - q[lo]).sum(1)) if gv[i] > top + 5e-3][:24]:
                d_hi = D[hi] if c < 2 else S.d(q[hi], ob)   # the moving class: the planets stay at the low pose's index
                if d_hi[grp].min() > top + 5e-3 and np.sort(d_hi[S.members[c]])[0] > top + 2e-3:
                    at = lambda t, a=q[hi], b=q[lo], ob=ob: (a + t * (b - a), ob)
                    want -= _land(S, c, grp, at, poses, key, want)
                    tried += 1
                    if not want or tried == 3:
                        break
    return poses


def _ball_segments(S, rng):
    """Moving class of the Ball scenes: the robot at a pool pose, the ball along a line from 1 m away to the robot
    shape's centroid."""
    sc = S.sc
    poses = []
    shapes = S.scene.shapes
    for p in S.members[2]:
        r = int(S.cls[p, 1])
        want = _targets(sc, 2)
        for _ in range(16):
            q = rng.uniform(S.scene.pos_lo, S.scene.pos_hi)
            fr = oracle.fk(S.scene, q)[shapes[r]["frame"]]
            centre = fr[:9].reshape(3, 3) @ shapes[r]["verts"].mean(0) + fr[9:]
            u = rng.normal(size=3)
            u /= np.linalg.norm(u)

            def at(t, start=centre + 1.0 * u, end=centre, q=q):
                ob = S.ob_far()
                ob[2:5] = start + t * (end - start)
                return q, ob
            want -= _land(S, 2, np.array([p]), at, poses, (r, 0), want)
            if not want:
                break
    return poses


@functools.lru_cache(maxsize=None)
def threshold_poses(name):
    """(Setup, [(q, ob, class, pair key, target or 'pen')]) of one scene, built once per test session."""
    S = Setup(name)
    rng = np.random.default_rng(30)
    poses = []
    for c in range(3):
        if len(S.members[c]) == 0:
            continue
        poses += _ball_segments(S, rng) if (c == 2 and S.ball) else _robot_segments(S, rng, c)
    return S, poses


def _check_class(S, c, dev, ref, strict):
    """Device values of class c against the oracle's.  strict: the pose was placed at a threshold of this class (no
    knife edge); otherwise values within EDGE of a threshold are exempt from the decision check."""
    edges, top, cap = class_edges(S.sc, c)
    coll = S.sc.collision_dist
    o_cap = S.sc.static_cap if c < 2 else S.sc.moving_query + 0.002   # what the oracle reports where nothing is closer
    above = (ref > top) | (ref == o_cap)
    clamp = lambda x: np.where(x < coll, 0.0, x)   # below 1 mm everything counts as collision (rewards.py:115)
    bad = np.where(above, dev != np.float32(cap), (np.abs(clamp(dev) - clamp(ref)) >= 1e-4) | (dev == np.float32(cap)))
    knife = np.zeros(len(ref), dtype=bool)
    for e in edges + [coll]:
        knife |= (np.abs(ref - e) < EDGE) & (ref != o_cap)
    if strict:
        assert not knife.any()
    else:
        bad &= ~knife
    bad |= ((dev < coll) != (ref < coll)) & ~knife
    return bad


@pytest.mark.parametrize("name", list(CONFIGS))
def test_distance_classes_at_their_thresholds(name):
    S, poses = threshold_poses(name)
    n = len(poses)
    cls = np.array([p[2] for p in poses])
    pen = np.array([isinstance(p[4], str) for p in poses])
    counts = {CLS[c]: (int(((cls == c) & ~pen).sum()), int(((cls == c) & pen).sum()),
                       len({p[3] for p in poses if p[2] == c})) for c in range(3) if len(S.members[c])}
    print("{}: threshold / penetrating poses and pairs (or robot shape, obstacle) per class: {}".format(S.name, counts))
    for c in range(3):
        if len(S.members[c]):
            assert ((cls == c) & ~pen).sum() >= 8 and ((cls == c) & pen).sum() >= 1, (S.name, CLS[c], counts)
    q = np.array([p[0] for p in poses])
    ob = np.array([p[1] for p in poses])
    ref = np.array([oracle.distances(S.scene, q[i], ob[i]) for i in range(n)])
    reps = max(2, -(-BATCH // n))
    order = np.random.default_rng(1).permutation(np.tile(np.arange(n), reps))   # each pose at >= 2 batch positions
    m = len(order)
    env = make_env(S.name, m)
    kin = np.zeros((m, abi.SM_KIN_STRIDE))
    kin[:, :S.scene.n_joints] = q[order]
    env.enable_counters(True)
    env.counters(reset=True)
    dev = np.stack([x.cpu().numpy() for x in env.distances(kin, ob[order])], 1)
    hist = env.counters()["gjk_iteration_histogram"]
    env.close()
    print("{}: {} envs, GJK iterations per pair <= 4, 8, 12, 16, 24, more: {}".format(S.name, m, hist))
    ref_o, cls_o, pen_o = ref[order], cls[order], pen[order]
    for c in range(3):
        target = (cls_o == c) & ~pen_o
        bad = _check_class(S, c, dev[:, c], ref_o[:, c], strict=False)
        strict_bad = np.zeros(m, dtype=bool)
        if target.any():
            strict_bad[target] = _check_class(S, c, dev[target, c], ref_o[target, c], strict=True)
        worst = np.where(bad | strict_bad)[0]
        assert len(worst) == 0, "{} {}: {} envs differ, e.g. device {} oracle {} (pose {})".format(
            S.name, CLS[c], len(worst), dev[worst[:4], c], ref_o[worst[:4], c], order[worst[:4]])
        p = (cls_o == c) & pen_o
        assert (dev[p, c] < S.sc.collision_dist).all(), "{} {}: penetrating poses report {}".format(
            S.name, CLS[c], dev[p & (dev[:, c] >= S.sc.collision_dist), c][:4])
    for i in range(n):   # the same pose reports the same distances wherever it sits in the batch
        rows = np.where(order == i)[0]
        assert (dev[rows] == dev[rows[0]]).all(), i


def _action_at_rest(scene, q):
    """Robot action that maps to a next-knot acceleration of 0 from rest (the safe range need not be symmetric)."""
    z = np.zeros_like(q)
    lo, hi, _ = oracle.safe_range(scene, q, z, z)
    u = np.where(hi > lo, 2.0 * (0.0 - lo) / np.where(hi > lo, hi - lo, 1.0) - 1.0, 0.0)
    return np.clip(u, -1, 1).astype(np.float32)


@pytest.mark.parametrize("name", ["space_bm", "ball_bm", "space_task_bm"])
def test_whole_step_at_static_and_self_thresholds(name):
    """The static and self threshold poses through the whole step, the robot at rest and the action that keeps the knot
    in place: collision flags, termination and reward as in the oracle.  The planets are set S sub-steps before the
    pose's index, so the distance is taken with the planets where the threshold batch had them; poses where a planet
    comes within 5 cm of the robot are left out (the sub-step contact check is not what this tests).  The ball is
    inactive."""
    S, poses = threshold_poses(name)
    sel = [p for p in poses if p[2] < 2]
    q = np.array([p[0] for p in sel])
    ob = np.array([p[1] for p in sel])
    if S.ball:
        ob[:] = 0.0
    else:
        keep = np.array([S.d(q[i], ob[i])[S.members[2]].min() > 0.05 for i in range(len(sel))])
        q, ob = q[keep], ob[keep]
        ob[:, 0] = (ob[:, 0] - S.sc.substeps) % S.sc.planet_steps
    n = len(q)
    assert n >= 16, n
    z = np.zeros_like(q)
    act = _action_at_rest(S.scene, q)
    ft = None
    if S.sc.use_target_points:
        ft = np.array([oracle.target_link_point(S.scene, x) for x in q]) + np.array([0.3, 0.0, 0.0])
    env = make_env(name, n)
    env.set_state(q, z, z, ob, first_target=ft)
    orc = oracle.OracleEnvs(S.scene, n)
    orc.set_state(q, z, z, ob, first_target=ft)
    _, rew, done, info = env.step(act)
    torch.cuda.synchronize()
    o_obs, o_rew, o_done, o_term, o_info = orc.step(act)
    info, rew, done, term = info.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), env.term_reason.cpu().numpy()
    kin = env.kin.cpu().numpy()
    env.close()
    assert np.array_equal(kin, orc.kin)
    assert np.abs(orc.kin[:, :S.scene.n_joints] - q).max() < 1e-6   # the knot stays where the threshold batch put it
    flags = [abi.INFO[k] for k in ("coll_static", "coll_self", "coll_moving")]
    print("{}: {} envs through the step, {} static and {} self collisions".format(
        name, n, int(o_info[:, flags[0]].sum()), int(o_info[:, flags[1]].sum())))
    assert np.array_equal(info[:, flags], o_info[:, flags]), np.where((info[:, flags] != o_info[:, flags]).any(1))[0]
    assert np.array_equal(done, o_done) and np.array_equal(term, o_term)
    assert np.allclose(rew, o_rew, rtol=1e-4, atol=1e-4), np.abs(rew - o_rew).max()
    assert o_info[:, flags[0]].any() and (o_info[:, flags[0]] == 0).any()
