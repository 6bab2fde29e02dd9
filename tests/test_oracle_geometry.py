"""Oracle FK and GJK against independent computations (closed forms, brute-force QP)."""
import numpy as np
import pytest
from scipy.optimize import minimize

from oracle import oracle
from safemotionsrisk_b200.config import ball_backup_config, space_backup_config, space_task_config
from safemotionsrisk_b200.scene import Scene

SCENES = {"space": space_backup_config, "space_bm": lambda: space_backup_config(ball_machine_mode=True),
          "ball": ball_backup_config, "ball_bm": lambda: ball_backup_config(ball_machine_mode=True),
          "space_task_bm": lambda: space_task_config(ball_machine_mode=True)}

IDENT = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], dtype=np.float64)


def rand_xf(rng, scale=0.3):
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    if np.linalg.det(q) < 0:
        q[:, 0] *= -1
    return np.concatenate([q.reshape(-1), rng.uniform(-scale, scale, 3)])


def qp_distance(a, b):
    na, nb = len(a), len(b)
    m = np.concatenate([a, -b]).T
    cons = [{"type": "eq", "fun": lambda x: x[:na].sum() - 1,
             "jac": lambda x: np.concatenate([np.ones(na), np.zeros(nb)])},
            {"type": "eq", "fun": lambda x: x[na:].sum() - 1,
             "jac": lambda x: np.concatenate([np.zeros(na), np.ones(nb)])}]
    x0 = np.concatenate([np.ones(na) / na, np.ones(nb) / nb])
    r = minimize(lambda x: ((m @ x) ** 2).sum(), x0, jac=lambda x: 2 * m.T @ (m @ x), bounds=[(0, 1)] * (na + nb),
                 constraints=cons, method="SLSQP", options=dict(maxiter=500, ftol=1e-16))
    return np.sqrt(max(r.fun, 0.0))


def test_fk_zero_pose_matches_urdf_chain(space_scene):
    # robot.urdf:4-231: world -> (-0.2,0,0) adapter -> (0,0,0.02) link0 -> J1 z@0.157 -> J2 @0.183 -> J3 @0.185 ->
    # J4 @0.215 -> J5 @0.4 -> J6 @0 -> J7 @0 ; all rpy = 0 (SURVEY 8a row a7)
    fr = oracle.fk(space_scene, np.zeros(7))
    z = np.cumsum([0.02 + 0.157, 0.183, 0.185, 0.215, 0.4, 0.0, 0.0])
    for j in range(7):
        assert np.allclose(fr[1 + j][9:], [-0.2, 0, z[j]], atol=1e-12)
        assert np.allclose(fr[1 + j][:9], IDENT[:9], atol=1e-12)


def test_fk_single_joint_rotations(space_scene):
    q = np.zeros(7)
    q[0] = 0.7                                   # J1 about +z
    fr = oracle.fk(space_scene, q)
    c, s = np.cos(0.7), np.sin(0.7)
    assert np.allclose(fr[1][:9].reshape(3, 3), [[c, -s, 0], [s, c, 0], [0, 0, 1]])
    q = np.zeros(7)
    q[3] = 0.5                                   # J4 about -y
    fr = oracle.fk(space_scene, q)
    c, s = np.cos(-0.5), np.sin(-0.5)
    assert np.allclose(fr[4][:9].reshape(3, 3), [[c, 0, s], [0, 1, 0], [-s, 0, c]])
    # the elbow bends the forearm: link 5 origin = link4 origin + R_y(-0.5) (0,0,0.4)
    assert np.allclose(fr[5][9:], fr[4][9:] + fr[4][:9].reshape(3, 3) @ [0, 0, 0.4])


def test_fk_is_a_rigid_chain(space_scene):
    rng = np.random.default_rng(0)
    for _ in range(20):
        fr = oracle.fk(space_scene, rng.uniform(space_scene.pos_lo, space_scene.pos_hi))
        for f in fr:
            r = f[:9].reshape(3, 3)
            assert np.allclose(r @ r.T, np.eye(3), atol=1e-12) and abs(np.linalg.det(r) - 1) < 1e-12
        for j, d in enumerate([0.183, 0.185, 0.215, 0.4, 0.0, 0.0]):   # link lengths are pose independent
            assert abs(np.linalg.norm(fr[2 + j][9:] - fr[1 + j][9:]) - d) < 1e-12


def test_gjk_analytic_boxes():
    box = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], dtype=np.float64) * 0.5
    t = IDENT.copy()
    t[9:] = [3.0, 0, 0]
    assert abs(oracle.gjk(box, IDENT, box, t) - 2.0) < 1e-12              # face - face
    t[9:] = [2.0, 2.0, 0]
    assert abs(oracle.gjk(box, IDENT, box, t) - np.sqrt(2.0)) < 1e-12     # edge - edge
    t[9:] = [2.0, 2.0, 2.0]
    assert abs(oracle.gjk(box, IDENT, box, t) - np.sqrt(3.0)) < 1e-12     # vertex - vertex
    t[9:] = [0.9, 0.2, 0.1]
    assert oracle.gjk(box, IDENT, box, t) == 0.0                           # overlapping
    # rotated 45 degrees about z: corner against face
    c = np.cos(np.pi / 4)
    t = np.array([c, -c, 0, c, c, 0, 0, 0, 1, 3.0, 0, 0])
    assert abs(oracle.gjk(box, IDENT, box, t) - (3.0 - 0.5 - np.sqrt(0.5))) < 1e-12


def test_gjk_early_out_contract():
    box = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], dtype=np.float64) * 0.5
    t = IDENT.copy()
    t[9:] = [3.0, 0.3, 0.1]
    exact = oracle.gjk(box, IDENT, box, t)
    d = oracle.gjk(box, IDENT, box, t, upper=1.0)
    assert d >= 1.0 and exact >= 1.0   # contract: some value >= upper once the distance is proven >= upper


def test_gjk_matches_qp_on_scene_hulls(space_bm_scene):
    rng = np.random.default_rng(1)
    shapes = space_bm_scene.shapes
    worst, separated = 0.0, 0
    for _ in range(40):
        ia, ib = rng.integers(0, len(shapes), 2)
        va, vb = shapes[ia]["verts"], shapes[ib]["verts"]
        va = va[rng.choice(len(va), min(len(va), 40), replace=False)]
        vb = vb[rng.choice(len(vb), min(len(vb), 40), replace=False)]
        ta, tb = rand_xf(rng), rand_xf(rng)
        d = oracle.gjk(va, ta, vb, tb)
        wa = va @ ta[:9].reshape(3, 3).T + ta[9:]
        wb = vb @ tb[:9].reshape(3, 3).T + tb[9:]
        worst = max(worst, abs(d - qp_distance(wa, wb)))
        separated += d > 0
    assert worst < 1e-7 and separated > 10


def test_distance_conventions(space_scene):
    """Bullet margins (SURVEY Appendix B.2): distance = core distance - 2 mm, capped at the query distance."""
    q = np.zeros(7)                                 # upright arm: nothing near the table or the planets' far side
    ob = np.zeros(16)
    ob[0] = 300
    ds, dself, dm = oracle.distances(space_scene, q, ob)
    assert ds == space_scene.struct.static_cap and dself == space_scene.struct.static_cap   # Q5: no self pairs
    assert 0 < dm <= 0.602
    ob2 = ob.copy()
    ob2[1] = 1.0                                    # latched contact short-circuits to exactly 0 (Q9)
    assert oracle.distances(space_scene, q, ob2)[2] == 0.0
    # random poses: recompose the static distance in Python from FK frames + pairwise GJK - 2 margins
    rng = np.random.default_rng(3)
    below = 0
    for _ in range(60):
        q = rng.uniform(space_scene.pos_lo, space_scene.pos_hi)
        ds, _, _ = oracle.distances(space_scene, q, ob)
        fr = oracle.fk(space_scene, q)
        best = space_scene.struct.static_cap
        for ia, ib in space_scene.static_pairs:
            a, b = space_scene.shapes[ia], space_scene.shapes[ib]
            d = oracle.gjk(a["verts"], fr[a["frame"]], b["verts"], fr[b["frame"]]) - a["margin"] - b["margin"]
            if d <= space_scene.struct.static_cap:
                best = min(best, d)
        assert abs(ds - best) < 1e-12
        below += ds < space_scene.struct.static_cap
    assert below > 5


def test_table_box_core_is_shrunk_by_the_margin(space_scene):
    table = [s for s in space_scene.shapes if s["frame"] == 0 and s["cnt"] == 8][-1]
    v = table["verts"]
    assert np.allclose(v.max(0), [0.6 - 0.001, 0.8 - 0.001, -0.001]) and np.allclose(v.min(0), [-0.599, -0.799, -0.199])


@pytest.mark.parametrize("name", ["space", "space_bm", "ball", "ball_bm", "space_task_bm"])
def test_pair_distances_rebuild_the_class_distances(name):
    """oracle.pair_distances lists every pair of the three distance classes (oracle.pair_classes order, the order of the
    device's pair table); with the class rules of oracle.distances applied to it (cap and query filters, inactive ball,
    latched contact) its class minima are the oracle's distances, exactly."""
    scene = Scene(SCENES[name]())
    sc = scene.struct
    cls = oracle.pair_classes(scene)
    assert [int((cls[:, 0] == c).sum()) for c in range(3)] == [
        sc.n_static_pairs, sc.n_self_pairs, sc.n_mov_reward * sum(sc.obst_shape_cnt[o] for o in range(sc.n_obstacles))]
    cap, query = sc.static_cap, sc.moving_query
    rng = np.random.default_rng(11)
    hits = np.zeros(3, dtype=int)
    for _ in range(300):
        q = rng.uniform(scene.pos_lo, scene.pos_hi)
        ob = np.zeros(16)
        if name.startswith("ball"):
            ob[2:5] = rng.uniform([-0.8, -0.8, 0.1], [0.6, 0.8, 1.3])
            ob[8:11] = rng.uniform(-1, 1, 3)
            ob[12] = rng.uniform(0, 0.05)
            ob[5:8] = rng.uniform(-1, 1, 3)
            ob[13] = rng.random() < 0.8
        else:
            ob[0] = rng.integers(0, sc.planet_steps)
        ob[1] = rng.random() < 0.1
        d = oracle.pair_distances(scene, q, ob)
        assert d.shape == (len(cls),)
        ref = oracle.distances(scene, q, ob)
        ds = min([cap] + [x for x in d[cls[:, 0] == 0] if x <= cap])
        dse = min([cap] + [x for x in d[cls[:, 0] == 1] if x <= cap])
        inactive = name.startswith("ball") and ob[13] == 0    # an inactive ball is not in the list of obstacles
        dm = min([query + 0.002] + [x for x in d[cls[:, 0] == 2] if x <= query and not inactive])
        if ob[1] != 0 or dm <= 0.0:                           # latched contact, or touching
            dm = 0.0
        assert (ds, dse, dm) == ref
        hits += [ds < cap, dse < cap, 0.0 < dm < query]
    # every class reports pair distances below its cap (the 1 mm moving query of space_task_bm aside)
    assert hits[0] > 5 and (hits[1] > 5 or sc.n_self_pairs == 0) and (hits[2] > 5 or query < 0.01), hits


def test_gjk_does_not_take_a_flat_simplex_for_an_enclosure(space_bm_scene):
    """At this space_bm pose the GJK search between the ball machine (shape 9, frame 7) and shape 6 (frame 5) converges
    at 0.0796 m, and its last support point closes a parallelogram with the simplex.  The tetrahedron is flat to
    rounding, the side tests of its faces see noise, and the oracle used to report the pair as touching (distance 0).
    The same hulls transformed to world coordinates first give the right distance."""
    q = [1.9779949815397064, -1.6819379156182812, -2.2868158860081147, -0.9867392662235596, -1.956367020523305,
         -0.3821141234131943, -2.2938491379058235]
    fr = oracle.fk(space_bm_scene, q)
    a, b = space_bm_scene.shapes[9], space_bm_scene.shapes[6]
    assert (a["frame"], b["frame"]) == (7, 5)
    d = oracle.gjk(a["verts"], fr[7], b["verts"], fr[5])
    world = lambda s, f: s["verts"] @ fr[f][:9].reshape(3, 3).T + fr[f][9:]
    ref = oracle.gjk(world(a, 7), IDENT, world(b, 5), IDENT)
    assert abs(ref - 0.0796) < 1e-4 and abs(d - ref) < 1e-12, (d, ref)
