"""Constants of the distance planning (csrc/smenv.cu plan_bounds), exported on the host through the C ABI: every bound
distance_plan_kernel culls pairs with must hold for the float32 vertices the kernels use.  The sphere and box lower
bounds, the support-width tables of the separating-axis bound and the centroid upper bound each decide which pairs reach
the GJK kernel; one that is slightly too tight drops the pair that holds a class minimum, and the class reports a larger
distance or the cap -- a collision is missed.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle
from safemotionsrisk_b200 import abi, cabi
from safemotionsrisk_b200.config import ball_backup_config, human_backup_config, space_backup_config, space_task_config
from safemotionsrisk_b200.scene import Scene

SCENES = {"space": space_backup_config, "space_bm": lambda: space_backup_config(ball_machine_mode=True),
          "ball": ball_backup_config, "ball_bm": lambda: ball_backup_config(ball_machine_mode=True),
          "space_task_bm": lambda: space_task_config(ball_machine_mode=True), "human": human_backup_config}
RES = 8   # cells per cube-map face edge of the support-width tables (the cell lut_cell picks in axis_lower_bound_d)


@pytest.fixture(scope="module", params=list(SCENES))
def bounds(request):
    try:
        lib = cabi.load()
    except Exception as e:   # pragma: no cover
        pytest.skip("libsmenv.so not built: {}".format(e))
    scene = Scene(SCENES[request.param]())   # keeps the arrays the struct points into alive
    out = abi.SmPlanBounds()
    cabi.check(lib.smenv_debug_plan_bounds(scene.pointer(), C.byref(out)), "smenv_debug_plan_bounds")
    sc = scene.struct
    v32 = np.ctypeslib.as_array(sc.verts, (sc.n_verts * 3,)).reshape(sc.n_verts, 3).astype(np.float32)
    verts = [v32[sc.shapes[i].vert_off:sc.shapes[i].vert_off + sc.shapes[i].vert_cnt].astype(np.float64)
             for i in range(sc.n_shapes)]
    return request.param, lib, scene, out, verts


def _f3(a):
    return np.array(a[:], dtype=np.float64)


def _pairs(b):
    tab = np.array(b.pair_tab[:b.n_pairs], dtype=np.uint32)
    return (tab & 0xfff).astype(int), ((tab >> 12) & 0xfff).astype(int), ((tab >> 24) & 3).astype(int), (tab >> 31) != 0


def test_pair_table_is_the_oracles_pair_list(bounds):
    """Same pairs, classes and order as oracle.pair_classes; the box flag marks exactly the pairs whose shape B sits in
    frame 0, and frame 0 is the world frame (the oracle's FK frame 0 is the identity)."""
    name, _, scene, b, _ = bounds
    sc = scene.struct
    ia, ib, cls, box = _pairs(b)
    assert np.array_equal(np.stack([cls, ia, ib], 1), oracle.pair_classes(scene))
    assert b.n_pairs_fixed == sc.n_static_pairs + sc.n_self_pairs and b.n_shapes == sc.n_shapes
    assert np.array_equal(box, np.array([sc.shapes[i].frame == 0 for i in ib], dtype=bool))
    assert box.any()
    f0 = oracle.fk(scene, np.random.default_rng(0).uniform(scene.pos_lo, scene.pos_hi))[0]
    assert np.array_equal(f0, [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0])
    want = min(sc.static_cap, max(sc.collision_dist, sc.d_self if sc.w_self != 0 else 0.0))
    assert b.self_query == want
    if name == "space_task_bm":
        assert b.self_query == sc.collision_dist   # the pruning distance is the termination threshold itself


def test_bounding_spheres_boxes_and_centroids(bounds):
    """Every vertex lies within radius of its shape's centre; the box of every shape B of a box-flagged pair holds all
    its vertices; the centroid is the vertex mean, so it lies in the hull (it is not beyond the support point of any
    direction)."""
    _, _, scene, b, verts = bounds
    _, ib, _, box = _pairs(b)
    rng = np.random.default_rng(1)
    dirs = rng.normal(size=(500, 3))
    worst_r = -np.inf
    for s, v in enumerate(verts):
        c = _f3(b.center[s])
        assert np.array_equal(c, np.array(scene.struct.shapes[s].center[:], dtype=np.float32))
        ex = np.linalg.norm(v - c, axis=1).max() - b.radius[s]
        worst_r = max(worst_r, ex)
        assert ex <= 0.0, (s, ex)
        g = _f3(b.centroid[s])
        assert np.abs(g - v.mean(0)).max() <= 1e-6 * (1.0 + np.abs(v).max()), s
        assert ((g @ dirs.T) <= (v @ dirs.T).max(0) + 1e-6).all(), s
    for s in set(ib[box].tolist()):
        v = verts[s]
        assert (v >= _f3(b.bmin[s])).all() and (v <= _f3(b.bmax[s])).all(), s
    print("largest vertex distance beyond the radius: {:.3e} m".format(worst_r))


def test_pair_bounds_subtract_margins_and_radii(bounds):
    """The centroid upper bound subtracts at most the sum of the margins; the sphere / box lower bound at least both
    radii and margins (0 for B's radius where B is bounded by its box)."""
    _, _, scene, b, _ = bounds
    ia, ib, _, box = _pairs(b)
    m = np.array([np.float32(scene.struct.shapes[i].margin) for i in range(b.n_shapes)], dtype=np.float64)
    r = np.array(b.radius[:b.n_shapes], dtype=np.float64)
    rm = np.array(b.pair_rm[:b.n_pairs], dtype=np.float64).reshape(-1, 2)
    assert (rm[:, 0] <= m[ia] + m[ib]).all()
    assert (rm[:, 1] >= r[ia] + np.where(box, 0.0, r[ib]) + m[ia] + m[ib]).all()


def _directions(rng):
    """4000 random float32 unit directions, plus directions on the cell borders and cube-map edges."""
    g = np.linspace(-1, 1, RES + 1)
    u = rng.uniform(-1, 1, 4)
    border = [[1.0, a, w] for a in g for w in u] + [[a, -1.0, w] for a in g for w in u] + [[w, a, 1.0] for a in g for w in u]
    edges = [[1.0, 1.0, w] for w in g] + [[1.0, w, -1.0] for w in g] + [[w, -1.0, 1.0] for w in g]
    d = np.concatenate([rng.normal(size=(4000, 3)), border, edges])
    d = np.concatenate([d, -d])
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def test_support_width_tables_cover_every_direction(bounds):
    """axis_lower_bound_d takes the extent of a hull about its centre along d from the table entry of d's cell.  That
    entry must not be below the true extent max_v (v - c) . d for any direction of the cell, including directions on
    the cell borders, where the float rounding of lut_cell may pick either neighbour."""
    name, lib, _, b, verts = bounds
    d32 = _directions(np.random.default_rng(7))
    cells = np.array([lib.smenv_debug_lut_cell(float(x), float(y), float(z), RES) for x, y, z in d32])
    assert cells.min() >= 0 and cells.max() < abi.SM_PLAN_HWIDTH_CELLS
    d64 = d32.astype(np.float64)
    short = np.array([(((v - _f3(b.center[s])) @ d64.T).max(0) - np.array(b.hwidth[s][:], dtype=np.float64)[cells]).max()
                      for s, v in enumerate(verts)])   # per shape: largest (true width - table entry)
    print("{}: smallest support-width slack {:.3e} m".format(name, -short.max()))
    assert (short <= 0.0).all(), "{} of {} tables fall short of the support width, by up to {:.3e} m (shape {})".format(
        int((short > 0).sum()), len(short), short.max(), int(short.argmax()))
