"""Bounding volumes of the human's braking-trajectory check (csrc/smenv.cu human_brake_bounds), exported on the host
through the C ABI: every culling layer of human_brake_plan_kernel must contain the shapes it stands for.  A volume that
misses part of a shape lets the kernel drop a pair that the oracle finds closer than the safety distance, and the human
does not brake where the reference would.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

from safemotionsrisk_b200 import abi, cabi
from safemotionsrisk_b200.config import human_backup_config
from safemotionsrisk_b200.scene import Scene

ARM_FRAMES = (3, 4, 7, 8)   # human frames of upper arm / forearm + hand of both arms, the order of hf_*
TOL = 1e-6                  # float32 rounding of the exported volumes


@pytest.fixture(scope="module")
def bounds():
    try:
        lib = cabi.load()
    except Exception as e:   # pragma: no cover
        pytest.skip("libsmenv.so not built: {}".format(e))
    scene = Scene(human_backup_config())   # keeps the arrays the struct points into alive
    out = abi.SmHumanBounds()
    cabi.check(lib.smenv_debug_human_bounds(scene.pointer(), C.byref(out)), "smenv_debug_human_bounds")
    return scene, out


def _shape(scene, i):
    """(core vertices [n, 3] in frame coordinates, margin, frame) of shape i."""
    sc = scene.struct
    verts = np.ctypeslib.as_array(sc.verts, (sc.n_verts * 3,)).reshape(sc.n_verts, 3)
    sh = sc.shapes[i]
    return np.array(verts[sh.vert_off:sh.vert_off + sh.vert_cnt], dtype=np.float64), sh.margin, sh.frame


def _seg(a, k):
    s = np.array(a[k], dtype=np.float64)
    return s[:3], s[3:]


def _segment_distance(p, a, b):
    d = b - a
    t = np.clip((p - a) @ d / max(d @ d, 1e-30), 0.0, 1.0)
    return np.linalg.norm(p - (a + t[:, None] * d), axis=1)


def _box_excess(p, margin, lo, hi):
    """How far the ball of radius margin around each vertex reaches outside the box (<= 0: inside)."""
    return np.maximum(np.asarray(lo, dtype=np.float64) - (p - margin), (p + margin) - np.asarray(hi, dtype=np.float64)).max(1)


def test_group_pairs_are_the_pair_list(bounds):
    """The link-group pairs list every pair of the check exactly once, with each side on the frame the kernel uses."""
    scene, b = bounds
    h = scene.struct.human
    listed = set()
    for g in range(b.n_gp):
        fa, fb = b.gp_fa[g], b.gp_fb[g]
        assert fa in ARM_FRAMES and (fb in ARM_FRAMES or fb in (0, -1))
        for ia in range(b.gp_a0[g], b.gp_a0[g] + b.gp_na[g]):
            assert _shape(scene, ia)[2] == 100 + fa
            for ib in range(b.gp_b0[g], b.gp_b0[g] + b.gp_nb[g]):
                assert _shape(scene, ib)[2] == (100 + fb if fb >= 0 else 0)
                assert (ia, ib) not in listed
                listed.add((ia, ib))
    assert listed == {(h.brake_pairs[i][0], h.brake_pairs[i][1]) for i in range(h.n_brake_pairs)}
    # the table against forearm + hand of both arms, an arm against the other, the arms against the trunk
    table = {b.gp_fa[g] for g in range(b.n_gp) if b.gp_fb[g] == -1}
    assert table == {4, 8}, table
    assert any(b.gp_fb[g] in ARM_FRAMES for g in range(b.n_gp)) and any(b.gp_fb[g] == 0 for g in range(b.n_gp))


def test_arm_frame_capsules_contain_their_shapes(bounds):
    scene, b = bounds
    h = scene.struct.human
    for fi, f in enumerate(ARM_FRAMES):
        on_frame = [h.shape_off + q for q in range(h.n_arm_shapes) if _shape(scene, h.shape_off + q)[2] == 100 + f]
        assert on_frame and list(range(b.hf_s0[fi], b.hf_s0[fi] + b.hf_sn[fi])) == on_frame
        a, c = _seg(b.hf_seg, fi)
        worst = max((_segment_distance(v, a, c) + m).max() for v, m, _ in (_shape(scene, i) for i in on_frame))
        assert worst <= b.hf_rad[fi] + TOL, (f, worst - b.hf_rad[fi])


def test_side_b_volumes_contain_their_shapes(bounds):
    """Trunk side: the capsule gp_sb / gp_srb (frame 0); table side: the box gp_bmin / gp_bmax (world frame); both sides:
    the bounding spheres gp_ca / gp_ra and gp_cb / gp_rb."""
    scene, b = bounds
    for g in range(b.n_gp):
        side_a = [_shape(scene, i) for i in range(b.gp_a0[g], b.gp_a0[g] + b.gp_na[g])]
        side_b = [_shape(scene, i) for i in range(b.gp_b0[g], b.gp_b0[g] + b.gp_nb[g])]
        for shapes, c, r in ((side_a, b.gp_ca[g], b.gp_ra[g]), (side_b, b.gp_cb[g], b.gp_rb[g])):
            worst = max((np.linalg.norm(v - np.array(c[:]), axis=1) + m).max() for v, m, _ in shapes)
            assert worst <= r + TOL, (g, worst - r)
        if b.gp_fb[g] == 0:
            a, c = _seg(b.gp_sb, g)
            worst = max((_segment_distance(v, a, c) + m).max() for v, m, _ in side_b)
            assert worst <= b.gp_srb[g] + TOL, (g, worst - b.gp_srb[g])
        elif b.gp_fb[g] == -1:
            worst = max(_box_excess(v, m, b.gp_bmin[g], b.gp_bmax[g]).max() for v, m, _ in side_b)
            assert worst <= TOL, (g, worst)


def test_table_test_covers_the_arm(bounds):
    """Against the table the kernel tests two spheres at 1/4 and 3/4 of the arm frame's capsule segment instead of the
    capsule.  Every vertex of the frame's shapes, with its margin, and the tips of the capsule's end caps must lie inside
    one of them: the capsule's segment is pulled in by its radius, so vertices do lie in the caps."""
    scene, b = bounds
    for g in range(b.n_gp):
        if b.gp_fb[g] != -1:
            continue
        fi = ARM_FRAMES.index(b.gp_fa[g])
        a, c = _seg(b.hf_seg, fi)
        centres = (a + 0.25 * (c - a), a + 0.75 * (c - a))
        R = b.hf_cover_rad[fi]
        worst = 0.0
        for i in range(b.hf_s0[fi], b.hf_s0[fi] + b.hf_sn[fi]):
            v, m, _ = _shape(scene, i)
            d = np.minimum(np.linalg.norm(v - centres[0], axis=1), np.linalg.norm(v - centres[1], axis=1)) + m
            worst = max(worst, d.max() - R)
        assert worst <= TOL, "frame {}: a vertex lies {:.4f} m outside the spheres of the table test".format(
            100 + ARM_FRAMES[fi], worst)
        u = (c - a) / np.linalg.norm(c - a)
        for tip in (a - b.hf_rad[fi] * u, c + b.hf_rad[fi] * u):
            assert min(np.linalg.norm(tip - x) for x in centres) <= R + TOL
