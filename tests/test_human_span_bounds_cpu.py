"""Inflation table of the span pass of the human's braking-trajectory check (csrc/smenv.cu human_brake_bounds, hf_rho),
exported on the host through the C ABI.  The span pass tests one pose of a run of poses and grows the volumes of arm frame
i by sum_j max |dq_j| hf_rho[i][j]; if some point it reads could move farther, the pass could clear a run in which the
per-pose pass would have found a pair closer than the safety distance.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle
from safemotionsrisk_b200 import abi, cabi
from safemotionsrisk_b200.config import human_backup_config
from safemotionsrisk_b200.scene import Scene

ARM_FRAMES = (3, 4, 7, 8)   # human frames of upper arm / forearm + hand of both arms, the order of hf_*


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


def _frame_points(scene, b, fi):
    """Points of arm frame fi the span pass reads, in frame coordinates: shape centres and the capsule's end points."""
    sc = scene.struct
    pts = [list(sc.shapes[i].center) for i in range(b.hf_s0[fi], b.hf_s0[fi] + b.hf_sn[fi])]
    seg = np.array(b.hf_seg[fi][:], dtype=np.float64)
    return np.array(pts + [seg[:3], seg[3:]], dtype=np.float64)


def _world(scene, hq, f, pts):
    fr = oracle.human_fk(scene, hq)[f]
    return pts @ fr[:9].reshape(3, 3).T + fr[9:]


def test_rho_covers_the_joints_that_move_the_frame(bounds):
    """Joints of the other arm and joints after the frame's own joint do not move it: their entries are 0."""
    _, b = bounds
    for fi, f in enumerate(ARM_FRAMES):
        jf = f - 1
        for j in range(8):
            moves = j // 4 == jf // 4 and j <= jf
            assert (b.hf_rho[fi][j] > 0) == moves, (f, j, b.hf_rho[fi][j])


def test_points_move_at_most_the_inflation(bounds):
    """For random arm poses and random joint offsets from 1e-4 to 0.5 rad, every point of arm frame i moves at most
    sum_j |delta_j| hf_rho[i][j]."""
    scene, b = bounds
    lo, hi = np.array(scene.human_pos_lo), np.array(scene.human_pos_hi)
    rng = np.random.default_rng(12)
    pts = [_frame_points(scene, b, fi) for fi in range(4)]
    rho = np.array([b.hf_rho[fi][:] for fi in range(4)], dtype=np.float64)
    worst = np.zeros(4)
    for _ in range(400):
        q = rng.uniform(lo, hi)
        delta = rng.uniform(-1, 1, 8) * 10.0 ** rng.uniform(-4, np.log10(0.5), 8)
        if rng.random() < 0.3:   # one joint alone: the bound of a single rotation
            delta = np.where(np.arange(8) == rng.integers(0, 8), delta, 0.0)
        for fi, f in enumerate(ARM_FRAMES):
            moved = np.linalg.norm(_world(scene, q + delta, f, pts[fi]) - _world(scene, q, f, pts[fi]), axis=1).max()
            bound = np.abs(delta) @ rho[fi]
            assert moved <= bound * (1 + 1e-9) + 1e-12, (f, moved, bound)
            worst[fi] = max(worst[fi], moved / bound if bound > 0 else 0.0)
    # the table is a chain bound, not a vacuous one: random moves use a fair part of it
    assert (worst > 0.3).all(), worst
