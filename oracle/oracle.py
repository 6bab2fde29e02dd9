"""ctypes front end of the C oracle (oracle/smenv_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs.  The product
package safemotionsrisk_b200/ never imports this module.  PARITY UNPINNED (no klimits / pybullet in this image and no
reference tests or golden vectors exist): see the header of smenv_oracle.c and DESIGN.md.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from safemotionsrisk_b200 import abi

_DIR = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_DIR, "libsmenv_oracle.so")
_lib = None


class SmoStepOut(C.Structure):
    _fields_ = [("reward", C.c_float), ("done", C.c_int32), ("term_reason", C.c_int32),
                ("info", C.c_float * abi.SM_INFO_STRIDE),
                ("range_lo", C.c_double * abi.SM_MAX_JOINTS), ("range_hi", C.c_double * abi.SM_MAX_JOINTS),
                ("a1", C.c_double * abi.SM_MAX_JOINTS),
                ("d_static", C.c_double), ("d_self", C.c_double), ("d_moving", C.c_double)]


def build(force=False):
    src = os.path.join(_DIR, "smenv_oracle.c")
    hdr = os.path.join(os.path.dirname(_DIR), "include", "smenv.h")
    if force or not os.path.exists(_LIB_PATH) or \
            os.path.getmtime(_LIB_PATH) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["make", "-C", _DIR, "-B", "libsmenv_oracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()  # no-op when the library is newer than its sources
        _lib = C.CDLL(_LIB_PATH)
        _lib.smo_gjk_flat.restype = C.c_double
        assert _lib.smo_sizeof_scene() == C.sizeof(abi.SmScene), "SmScene layout mismatch"
        assert _lib.smo_sizeof_stepout() == C.sizeof(SmoStepOut)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def safe_range(scene, q, v, a):
    """(lo, hi, code) of the next-knot acceleration for a batch [n, n_joints] (actions.py:206-211)."""
    L = lib()
    q, v, a = (np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64) for x in (q, v, a))
    n, nj = q.shape
    lo, hi, code = np.zeros((n, nj)), np.zeros((n, nj)), np.zeros((n, nj), dtype=np.int32)
    for i in range(n):
        L.smo_safe_range(scene.pointer(), _p(q[i], C.c_double), _p(v[i], C.c_double), _p(a[i], C.c_double),
                         _p(lo[i], C.c_double), _p(hi[i], C.c_double), _p(code[i], C.c_int32))
    return lo, hi, code


def fk(scene, q):
    """Frames [1 + n_joints, 12] (R row major, t) for one joint vector."""
    out = np.zeros((1 + scene.n_joints, 12))
    q = np.ascontiguousarray(q, dtype=np.float64)
    lib().smo_fk_flat(scene.pointer(), _p(q, C.c_double), _p(out, C.c_double))
    return out


def gjk(verts_a, xf_a, verts_b, xf_b, upper=0.0):
    va = np.ascontiguousarray(verts_a, dtype=np.float64)
    vb = np.ascontiguousarray(verts_b, dtype=np.float64)
    ta = np.ascontiguousarray(xf_a, dtype=np.float64).reshape(12)
    tb = np.ascontiguousarray(xf_b, dtype=np.float64).reshape(12)
    return lib().smo_gjk_flat(_p(va, C.c_double), len(va), _p(ta, C.c_double), _p(vb, C.c_double), len(vb),
                              _p(tb, C.c_double), C.c_double(upper))


def distances(scene, q, obst):
    """(d_static, d_self, d_moving) raw (before the 1 mm clamp) for one env."""
    q = np.ascontiguousarray(q, dtype=np.float64)
    ob = np.ascontiguousarray(obst, dtype=np.float64)
    ds, dse, dm = C.c_double(), C.c_double(), C.c_double()
    lib().smo_distances(scene.pointer(), _p(q, C.c_double), _p(ob, C.c_double), C.byref(ds), C.byref(dse),
                        C.byref(dm))
    return ds.value, dse.value, dm.value


def distances_h(scene, q, obst, hq):
    """(d_static, d_self, d_moving) raw (before the 1 mm clamp) for one env of the Human scene, the human at joint
    angles hq [8]."""
    q = np.ascontiguousarray(q, dtype=np.float64)
    ob = np.ascontiguousarray(obst, dtype=np.float64)
    hq = np.ascontiguousarray(hq, dtype=np.float64)
    ds, dse, dm = C.c_double(), C.c_double(), C.c_double()
    lib().smo_distances_h(scene.pointer(), _p(q, C.c_double), _p(ob, C.c_double), _p(hq, C.c_double), C.byref(ds),
                          C.byref(dse), C.byref(dm))
    return ds.value, dse.value, dm.value


def pair_classes(scene):
    """(class, shape A, shape B) of every pair of the distance classes, in the order of pair_distances: [n_pairs, 3],
    class 0 = static, 1 = self, 2 = moving."""
    sc = scene.struct
    rows = [(0, sc.static_pairs[i][0], sc.static_pairs[i][1]) for i in range(sc.n_static_pairs)]
    rows += [(1, sc.self_pairs[i][0], sc.self_pairs[i][1]) for i in range(sc.n_self_pairs)]
    rows += [(2, sc.mov_reward[r], sc.obst_shape_off[o] + k) for o in range(sc.n_obstacles)
             for r in range(sc.n_mov_reward) for k in range(sc.obst_shape_cnt[o])]
    return np.array(rows, dtype=np.int64).reshape(-1, 3)


def pair_distances(scene, q, obst, hq=None):
    """Distance of every pair of the distance classes (pair_classes order) for one env, margins subtracted, without
    early stop: [n_pairs].  The class rules of distances() (cap and query filters, inactive ball, latched contact) are
    not applied; hq: the human's joint angles in the Human scene."""
    q = np.ascontiguousarray(q, dtype=np.float64)
    ob = np.ascontiguousarray(obst, dtype=np.float64)
    hq = None if hq is None else np.ascontiguousarray(hq, dtype=np.float64)
    sc = scene.struct
    out = np.zeros(sc.n_static_pairs + sc.n_self_pairs +
                   sc.n_mov_reward * sum(sc.obst_shape_cnt[o] for o in range(sc.n_obstacles)))
    lib().smo_plan_pair_distances(scene.pointer(), _p(q, C.c_double), _p(ob, C.c_double),
                                  _p(hq, C.c_double) if hq is not None else None, _p(out, C.c_double))
    return out


def observation(scene, kin, obst):
    kin = np.ascontiguousarray(kin, dtype=np.float64)
    ob = np.ascontiguousarray(obst, dtype=np.float64)
    obs = np.zeros(scene.obs_size, dtype=np.float32)
    lib().smo_observation(scene.pointer(), _p(kin, C.c_double), _p(ob, C.c_double), _p(obs, C.c_float))
    return obs


class OracleEnvs:
    """N independent oracle envs with the same buffer layout as the CUDA library (SM_*_STRIDE records)."""

    def __init__(self, scene, n):
        self.scene, self.n = scene, n
        self.kin = np.zeros((n, abi.SM_KIN_STRIDE))
        self.obst = np.zeros((n, abi.SM_OBST_STRIDE))
        self.episode = np.zeros((n, 4), dtype=np.int32)
        self.ep_return = np.zeros(n)
        self.obs = np.zeros((n, scene.obs_size), dtype=np.float32)
        self.reward = np.zeros(n, dtype=np.float32)
        self.done = np.zeros(n, dtype=np.uint8)
        self.term = np.zeros(n, dtype=np.int32)
        self.info = np.zeros((n, abi.SM_INFO_STRIDE), dtype=np.float32)
        self.tp = np.zeros((n, abi.SM_TP_STRIDE)) if scene.struct.use_target_points else None
        self.human = bool(scene.struct.human.enabled)
        if self.human:   # state of the nested env that moves the human (ctlp.py:4647-4959)
            self.hkin = np.zeros((n, abi.SM_KIN_STRIDE))
            self.hstate = np.zeros((n, abi.SM_HSTATE_STRIDE))
            self.hbrake = np.zeros((n, abi.SM_HBRAKE_STEPS * abi.SM_HUMAN_JOINTS))
            self.hobs = np.zeros((n, abi.SM_HOBS_STRIDE), dtype=np.float32)
            self.hinfo = np.zeros((n, 4), dtype=np.int32)
            # smallest |d_min - brake_safety| over the poses the last step's braking check visited (inf: no check)
            self.hmargin = np.full(n, np.inf)

    def set_human_state(self, hq, hv, ha, first_target, active_arm):
        """Start state of the nested env: joint state [n, 8], first target point [n, 3] of arm active_arm [n]."""
        hq, hv, ha = (np.ascontiguousarray(x, dtype=np.float64).reshape(self.n, 8) for x in (hq, hv, ha))
        ft = np.ascontiguousarray(first_target, dtype=np.float64).reshape(self.n, 3)
        arm = np.asarray(active_arm, dtype=np.int32).reshape(self.n)
        self.hbrake[:] = 0
        for e in range(self.n):
            lib().smo_human_init(self.scene.pointer(), _p(self.hkin[e], C.c_double), _p(self.hstate[e], C.c_double),
                                 _p(hq[e], C.c_double), _p(hv[e], C.c_double), _p(ha[e], C.c_double),
                                 _p(ft[e], C.c_double), int(arm[e]), _p(self.hobs[e], C.c_float))
            lib().smo_human_initial_braking(self.scene.pointer(), _p(self.hkin[e], C.c_double),
                                            _p(self.hstate[e], C.c_double), _p(self.hbrake[e], C.c_double))
        nh = 3 * abi.SM_HUMAN_JOINTS
        self.obs[:, self.scene.obs_size - nh:] = self.hobs[:, :nh]

    def step_human(self, actions, hactions, next_target=None):
        """One step of the Human scene: robot actions [n, 7], actions of the human's policy [n, 8], the target point
        [n, 3] that replaces a reached one."""
        actions = np.ascontiguousarray(actions, dtype=np.float32)
        hact = np.ascontiguousarray(hactions, dtype=np.float32).reshape(self.n, abi.SM_HUMAN_JOINTS)
        nt = None if next_target is None else np.ascontiguousarray(next_target, dtype=np.float64).reshape(self.n, 3)
        lib().smo_step_batch_human(self.scene.pointer(), self.n, _p(self.kin, C.c_double), _p(self.obst, C.c_double),
                                   _p(self.hkin, C.c_double), _p(self.hstate, C.c_double), _p(self.hbrake, C.c_double),
                                   _p(self.episode, C.c_int32), _p(self.ep_return, C.c_double), _p(actions, C.c_float),
                                   _p(hact, C.c_float), _p(nt, C.c_double) if nt is not None else None,
                                   _p(self.obs, C.c_float), _p(self.hobs, C.c_float), _p(self.reward, C.c_float),
                                   _p(self.done, C.c_uint8), _p(self.term, C.c_int32), _p(self.info, C.c_float),
                                   _p(self.hinfo, C.c_int32), _p(self.hmargin, C.c_double))
        return self.obs, self.reward, self.done, self.term, self.info

    def set_state(self, q, v, a, obst=None, first_target=None):
        nj = self.scene.n_joints
        self.kin[:] = 0
        self.kin[:, 0:nj], self.kin[:, 8:8 + nj], self.kin[:, 16:16 + nj] = q, v, a
        # the reset of the reference poses the robot and runs one stepSimulation with the start state as motor
        # target (safe_motions_base.py:959-978): the tracked pose leaves the start position by track_vel*dt*v0
        sc = self.scene.struct
        self.kin[:, 24:24 + nj] = np.asarray(q) + (sc.track_vel * (sc.ts / sc.substeps)) * np.asarray(v)
        if obst is not None:
            self.obst[:] = obst
        self.episode[:] = 0
        self.ep_return[:] = 0
        if self.tp is not None:
            ft = np.ascontiguousarray(first_target, dtype=np.float64).reshape(self.n, 3)
            for e in range(self.n):
                lib().smo_target_init(self.scene.pointer(), _p(self.kin[e], C.c_double), _p(self.tp[e], C.c_double),
                                      _p(ft[e], C.c_double))
        for e in range(self.n):
            if self.tp is not None:
                lib().smo_observation_tp(self.scene.pointer(), _p(self.kin[e], C.c_double), _p(self.obst[e], C.c_double),
                                         _p(self.tp[e], C.c_double), _p(self.obs[e], C.c_float))
            else:
                self.obs[e] = observation(self.scene, self.kin[e], self.obst[e])

    def step(self, actions, next_ball=None, next_target=None):
        actions = np.ascontiguousarray(actions, dtype=np.float32)
        nb = None
        if next_ball is not None:
            nb = np.ascontiguousarray(next_ball, dtype=np.float64)
        nt = None
        if next_target is not None:
            nt = np.ascontiguousarray(next_target, dtype=np.float64).reshape(self.n, 3)
        lib().smo_step_batch_tp(self.scene.pointer(), self.n, _p(self.kin, C.c_double), _p(self.obst, C.c_double),
                                _p(self.tp, C.c_double) if self.tp is not None else None,
                                _p(self.episode, C.c_int32), _p(self.ep_return, C.c_double), _p(actions, C.c_float),
                                _p(nb, C.c_double) if nb is not None else None,
                                _p(nt, C.c_double) if nt is not None else None, _p(self.obs, C.c_float),
                                _p(self.reward, C.c_float), _p(self.done, C.c_uint8), _p(self.term, C.c_int32),
                                _p(self.info, C.c_float))
        return self.obs, self.reward, self.done, self.term, self.info


def human_fk(scene, hq):
    """Frames [9, 12] of the human (base, then the child link of every joint) for one joint vector [8]."""
    out = np.zeros((1 + abi.SM_HUMAN_JOINTS, 12))
    hq = np.ascontiguousarray(hq, dtype=np.float64)
    lib().smo_human_fk_flat(scene.pointer(), _p(hq, C.c_double), _p(out, C.c_double))
    return out


def human_link_points(scene, hq):
    out = np.zeros((2, 3))
    hq = np.ascontiguousarray(hq, dtype=np.float64)
    lib().smo_human_link_points(scene.pointer(), _p(hq, C.c_double), _p(out, C.c_double))
    return out


def human_safe_range(scene, q, v, a):
    q, v, a = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, v, a))
    lo, hi, code = np.zeros(8), np.zeros(8), np.zeros(8, dtype=np.int32)
    lib().smo_human_safe_range(scene.pointer(), _p(q, C.c_double), _p(v, C.c_double), _p(a, C.c_double),
                               _p(lo, C.c_double), _p(hi, C.c_double), _p(code, C.c_int32))
    return lo, hi, code


def human_pose_collides(scene, hq):
    hq = np.ascontiguousarray(hq, dtype=np.float64)
    return bool(lib().smo_human_pose_collides(scene.pointer(), _p(hq, C.c_double)))


def _check_braking(scene, q, v, a, a_target):
    q, v, a, at = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, v, a, a_target))
    acc = np.zeros((abi.SM_HBRAKE_STEPS, 8))
    k, poses, coll, margin = C.c_int(), C.c_int(), C.c_int(), C.c_double()
    ex = lib().smo_human_check_braking(scene.pointer(), _p(q, C.c_double), _p(v, C.c_double), _p(a, C.c_double),
                                       _p(at, C.c_double), _p(acc, C.c_double), C.byref(k), C.byref(poses),
                                       C.byref(coll), C.byref(margin))
    return bool(ex), acc[:min(k.value, abi.SM_HBRAKE_STEPS)], poses.value, coll.value, margin.value


def human_check_braking(scene, q, v, a, a_target):
    """(execute braking?, braking accelerations [k, 8], poses visited, first colliding pose) of the nested env's
    braking-trajectory check (ctlp.py:3026-3207)."""
    return _check_braking(scene, q, v, a, a_target)[:4]


def human_check_braking_margin(scene, q, v, a, a_target):
    """How far the braking-trajectory check of human_check_braking is from flipping: the smallest |d_min - brake_safety|
    over the poses it visited, d_min the smallest pair distance of a pose (exact up to 1e-3 m, a lower bound beyond)."""
    return _check_braking(scene, q, v, a, a_target)[4]


def human_brake_pair_distances(scene, hq):
    """Distance of every pair of the braking check (scene.struct.human.brake_pairs order) at pose hq [8], margins
    subtracted, without early stop: [n_brake_pairs]."""
    h = scene.struct.human
    hq = np.ascontiguousarray(hq, dtype=np.float64)
    out = np.zeros(h.n_brake_pairs)
    lib().smo_human_brake_pair_distances(scene.pointer(), _p(hq, C.c_double), _p(out, C.c_double))
    return out


def target_link_point(scene, q):
    out = np.zeros(3)
    qq = np.zeros(8)
    qq[:scene.n_joints] = q
    lib().smo_target_link_point(scene.pointer(), _p(qq, C.c_double), _p(out, C.c_double))
    return out


def philox(c0, c1, c2, c3, k0, k1):
    out = (C.c_uint32 * 4)()
    lib().smo_philox(C.c_uint32(c0), C.c_uint32(c1), C.c_uint32(c2), C.c_uint32(c3), C.c_uint32(k0), C.c_uint32(k1),
                     out)
    return list(out)
