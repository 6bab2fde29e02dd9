"""ctypes loader of libsmenv.so.  There is no fallback: a missing library or a failing call raises."""
import ctypes as C
import os

from . import abi
from .build import LIB

_lib = None


class SmEnvError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB):
        raise SmEnvError("libsmenv.so is missing ({}); build it with `python -m safemotionsrisk_b200.build` or "
                         "__graft_entry__.build(). There is no CPU fallback.".format(LIB))
    lib = C.CDLL(LIB)
    lib.smenv_last_error.restype = C.c_char_p
    vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int
    lib.smenv_create.argtypes = [C.POINTER(abi.SmScene), i32, i32, u64, C.POINTER(vp)]
    lib.smenv_destroy.argtypes = [vp]
    lib.smenv_pool_sizes.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    lib.smenv_pool_ptrs.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.smenv_copy_pools.argtypes = [vp, vp, vp]
    lib.smenv_fill_pools.argtypes = [vp, u64, vp]
    lib.smenv_set_state.argtypes = [vp, C.POINTER(abi.SmBuffers), vp, vp, vp, vp, vp, vp]
    lib.smenv_reset.argtypes = [vp, C.POINTER(abi.SmBuffers), vp, vp]
    lib.smenv_step.argtypes = [vp, C.POINTER(abi.SmBuffers), i32, vp]
    lib.smenv_step_random.argtypes = [vp, C.POINTER(abi.SmBuffers), i32, vp]
    lib.smenv_set_step_ranges.argtypes = [vp, i32]
    lib.smenv_step_host.argtypes = [vp, C.POINTER(abi.SmBuffers), vp, vp, vp, vp, i32, i32, vp]
    lib.smenv_safe_range.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    lib.smenv_distances.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.smenv_observation.argtypes = [vp, C.POINTER(abi.SmBuffers), vp]
    lib.smenv_counters.argtypes = [vp, C.POINTER(abi.SmCounters), i32]
    lib.smenv_enable_counters.argtypes = [vp, i32]
    lib.smenv_launch_count.argtypes = [vp, C.POINTER(C.c_ulonglong)]
    lib.smenv_set_targets.argtypes = [vp, C.POINTER(abi.SmBuffers), vp, vp, vp]
    lib.smenv_mlp_load.argtypes = [vp, i32, i32, vp, i32, i32, vp]
    lib.smenv_mlp_forward.argtypes = [vp, i32, vp, i32, vp, i32, vp, i32, i32, vp]
    lib.smenv_risk_gate.argtypes = [vp, C.POINTER(abi.SmBuffers), C.c_float, vp, vp, vp]
    lib.smenv_set_human_actions_external.argtypes = [vp, i32]
    lib.smenv_set_human_state.argtypes = [vp, C.POINTER(abi.SmBuffers), vp, vp, vp, vp, vp, vp, vp]
    lib.smenv_human_pool_sizes.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    lib.smenv_copy_human_pools.argtypes = [vp, vp, vp]
    lib.smenv_measure_fma_peaks.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.smenv_launch_config.argtypes = [vp, C.POINTER(i32)]
    lib.smenv_set_gate_exact.argtypes = [vp, i32, C.c_float]
    lib.smenv_mlp_forward_exact.argtypes = [vp, i32, vp, i32, vp, i32, vp, i32, i32, i32, vp]
    lib.smenv_mlp_shape.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32)]
    lib.smenv_set_seed.argtypes = [vp, u64]
    lib.smenv_debug_build_lut.argtypes = [vp, i32, i32, vp, i32]
    lib.smenv_debug_lut_cell.argtypes = [C.c_float, C.c_float, C.c_float, i32]
    lib.smenv_debug_human_bounds.argtypes = [C.POINTER(abi.SmScene), C.POINTER(abi.SmHumanBounds)]
    lib.smenv_debug_plan_bounds.argtypes = [C.POINTER(abi.SmScene), C.POINTER(abi.SmPlanBounds)]
    lib.smenv_set_risk_gate.argtypes = [vp, C.c_float]
    lib.smenv_set_risk_lookahead.argtypes = [vp, i32]
    lib.smenv_set_risk_next_state.argtypes = [vp, i32]
    lib.smenv_set_initial_backup_check.argtypes = [vp, i32, vp]
    lib.smenv_initial_backup_check_counts.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    lib.smenv_random_actions.argtypes = [vp, C.POINTER(abi.SmBuffers), vp]
    lib.smenv_set_agent_head.argtypes = [vp, C.c_float, C.c_float]
    lib.smenv_step_agent.argtypes = [vp, C.POINTER(abi.SmBuffers), i32, i32, vp, vp, vp, vp]
    lib.smenv_kernel_timing.argtypes = [vp, i32]
    lib.smenv_kernel_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i32), i32]
    if lib.smenv_sizeof_scene() != C.sizeof(abi.SmScene) or lib.smenv_sizeof_shape() != C.sizeof(abi.SmShape):
        raise SmEnvError("SmScene layout mismatch between abi.py ({}) and libsmenv.so ({}); rebuild".format(
            C.sizeof(abi.SmScene), lib.smenv_sizeof_scene()))
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().smenv_last_error()
        raise SmEnvError("{} failed ({}): {}".format(what, rc, msg.decode() if msg else ""))
