"""ctypes mirror of ``include/smenv.h`` (the C ABI of libsmenv.so).

The field order and sizes must match the header exactly; ``tests/test_abi.py`` checks ``ctypes.sizeof`` against
``smenv_sizeof_scene()`` / ``smenv_sizeof_shape()`` and that every symbol the header declares is exported.
"""
import ctypes as C

SM_MAX_JOINTS = 8
SM_MAX_SHAPES = 96
SM_MAX_OBSTACLES = 2
SM_MAX_PAIRS = 48
SM_MAX_MOV_ROBOT = 24
SM_KIN_STRIDE = 32
SM_OBST_STRIDE = 16
SM_INFO_STRIDE = 32
SM_TP_STRIDE = 12
SM_EP_SCALARS, SM_EP_STRIDE = 16, 64
# per-step scalars aggregated per episode (include/smenv.h SmEpisodeScalar), with the reference's info key names
EP_SCALARS = ["collision_rate_self", "collision_rate_static_obstacles", "collision_rate_moving_obstacles",
              "action_punishment", "self_collision_reward", "static_obstacles_collision_reward",
              "moving_obstacles_collision_reward", "reward", "target_point_reward", "risky_action_rate", "joint_vel_norm",
              "joint_pos_violation", "joint_vel_violation", "joint_acc_violation", "joint_jerk_violation",
              "observation_clipping_rate"]
EPC = dict(balls_hit_robot=48, balls_missed=49, targets_reached=50, first_risky_step=51, length=52, ret=53, reason=54,
           human_braked=55)
TP_POS, TP_LAST_DIST, TP_INIT_DIST, TP_ACTIVE, TP_REACHED_N, TP_LINK_POS, TP_DRAWS, TP_REACHED = 0, 3, 4, 5, 6, 7, 10, 11

SM_OBST_NONE, SM_OBST_PLANET, SM_OBST_BALL, SM_OBST_HUMAN = 0, 1, 2, 3
SM_HUMAN_JOINTS, SM_MAX_OBST_FRAMES, SM_MAX_HLINKS, SM_MAX_HPAIRS, SM_HBRAKE_STEPS, SM_HBRAKE_POSES = 8, 9, 16, 256, 24, 72
SM_HSTATE_STRIDE, SM_HOBS_STRIDE = 32, 40
HTP_SAMPLE_NEW, HTP_REACHED, HS_BRAKE_COUNT, HS_DRAWS, HS_BRAKED, HS_STEPS = 10, 11, 24, 25, 26, 27
SM_NET_RISK, SM_NET_BACKUP, SM_NET_HUMAN, SM_NET_AGENT = 0, 1, 2, 3

# termination reasons (safe_motions_base.py:64-70)
TERMINATION_UNSET = -1
TERMINATION_SUCCESS = 0
TERMINATION_JOINT_LIMITS = 1
TERMINATION_TRAJECTORY_LENGTH = 2
TERMINATION_SELF_COLLISION = 3
TERMINATION_COLLISION_WITH_STATIC_OBSTACLE = 4
TERMINATION_COLLISION_WITH_MOVING_OBSTACLE = 5

INFO_SLOTS = ["d_static", "d_self", "d_moving", "coll_static", "coll_self", "coll_moving", "action_punishment",
              "r_static", "r_self", "r_moving", "episode_length", "episode_return", "range_code", "contact_latch",
              "max_jerk_rel", "tp_reward", "risky_action", "risk", "first_risky_step", "reward_raw"]
INFO = {name: i for i, name in enumerate(INFO_SLOTS)}

OB_INDEX, OB_LATCH, OB_BALL_P0, OB_BALL_V0, OB_BALL_EULER0, OB_BALL_OMEGA, OB_BALL_T, OB_BALL_ACTIVE, \
    OB_BALL_NMAX, OB_BALL_NHIT = 0, 1, 2, 5, 8, 11, 12, 13, 14, 15

d, i32 = C.c_double, C.c_int32
dp = C.POINTER(C.c_double)


class SmShape(C.Structure):
    _fields_ = [("frame", i32), ("vert_off", i32), ("vert_cnt", i32), ("link", i32), ("margin", d),
                ("center", d * 3), ("radius", d)]


class SmHumanBounds(C.Structure):
    """Bounding volumes of the human's braking-trajectory check (include/smenv.h, smenv_debug_human_bounds)."""
    f = C.c_float
    _fields_ = [
        ("n_gp", i32), ("gp_fa", i32 * 8), ("gp_fb", i32 * 8), ("gp_a0", i32 * 8), ("gp_na", i32 * 8), ("gp_b0", i32 * 8),
        ("gp_nb", i32 * 8),
        ("gp_ca", (f * 3) * 8), ("gp_ra", f * 8), ("gp_cb", (f * 3) * 8), ("gp_rb", f * 8),
        ("gp_bmin", (f * 3) * 8), ("gp_bmax", (f * 3) * 8),
        ("gp_sa", (f * 6) * 8), ("gp_sra", f * 8), ("gp_sb", (f * 6) * 8), ("gp_srb", f * 8),
        ("hf_s0", i32 * 4), ("hf_sn", i32 * 4),
        ("hf_seg", (f * 6) * 4), ("hf_rad", f * 4), ("hf_cover_rad", f * 4), ("hf_rho", (f * 8) * 4)]
    del f


SM_PLAN_HWIDTH_CELLS = 384
SM_PLAN_MAX_PAIRS = 512


class SmPlanBounds(C.Structure):
    """Constants of the distance planning (include/smenv.h, smenv_debug_plan_bounds)."""
    f = C.c_float
    _fields_ = [
        ("n_shapes", i32), ("n_pairs_fixed", i32), ("n_pairs", i32), ("self_query", C.c_double),
        ("center", (f * 3) * SM_MAX_SHAPES), ("radius", f * SM_MAX_SHAPES),
        ("bmin", (f * 3) * SM_MAX_SHAPES), ("bmax", (f * 3) * SM_MAX_SHAPES), ("centroid", (f * 3) * SM_MAX_SHAPES),
        ("pair_tab", C.c_uint32 * SM_PLAN_MAX_PAIRS), ("pair_rm", (f * 2) * SM_PLAN_MAX_PAIRS),
        ("hwidth", (f * SM_PLAN_HWIDTH_CELLS) * SM_MAX_SHAPES)]
    del f


class SmHuman(C.Structure):
    _fields_ = [
        ("enabled", i32), ("n_joints", i32),
        ("joint_parent", i32 * SM_HUMAN_JOINTS),
        ("base_R", d * 9), ("base_t", d * 3),
        ("joint_R", (d * 9) * SM_HUMAN_JOINTS), ("joint_t", (d * 3) * SM_HUMAN_JOINTS),
        ("joint_axis", (d * 3) * SM_HUMAN_JOINTS),
        ("pos_lo", d * SM_HUMAN_JOINTS), ("pos_hi", d * SM_HUMAN_JOINTS), ("vel_max", d * SM_HUMAN_JOINTS),
        ("acc_max", d * SM_HUMAN_JOINTS), ("jerk_max", d * SM_HUMAN_JOINTS),
        ("shape_off", i32), ("n_arm_shapes", i32), ("n_shapes", i32),
        ("shape_link", i32 * 64),
        ("contact_thresh", (d * SM_MAX_MOV_ROBOT) * SM_MAX_HLINKS),
        ("check_braking", i32), ("brake_checks", i32), ("n_brake_pairs", i32),
        ("brake_pairs", (i32 * 2) * SM_MAX_HPAIRS),
        ("brake_safety", d), ("brake_timeout", d),
        ("tp_local", (d * 3) * 2),
        ("tp_box_min", d * 3), ("tp_box_max", d * 3), ("tp_rel_min", d * 3), ("tp_rel_max", d * 3), ("tp_radius", d),
        ("tp_min_static", d), ("tp_min_self", d),
        ("log_std_lo", d), ("log_std_hi", d),
        ("start_box_min", d * 3), ("start_box_max", d * 3),
        ("kinematic_sampling_probability", d), ("stay_in_state_probability", d),
        ("min_start_static", d), ("min_start_self", d),
        ("obs_size", i32), ("initial_braking_trajectory", i32),
    ]


class SmScene(C.Structure):
    _fields_ = [
        ("n_joints", i32),
        ("joint_parent", i32 * SM_MAX_JOINTS),
        ("joint_R", (d * 9) * SM_MAX_JOINTS),
        ("joint_t", (d * 3) * SM_MAX_JOINTS),
        ("joint_axis", (d * 3) * SM_MAX_JOINTS),
        ("pos_lo", d * SM_MAX_JOINTS), ("pos_hi", d * SM_MAX_JOINTS),
        ("vel_max", d * SM_MAX_JOINTS), ("acc_max", d * SM_MAX_JOINTS), ("jerk_max", d * SM_MAX_JOINTS),
        ("ts", d),
        ("substeps", i32),
        ("limit_velocity", i32), ("limit_position", i32),
        ("action_mapping_factor", d),
        ("track_kp", d), ("track_vel", d),
        ("contact_stride", i32), ("reserved0", i32),
        ("n_shapes", i32), ("n_verts", i32),
        ("shapes", SmShape * SM_MAX_SHAPES),
        ("verts", dp),
        ("n_static_pairs", i32), ("static_pairs", (i32 * 2) * SM_MAX_PAIRS),
        ("n_self_pairs", i32), ("self_pairs", (i32 * 2) * SM_MAX_PAIRS),
        ("n_mov_reward", i32), ("mov_reward", i32 * SM_MAX_MOV_ROBOT),
        ("n_mov_contact", i32), ("mov_contact", i32 * SM_MAX_MOV_ROBOT),
        ("n_obstacles", i32),
        ("obst_kind", i32 * SM_MAX_OBSTACLES),
        ("obst_shape_off", i32 * SM_MAX_OBSTACLES), ("obst_shape_cnt", i32 * SM_MAX_OBSTACLES),
        ("obst_center", (d * 3) * SM_MAX_OBSTACLES),
        ("obst_radius", d * SM_MAX_OBSTACLES),
        ("contact_thresh", (d * SM_MAX_MOV_ROBOT) * SM_MAX_OBSTACLES),
        ("planet_steps", i32), ("planet_shift", i32),
        ("planet_pos", dp * SM_MAX_OBSTACLES),
        ("planet_quat", dp * SM_MAX_OBSTACLES),
        ("planet_local_xy", dp),
        ("planet_obs_half", d * 2),
        ("obs_planet_size", i32), ("reserved1", i32),
        ("ball_obs_pos_min", d * 3), ("ball_obs_pos_max", d * 3),
        ("ball_obs_vel_min", d * 3), ("ball_obs_vel_max", d * 3),
        ("ball_active_xy", d),
        ("static_cap", d), ("moving_query", d), ("collision_dist", d),
        ("w_self", d), ("w_static", d), ("w_moving", d),
        ("d_self", d), ("d_static", d), ("d_moving", d),
        ("w_low_acc", d), ("thr_low_acc", d), ("w_low_vel", d), ("thr_low_vel", d),
        ("punish_action", i32),
        ("terminate_self", i32), ("terminate_static", i32), ("terminate_moving", i32),
        ("action_thresh", d), ("action_max_punishment", d),
        ("termination_bonus", d), ("early_termination_punishment", d),
        ("episode_steps", i32), ("obs_size", i32),
        ("start_box_min", d * 3), ("start_box_max", d * 3),
        ("target_offset", d * 3),
        ("target_R", d * 9), ("target_t", d * 3),
        ("kinematic_sampling_probability", d), ("stay_in_state_probability", d),
        ("min_start_distance", d),
        ("ball_sphere_center", d * 3), ("ball_sphere_radius", d),
        ("ball_height_min", d), ("ball_height_max", d), ("ball_angle_min", d), ("ball_angle_max", d),
        ("ball_speed", d), ("ball_radius", d), ("ball_high_angle_probability", d),
        ("ball_target_box_min", d * 3), ("ball_target_box_max", d * 3),
        ("ball_invalid_min", d * 3), ("ball_invalid_max", d * 3),
        ("ball_final_min", d * 3), ("ball_final_max", d * 3),
        ("plane_z", d),
        ("ball_check_invalid", i32), ("ball_random_initial", i32),
        ("min_start_self", d), ("ball_target_min_static", d), ("ball_target_min_self", d),
        ("has_table", i32), ("start_at_rest", i32),
        ("use_target_points", i32), ("tp_normalize", i32), ("obs_add_tp_pos", i32), ("obs_add_tp_rel", i32),
        ("tp_radius", d), ("tp_bonus", d), ("tp_reward_factor", d),
        ("tp_box_min", d * 3), ("tp_box_max", d * 3), ("tp_rel_min", d * 3), ("tp_rel_max", d * 3),
        ("tp_min_static", d), ("tp_min_self", d),
        ("reward_scale", d),
        ("human", SmHuman),
    ]


class SmBuffers(C.Structure):
    _fields_ = [
        ("kin", C.c_void_p), ("obst", C.c_void_p), ("episode", C.c_void_p), ("ep_return", C.c_void_p),
        ("actions", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("term_reason", C.c_void_p), ("info", C.c_void_p), ("stats", C.c_void_p), ("target", C.c_void_p),
        ("hkin", C.c_void_p), ("hstate", C.c_void_p), ("hbrake", C.c_void_p), ("hobs", C.c_void_p),
        ("epacc", C.c_void_p), ("epinfo", C.c_void_p),
        ("hactions", C.c_void_p),
    ]


class SmCounters(C.Structure):
    _fields_ = [("gjk_calls", C.c_ulonglong), ("gjk_iters", C.c_ulonglong), ("support_dots", C.c_ulonglong),
                ("distance_items", C.c_ulonglong), ("env_steps", C.c_ulonglong), ("contact_envs", C.c_ulonglong),
                ("contact_items", C.c_ulonglong), ("reserved", C.c_ulonglong), ("heavy_joints", C.c_ulonglong), ("heavy_solves", C.c_ulonglong), ("aux", C.c_ulonglong * 6),
                ("brake_poses", C.c_ulonglong), ("brake_pair_bounds", C.c_ulonglong), ("brake_spans", C.c_ulonglong),
                ("brake_fine_poses", C.c_ulonglong)]


# every extern "C" symbol include/smenv.h declares
EXPORTED_SYMBOLS = [
    "smenv_last_error", "smenv_abi_version", "smenv_sizeof_scene", "smenv_sizeof_shape", "smenv_create",
    "smenv_destroy", "smenv_pool_sizes", "smenv_fill_pools", "smenv_pool_ptrs", "smenv_copy_pools", "smenv_set_state", "smenv_reset",
    "smenv_step", "smenv_step_random", "smenv_step_host", "smenv_set_step_ranges", "smenv_safe_range", "smenv_distances", "smenv_observation",
    "smenv_counters", "smenv_enable_counters", "smenv_launch_count", "smenv_debug_gjk", "smenv_debug_build_lut", "smenv_debug_lut_cell", "smenv_debug_human_bounds", "smenv_debug_plan_bounds", "smenv_kernel_timing",
    "smenv_kernel_times", "smenv_set_targets", "smenv_mlp_load", "smenv_mlp_forward", "smenv_risk_gate", "smenv_random_actions",
    "smenv_set_seed", "smenv_set_risk_gate", "smenv_set_human_actions_external", "smenv_set_human_state",
    "smenv_human_pool_sizes", "smenv_copy_human_pools", "smenv_measure_fma_peaks", "smenv_launch_config", "smenv_set_gate_exact", "smenv_mlp_forward_exact",
    "smenv_set_risk_lookahead", "smenv_set_risk_next_state", "smenv_set_initial_backup_check",
    "smenv_initial_backup_check_counts", "smenv_mlp_shape", "smenv_set_agent_head", "smenv_step_agent",
]
