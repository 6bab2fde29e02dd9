/*
 * smenv.h -- C ABI of the B200-native SafeMotions environment step ("libsmenv.so").
 *
 * This is the drop-in boundary of the hot path (SURVEY.md section 8b).  Every entry point replaces a piece of the
 * reference's gym.Env surface for N independent environments at once:
 *
 *   smenv_create / smenv_destroy   <- SafeMotionsBase.__init__ / close()          (safe_motions_base.py:85, :1487)
 *   smenv_set_state                <- the injected start state of reset()          (safe_motions_base.py:913-1022,
 *                                     collision_torque_limit_prevention.py:1461-1656, parity protocol SURVEY 8c)
 *   smenv_fill_pools               <- get_starting_point_joint_pos_vel_acc + Planet.reset + _add_moving_object
 *                                     (ctlp.py:1461-1656, :4470-4501, :1723-1931) as device-side rejection sampling
 *   smenv_reset                    <- SafeObservation.reset()                       (observations.py:144-187)
 *   smenv_step                     <- SafeMotionsBase.step()                        (safe_motions_base.py:1043-1227)
 *   smenv_safe_range               <- _calculate_safe_acc_range()                   (actions.py:206-211)
 *   smenv_distances                <- get_minimum_distance(+_to_moving_obstacles)   (ctlp.py:3217-3374)
 *
 * Conventions: plain pointers and sizes only, no torch types.  All device pointers are caller-owned (the Python host
 * allocates them as torch CUDA tensors); the library owns only the read-only scene constants it uploads in
 * smenv_create.  Every call is stream-ordered on the caller's cudaStream_t and returns 0 on success or a negative
 * SmStatus; smenv_last_error() gives the message.  Nothing in this library has a CPU fallback.
 */
#ifndef SMENV_H
#define SMENV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SM_MAX_JOINTS 8
#define SM_MAX_SHAPES 96
#define SM_MAX_OBSTACLES 2
#define SM_MAX_PAIRS 48
#define SM_MAX_MOV_ROBOT 24
#define SM_MAX_OBS 64
#define SM_KIN_STRIDE 32  /* doubles per env in the kinematic record: q[8] v[8] a[8] q_act[8] */
#define SM_OBST_STRIDE 16 /* doubles per env in the obstacle record */
#define SM_INFO_STRIDE 32 /* floats per env in the step-info record */

enum SmStatus { SM_OK = 0, SM_ERR_ARG = -1, SM_ERR_CUDA = -2, SM_ERR_SCENE = -3, SM_ERR_STATE = -4 };
enum SmObstacleKind { SM_OBST_NONE = 0, SM_OBST_PLANET = 1, SM_OBST_BALL = 2, SM_OBST_HUMAN = 3 };

/* Termination reasons: SafeMotionsBase.TERMINATION_* (safe_motions_base.py:64-70). */
enum SmTermination {
    SM_TERM_UNSET = -1,
    SM_TERM_JOINT_LIMITS = 1,
    SM_TERM_TRAJECTORY_LENGTH = 2,
    SM_TERM_SELF_COLLISION = 3,
    SM_TERM_STATIC_COLLISION = 4,
    SM_TERM_MOVING_COLLISION = 5
};

/* Slots of the per-env float info record written by smenv_step (SM_INFO_STRIDE floats per env). */
enum SmInfoSlot {
    SM_INFO_D_STATIC = 0,       /* min distance to static obstacles after the <1 mm clamp (rewards.py:115-117) */
    SM_INFO_D_SELF = 1,         /* idem self collision (rewards.py:119-121) */
    SM_INFO_D_MOVING = 2,       /* idem moving obstacles (rewards.py:153-155) */
    SM_INFO_COLL_STATIC = 3,    /* collision_rate_static_obstacles (safe_motions_base.py:1350-1355) */
    SM_INFO_COLL_SELF = 4,
    SM_INFO_COLL_MOVING = 5,
    SM_INFO_ACTION_PUNISH = 6,  /* rewards.py:164-169 */
    SM_INFO_R_STATIC = 7,       /* static_obstacles_collision_reward (rewards.py:128-131) */
    SM_INFO_R_SELF = 8,
    SM_INFO_R_MOVING = 9,
    SM_INFO_EPISODE_LENGTH = 10,
    SM_INFO_EPISODE_RETURN = 11,
    SM_INFO_RANGE_CODE = 12,    /* OR of the per-joint violation codes of the range used for this step */
    SM_INFO_CONTACT_LATCH = 13, /* 1 if a sub-step contact with a moving obstacle was latched (ctlp.py:2631-2637) */
    SM_INFO_MAX_JERK_REL = 14,  /* max_j |jerk_j| / jerk_max_j of the step (rewards.py:181-203) */
    SM_INFO_TP_REWARD = 15,     /* target_point_reward (rewards.py:345-348) */
    SM_INFO_RISKY_ACTION = 16,  /* risky_action_rate of the step: 1 if the risk gate replaced the action (actions.py:335-340) */
    SM_INFO_RISK = 17,          /* the risk network's prediction for the proposed action (safe_motions_base.py:1600) */
    SM_INFO_FIRST_RISKY_STEP = 18, /* risk_network_first_risky_action_step of the episode, -1 = none so far
                                      (actions.py:337-338, safe_motions_base.py:1378) */
    SM_INFO_REWARD_RAW = 19     /* reward before normalize_reward_to_frequency (rewards.py:172-176) */
};

/* Slots of the per-env obstacle record (SM_OBST_STRIDE doubles per env; integers are stored exactly as doubles). */
enum SmObstSlot {
    SM_OB_INDEX = 0,        /* planets: current_time_step_index of planet one (planet two is phase-coupled,
                               ctlp.py:4470-4531); ball: position_update_step_counter (ctlp.py:4103-4105) */
    SM_OB_LATCH = 1,        /* latched contact: Planet._collision_detected / Ball final state HIT_ROBOT */
    SM_OB_BALL_P0 = 2,      /* release point xyz (ctlp.py:1933-1954) */
    SM_OB_BALL_V0 = 5,      /* initial speed vector xyz (ctlp.py:1792-1809) */
    SM_OB_BALL_EULER0 = 8,  /* initial orientation as euler xyz (ctlp.py:4029-4034) */
    SM_OB_BALL_OMEGA = 11,  /* angular velocity of euler-y in rad/s (ctlp.py:4056-4057) */
    SM_OB_BALL_T = 12,      /* accumulated flight time self._t (ctlp.py:4105) */
    SM_OB_BALL_ACTIVE = 13, /* moving_object_active_list[0] (ctlp.py:2836-2861) */
    SM_OB_BALL_NMAX = 14,   /* max_time_update_step_counter (ctlp.py:4101) */
    SM_OB_BALL_NHIT = 15    /* obstacle_hit_time (ctlp.py:1889-1917) */
};

/* ---- Human scene (Human, ctlp.py:4647-4959: a nested SafeMotionsEnv(robot_scene=9) drives a human's two arms) ---- */
#define SM_HUMAN_JOINTS 8      /* two arms x (flexion, adduction, rotation, forearm), description/urdf/human.urdf:140-416 */
#define SM_MAX_OBST_FRAMES 9   /* frames of obstacle shapes: 100 = obstacle 0 (human: its base), 101 = obstacle 1 (human:
                                  child link of human joint 0), ..., 108 = child link of human joint 7 */
#define SM_MAX_HLINKS 16       /* human URDF links carrying collision shapes */
#define SM_MAX_HPAIRS 256      /* convex pairs of the human's braking-trajectory collision check */
#define SM_HBRAKE_STEPS 24     /* stored braking accelerations per env (braking timeout 2 s = 21 steps, ctlp.py:3467-3473) */
#define SM_HBRAKE_POSES 72     /* poses one braking-trajectory check can visit: 3 per step x (1 + 21 braking steps), rounded up */
#define SM_HSTATE_STRIDE 32    /* doubles per env in the human's state record */
#define SM_HOBS_STRIDE 40      /* floats per env in the human's observation record (38 used, observations.py:54-117) */
/* Slots of the human's state record (SmBuffers.hstate).  Per arm r (0, 1) a target-point block at 12 * r with the
 * layout of SmTargetSlot up to SM_TP_LINK_POS, then: */
#define SM_HTP_SAMPLE_NEW 10   /* _sample_new_target_point_list[r] (ctlp.py:2813-2818) */
#define SM_HTP_REACHED 11      /* _target_point_reached_list[r] */
enum SmHumanSlot {
    SM_HS_BRAKE_COUNT = 24,    /* accelerations left in _valid_braking_trajectories['current'] (0 = None, ctlp.py:3000-3024) */
    SM_HS_DRAWS = 25,          /* target points drawn from the pool so far (Philox counter) */
    SM_HS_BRAKED = 26,         /* 1 if the last step executed the stored braking trajectory (adaptation_punishment) */
    SM_HS_STEPS = 27           /* steps of the nested env in this episode (Philox counter of the policy noise) */
};

typedef struct SmHuman {
    int32_t enabled;
    int32_t n_joints;                          /* 8 */
    int32_t joint_parent[SM_HUMAN_JOINTS];     /* parent human frame: 0 = base, 1 + j = child link of joint j */
    double base_R[9], base_t[3];               /* world pose of the human's root link (robot_scene_base.py:175-183) */
    double joint_R[SM_HUMAN_JOINTS][9], joint_t[SM_HUMAN_JOINTS][3], joint_axis[SM_HUMAN_JOINTS][3];
    double pos_lo[SM_HUMAN_JOINTS], pos_hi[SM_HUMAN_JOINTS], vel_max[SM_HUMAN_JOINTS], acc_max[SM_HUMAN_JOINTS],
        jerk_max[SM_HUMAN_JOINTS];             /* robot_scene_base.py:24-25, :347-371 (no safety buffer for the human) */
    int32_t shape_off, n_arm_shapes, n_shapes; /* SmScene.shapes[shape_off ...]: first the parts of upper arm / forearm / hand
                                                  of both arms (the obstacle links, ctlp.py:4772-4774), then the body parts */
    int32_t shape_link[64];                    /* per human shape: index of its URDF link in contact_thresh */
    double contact_thresh[SM_MAX_HLINKS][SM_MAX_MOV_ROBOT]; /* manifold threshold per (human link, robot contact slot) */
    /* braking-trajectory collision check of the nested env (ctlp.py:3026-3207; human_network/params.json) */
    int32_t check_braking;
    int32_t brake_checks;                      /* collision_checks_per_time_step (ctlp.py:99-103) */
    int32_t n_brake_pairs;
    int32_t brake_pairs[SM_MAX_HPAIRS][2];     /* (human shape, static obstacle shape or human shape), ctlp.py:3282-3374 */
    double brake_safety;                       /* closest_point_safety_distance of the nested env */
    double brake_timeout;                      /* 2.0 s (ctlp.py:3467-3473) */
    /* target points of the nested env: target_point_sequence = 1, alternating between the arms (ctlp.py:2210-2350) */
    double tp_local[2][3];                     /* target link point ("hand" + target_link_offset) in the frame of the
                                                  arm's last joint */
    double tp_box_min[3], tp_box_max[3], tp_rel_min[3], tp_rel_max[3], tp_radius;
    double tp_min_static, tp_min_self;         /* clearances of the pose a target point is sampled from */
    /* stochastic policy head (keras_fcnet_last_layer_activation.py:187-202) */
    double log_std_lo, log_std_hi;
    /* start-state sampling of the nested env (ctlp.py:1461-1656 with the human_network_* keys) */
    double start_box_min[3], start_box_max[3];
    double kinematic_sampling_probability, stay_in_state_probability, min_start_static, min_start_self;
    int32_t obs_size;                          /* 38 */
    int32_t initial_braking_trajectory;        /* the reset seeds the stored braking trajectory from the start state
                                                  (always_use_collision_avoidance_starting_point_sampling,
                                                  safe_motions_base.py:961-967, ctlp.py:1120-1139) */
} SmHuman;

typedef struct SmShape {
    int32_t frame;    /* 0 = world, 1..n_joints = robot link frame of joint (frame-1), 100+k = obstacle frame k */
    int32_t vert_off; /* first vertex in SmScene.verts */
    int32_t vert_cnt;
    int32_t link;     /* URDF link index of the robot link carrying the shape, -1 for obstacles */
    double margin;    /* Bullet collision margin subtracted from the core distance (1 mm for URDF shapes) */
    double center[3]; /* bounding sphere of the core vertices, in frame coordinates */
    double radius;
} SmShape;

/*
 * Scene constants for one env configuration.  Built on the host by safemotionsrisk_b200/scene.py from the compiled
 * URDF/mesh assets and the reference's env_config keys; uploaded once per smenv_create.
 */
typedef struct SmScene {
    /* --- kinematics: frame f = 1+j is the URDF child link of revolute joint j (SURVEY 8a row a7) */
    int32_t n_joints;
    int32_t joint_parent[SM_MAX_JOINTS]; /* parent frame (0 = world) */
    double joint_R[SM_MAX_JOINTS][9];    /* fixed rotation parent frame -> joint frame (row major) */
    double joint_t[SM_MAX_JOINTS][3];
    double joint_axis[SM_MAX_JOINTS][3];
    /* --- limits (robot_scene_base.py:20-22, :347-371, :441-455) */
    double pos_lo[SM_MAX_JOINTS], pos_hi[SM_MAX_JOINTS];
    double vel_max[SM_MAX_JOINTS], acc_max[SM_MAX_JOINTS], jerk_max[SM_MAX_JOINTS];
    double ts;            /* trajectory_time_step */
    int32_t substeps;     /* obstacle_client_update_steps_per_action = round(ts / (1/240)) */
    int32_t limit_velocity, limit_position; /* actions.py:31-32 */
    double action_mapping_factor;           /* actions.py:35, :271-276 */
    /* --- motor tracking model of the simulation client (SURVEY Appendix B.4; robot_scene_base.py:789-805) */
    double track_kp;      /* 0.1: PyBullet default positionGain */
    double track_vel;     /* 0.87 with use_controller_target_velocities, else 0 */
    int32_t contact_stride; /* test contacts every contact_stride sub-steps (1 = every 1/240 s as the reference) */
    int32_t reserved0;
    /* --- collision geometry */
    int32_t n_shapes;
    int32_t n_verts;
    SmShape shapes[SM_MAX_SHAPES];
    const double* verts; /* n_verts x 3, host pointer */
    int32_t n_static_pairs;
    int32_t static_pairs[SM_MAX_PAIRS][2]; /* (robot shape, static obstacle shape) */
    int32_t n_self_pairs;
    int32_t self_pairs[SM_MAX_PAIRS][2];
    int32_t n_mov_reward;                    /* robot shapes observed for the moving-obstacle distance */
    int32_t mov_reward[SM_MAX_MOV_ROBOT];
    int32_t n_mov_contact;                   /* robot shapes that can make contact in the simulation client */
    int32_t mov_contact[SM_MAX_MOV_ROBOT];
    /* --- moving obstacles */
    int32_t n_obstacles;
    int32_t obst_kind[SM_MAX_OBSTACLES];
    int32_t obst_shape_off[SM_MAX_OBSTACLES], obst_shape_cnt[SM_MAX_OBSTACLES];
    double obst_center[SM_MAX_OBSTACLES][3]; /* bounding sphere of the whole obstacle body (incl. margins) */
    double obst_radius[SM_MAX_OBSTACLES];
    double contact_thresh[SM_MAX_OBSTACLES][SM_MAX_MOV_ROBOT]; /* manifold contact-breaking threshold per link */
    /* planets */
    int32_t planet_steps;                         /* table length (1200) */
    int32_t planet_shift;                         /* time_step_index_shift of planet two (ctlp.py:4435-4437) */
    const double* planet_pos[SM_MAX_OBSTACLES];   /* planet_steps x 3 */
    const double* planet_quat[SM_MAX_OBSTACLES];  /* planet_steps x 4 (xyzw) */
    const double* planet_local_xy;                /* planet_steps x 2, planet one, for the observation */
    double planet_obs_half[2];                    /* 1.05 * radius_xy (observations.py:280-288) */
    int32_t obs_planet_size;                      /* obs_planet_size_per_planet: 1 or 2 */
    int32_t reserved1;
    /* ball */
    double ball_obs_pos_min[3], ball_obs_pos_max[3]; /* ctlp.py:303-333 */
    double ball_obs_vel_min[3], ball_obs_vel_max[3]; /* ctlp.py:335-348 */
    double ball_active_xy;                           /* 1.25 m (ctlp.py:2830) */
    /* --- distances / reward (rewards.py:95-169, :432-502) */
    double static_cap;       /* closest_point_maximum_relevant_distance (ctlp.py:354-366) */
    double moving_query;     /* query distance for moving obstacles (rewards.py:142-151) */
    double collision_dist;   /* 0.001 */
    double w_self, w_static, w_moving;
    double d_self, d_static, d_moving;
    double w_low_acc, thr_low_acc, w_low_vel, thr_low_vel;
    int32_t punish_action;
    int32_t terminate_self, terminate_static, terminate_moving;
    double action_thresh, action_max_punishment;
    double termination_bonus, early_termination_punishment;
    int32_t episode_steps;   /* round(trajectory_duration / ts) (trajectory_manager.py:87, :187-192) */
    int32_t obs_size;
    /* --- start-state sampling (ctlp.py:171-183, :1461-1656) */
    double start_box_min[3], start_box_max[3];
    double target_offset[3];   /* target_link_offset in the frame of the last joint (after the fixed EE transform) */
    double target_R[9], target_t[3]; /* fixed transform last joint frame -> target link frame */
    double kinematic_sampling_probability, stay_in_state_probability;
    double min_start_distance;  /* 0.001 in collision-avoidance mode */
    /* ball launch (ctlp.py:1723-1954) */
    double ball_sphere_center[3], ball_sphere_radius, ball_height_min, ball_height_max, ball_angle_min, ball_angle_max;
    double ball_speed, ball_radius, ball_high_angle_probability;
    double ball_target_box_min[3], ball_target_box_max[3];   /* target_point_cartesian_range */
    double ball_invalid_min[3], ball_invalid_max[3];         /* invalid target link point area */
    double ball_final_min[3], ball_final_max[3];             /* final_ball_position_min_max */
    double plane_z;                                          /* plane_z_offset */
    int32_t ball_check_invalid, ball_random_initial;
    double min_start_self;         /* self-collision clearance of a start pose (ctlp.py:1468-1477) */
    double ball_target_min_static; /* clearances of the random pose a ball is aimed at (ctlp.py:1725-1728) */
    double ball_target_min_self;
    int32_t has_table;             /* obstacle_scene != 0 (ctlp.py:1890) */
    int32_t start_at_rest;         /* not collision_avoidance_mode: start states have zero velocity and acceleration
                                      (ctlp.py:1461-1500) */
    /* --- target points of the reaching task (SafeMotionsEnv / TargetPointReachingReward: rewards.py:303-396;
     *     ctlp.py:1658-1720, :2210-2350, :2787-2821); single robot, target_point_sequence 0 */
    int32_t use_target_points;
    int32_t tp_normalize;          /* normalize_reward_to_initial_target_point_distance */
    int32_t obs_add_tp_pos, obs_add_tp_rel; /* obs_add_target_point_pos / _relative_pos (observations.py:326-340) */
    double tp_radius;              /* target_point_radius */
    double tp_bonus;               /* target_point_reached_reward_bonus */
    double tp_reward_factor;       /* target_point_reward_factor */
    double tp_box_min[3], tp_box_max[3]; /* target_point_cartesian_range (sampling and position normalisation) */
    double tp_rel_min[3], tp_rel_max[3]; /* target_point_relative_pos_min_max (ctlp.py:184) */
    double tp_min_static, tp_min_self;   /* clearances of the pose a target point is sampled from (ctlp.py:1661-1664) */
    double reward_scale;           /* trajectory_time_step / 0.1 with normalize_reward_to_frequency, else 1 (rewards.py:172-176) */
    SmHuman human;                 /* the human obstacle (human_network_checkpoint), else enabled = 0 */
} SmScene;

#define SM_TP_STRIDE 12 /* doubles per env in the target-point record */
/* Slots of the per-env target-point record (SmBuffers.target). */
enum SmTargetSlot {
    SM_TP_POS = 0,        /* target point xyz */
    SM_TP_LAST_DIST = 3,  /* _last_target_point_distance_list (ctlp.py:2242) */
    SM_TP_INIT_DIST = 4,  /* _initial_target_point_distance_list[-1] (ctlp.py:2244-2245) */
    SM_TP_ACTIVE = 5,     /* _target_point_active_list */
    SM_TP_REACHED_N = 6,  /* _num_target_points_reached_list */
    SM_TP_LINK_POS = 7,   /* _target_link_pos_list: target link point at the current knot (setpoint pose) xyz */
    SM_TP_DRAWS = 10,     /* target points drawn from the pool so far (Philox counter) */
    SM_TP_REACHED = 11    /* 1 if the target point was reached in the step just finished */
};

/* Per-episode aggregation of the step info (what train.py:59-117 computes from the per-step info dicts of the reference:
 * custom_metrics[key + "_average" / "_max" / "_min"]).  SM_EP_SCALARS step scalars are accumulated on the device in
 * SmBuffers.epacc (sum, max, min); when an episode ends the record is copied to SmBuffers.epinfo (which survives the
 * auto reset) and the accumulators restart. */
#define SM_EP_SCALARS 16
#define SM_EP_STRIDE 64   /* floats: sum[16] max[16] min[16], then the episode counters below, spare */
enum SmEpisodeScalar {
    SM_EP_COLL_SELF = 0, SM_EP_COLL_STATIC = 1, SM_EP_COLL_MOVING = 2,   /* collision_rate_* (safe_motions_base.py:1350-1355) */
    SM_EP_ACTION_PUNISH = 3, SM_EP_R_SELF = 4, SM_EP_R_STATIC = 5, SM_EP_R_MOVING = 6, /* rewards.py:490-498 */
    SM_EP_REWARD = 7,              /* reward (rewards.py:177-178) */
    SM_EP_TP_REWARD = 8,           /* target_point_reward (rewards.py:380-389) */
    SM_EP_RISKY_ACTION = 9,        /* risky_action_rate (actions.py:339-340) */
    SM_EP_JOINT_VEL_NORM = 10,     /* joint_vel_norm (observations.py:405) */
    SM_EP_POS_VIOLATION = 11, SM_EP_VEL_VIOLATION = 12, SM_EP_ACC_VIOLATION = 13, /* joint_*_violation (observations.py:406-408) */
    SM_EP_JERK_VIOLATION = 14,     /* joint_jerk_violation (rewards.py:195-203) */
    SM_EP_OBS_CLIPPING = 15        /* observation_clipping_rate (observations.py:410-413), kinematic entries */
};
enum SmEpisodeCounter {
    SM_EPC_BALLS_HIT_ROBOT = 48,   /* moving_object_hit_robot_total (ctlp.py:1186-1206) */
    SM_EPC_BALLS_MISSED = 49,      /* moving_object_missed_robot_total + moving_object_hit_obstacle_total */
    SM_EPC_TARGETS_REACHED = 50,   /* obstacles_num_target_points_reached (ctlp.py:1158-1163) */
    SM_EPC_FIRST_RISKY_STEP = 51,  /* risk_network_first_risky_action_step, -1 = none (safe_motions_base.py:1378) */
    SM_EPC_LENGTH = 52, SM_EPC_RETURN = 53, SM_EPC_REASON = 54,
    SM_EPC_HUMAN_BRAKED = 55       /* steps in which the human's nested env executed its braking trajectory */
};

/* Device buffers of one call (all caller-owned, N = num_envs). */
typedef struct SmBuffers {
    double* kin;          /* [N][SM_KIN_STRIDE]  q, v, a, q_act */
    double* obst;         /* [N][SM_OBST_STRIDE] */
    int32_t* episode;     /* [N][4]  episode_length, reset_count, ball draws, 1 + first risky step of the episode (0 = none) */
    double* ep_return;    /* [N] running episode return */
    const float* actions; /* [N][n_joints] in [-1, 1] */
    float* obs;           /* [N][obs_size] */
    float* reward;        /* [N] */
    uint8_t* done;        /* [N] */
    int32_t* term_reason; /* [N] */
    float* info;          /* [N][SM_INFO_STRIDE] */
    double* stats;        /* [32] episode statistics accumulated with atomics (train.py:59-117); may be NULL */
    double* target;       /* [N][SM_TP_STRIDE] target-point records; NULL unless the scene uses target points */
    /* Human scene only (else NULL): state of the nested env that moves the human's arms */
    double* hkin;         /* [N][SM_KIN_STRIDE]  q, v, a, q_act of the human's joints */
    double* hstate;       /* [N][SM_HSTATE_STRIDE] target points of both arms, braking-trajectory bookkeeping */
    double* hbrake;       /* [N][SM_HBRAKE_STEPS][SM_HUMAN_JOINTS] accelerations of the stored braking trajectory */
    float* hobs;          /* [N][SM_HOBS_STRIDE] observation of the nested env (input of the human's policy) */
    float* epacc;         /* [N][SM_EP_STRIDE] running aggregates of the current episode; may be NULL (no aggregation) */
    float* epinfo;        /* [N][SM_EP_STRIDE] aggregates of the last finished episode of every env; NULL iff epacc is */
    float* hactions;      /* [N][SM_HUMAN_JOINTS] actions of the human's policy: written by the step (policy network +
                             Philox noise), or read from here when smenv_set_human_actions_external(1) (parity tests) */
} SmBuffers;

typedef struct SmCounters {
    unsigned long long gjk_calls;      /* convex pair queries run by the GJK kernel (= work items) */
    unsigned long long gjk_iters;      /* GJK iterations summed over the pairs */
    unsigned long long support_dots;   /* vertex . direction products evaluated in support searches */
    unsigned long long distance_items; /* pairs the distance planning could not cull (emitted items) */
    unsigned long long env_steps;
    unsigned long long contact_envs;   /* spans of sub-steps the coarse contact phase passed on to the fine planning */
    unsigned long long contact_items;  /* (sub-step, pair) contact candidates emitted by the contact planning */
    unsigned long long reserved;       /* braking-profile intervals evaluated by the iterative position-bound solves */
    unsigned long long heavy_joints;   /* (env, joint) instances that went through joint_heavy_kernel */
    unsigned long long heavy_solves;   /* position bounds that needed the iterative solve */
    unsigned long long aux[6];         /* GJK pairs by iteration count: <= 4, <= 8, <= 12, <= 16, <= 24, more */
    unsigned long long brake_poses;        /* Human: poses the braking-trajectory check visited */
    unsigned long long brake_pair_bounds;  /* Human: sphere bounds of convex pairs evaluated by the per-pose pass */
    unsigned long long brake_spans;        /* Human: spans of consecutive poses the inflated span pass tested */
    unsigned long long brake_fine_poses;   /* Human: poses of the spans it could not clear, passed to the per-pose pass */
} SmCounters;

/* Kernels of one step, in launch order (smenv_kernel_times). */
enum SmKernel {
    /* Human scene only (zero elsewhere): policy network + noise, safe range of the human's joints, braking trajectory in
     * joint space, its pose checks (planning, GJK), bookkeeping + setpoints + outcome of the nested env */
    SM_K_HUMAN_POLICY = 0, SM_K_HUMAN_JOINT = 1, SM_K_HUMAN_BRAKE_TRAJ = 2, SM_K_HUMAN_BRAKE_PLAN = 3,
    SM_K_HUMAN_BRAKE_GJK = 4, SM_K_HUMAN_ADVANCE = 5,
    SM_K_JOINT = 6, SM_K_JOINT_HEAVY = 7, SM_K_CONTACT_PLAN = 8, SM_K_DISTANCE_PLAN = 9, SM_K_GJK = 10, SM_K_FINISH = 11,
    SM_K_COUNT = 12
};

typedef struct SmEnv SmEnv;
typedef void* SmStream; /* cudaStream_t */

const char* smenv_last_error(void);
int smenv_abi_version(void);
int smenv_sizeof_scene(void);
int smenv_sizeof_shape(void);

int smenv_create(const SmScene* scene, int num_envs, int device, uint64_t seed, SmEnv** out);
int smenv_destroy(SmEnv* env);
/* SafeMotionsBase.set_seed (safe_motions_base.py:1704-1710): new Philox key for every draw made from now on (pool
 * picks of resets / balls / target points, random actions); the step counter of the random actions restarts at 0.
 * Re-draw the pools with smenv_fill_pools(seed) to reproduce an env created with that seed. */
int smenv_set_seed(SmEnv* env, uint64_t seed);

/* Start-state / ball pools, sampled on the device (rejection sampling with Philox). */
int smenv_pool_sizes(SmEnv* env, int* start_pool, int* ball_pool);
int smenv_fill_pools(SmEnv* env, uint64_t seed, SmStream stream);
int smenv_pool_ptrs(SmEnv* env, double** start_pool, double** ball_pool);
/* Copies the pools to host arrays of pool_size x 48 / x 12 doubles (either may be NULL); synchronises the device. */
int smenv_copy_pools(SmEnv* env, double* host_start, double* host_ball);

/* Injects a start state (parity protocol).  Host or device pointers are both accepted; mask==NULL means all envs. */
int smenv_set_state(SmEnv* env, const SmBuffers* buf, const double* q, const double* v, const double* a,
                    const double* obst, const uint8_t* mask, SmStream stream);
/* Reaching task: injects the first target point of every (masked) env ([N][3], host or device) after smenv_set_state
 * (parity protocol; the reference samples it by rejection, ctlp.py:1658-1720) and rewrites the observation. */
int smenv_set_targets(SmEnv* env, const SmBuffers* buf, const double* first_target, const uint8_t* mask,
                      SmStream stream);
/* Resets the masked envs (NULL = all) from the pools and writes their first observation. */
int smenv_reset(SmEnv* env, const SmBuffers* buf, const uint8_t* mask, SmStream stream);
/* One env step for all N envs.  auto_reset != 0 re-initialises finished envs from the pools inside the same launch
 * (obs is then the first observation of the new episode; done/reward/info describe the finished step). */
int smenv_step(SmEnv* env, const SmBuffers* buf, int auto_reset, SmStream stream);
/* Same launch with device-generated U(-1,1) actions (get_random_action, safe_motions_base.py:1327-1328). */
int smenv_step_random(SmEnv* env, const SmBuffers* buf, int auto_reset, SmStream stream);
/* Number of env ranges (1..8) smenv_step / smenv_step_random run side by side on internal streams (joined on the
 * caller's stream before the call returns control of it).  Results do not depend on it.  Default: 2 from 16 384 envs,
 * else 1.  The measurement mode (smenv_kernel_timing) always uses one range. */
int smenv_set_step_ranges(SmEnv* env, int ranges);
/* The step as an RL sampler calls it, with HOST buffers (pinned for full speed): actions [N][n_joints] in, observation
 * [N][obs_size], reward [N] and done [N] out; the state stays on the device in `buf` (buf->actions / obs / reward / done
 * are the device staging buffers).  The envs are cut into `chunks` (1..8) ranges that run on internal streams, so the
 * host<->device copies of one range overlap the kernels of the others; results do not depend on `chunks`.  Ordered
 * after the work already queued on `stream`; returns when the host buffers are complete.
 * Replaces the per-env `env.step(action)` loop of the RLlib sampler / evaluate.py:198-303 over num_envs envs. */
int smenv_step_host(SmEnv* env, const SmBuffers* buf, const float* h_actions, float* h_obs, float* h_reward,
                    uint8_t* h_done, int auto_reset, int chunks, SmStream stream);

/* Pieces of the step exposed for parity tests. */
int smenv_safe_range(SmEnv* env, const double* kin, double* range_lo, double* range_hi, int32_t* code, int n,
                     SmStream stream);
/* hkin: [n][SM_KIN_STRIDE] joint state of the human (Human scene), else NULL */
int smenv_distances(SmEnv* env, const double* kin, const double* obst, const double* hkin, float* d_static, float* d_self,
                    float* d_moving, int n, SmStream stream);
int smenv_observation(SmEnv* env, const SmBuffers* buf, SmStream stream);

/* Human scene: with external != 0 the step takes the human's actions from buf->hactions instead of evaluating the
 * human's policy (parity protocol: the reference samples them from a stochastic policy, ctlp.py:4701, :4827). */
int smenv_set_human_actions_external(SmEnv* env, int external);
/* Human scene: injects the nested env's start state after smenv_set_state (hq, hv, ha [N][8]; first target point of the
 * active arm [N][3]; active_arm [N] int32), host or device pointers, and rewrites both observations. */
int smenv_set_human_state(SmEnv* env, const SmBuffers* buf, const double* hq, const double* hv, const double* ha,
                          const double* first_target, const int32_t* active_arm, const uint8_t* mask, SmStream stream);
/* Human scene: pools of the nested env's start states / target points (sampled by smenv_fill_pools). */
int smenv_human_pool_sizes(SmEnv* env, int* start_pool, int* target_pool);
int smenv_copy_human_pools(SmEnv* env, double* host_start /* [P][64] */, double* host_target /* [2][T][4] */);

int smenv_counters(SmEnv* env, SmCounters* out, int reset);
int smenv_enable_counters(SmEnv* env, int enable);
int smenv_launch_count(SmEnv* env, unsigned long long* out);
/* out[8]: GJK grid, GJK threads per CTA, GJK dynamic shared memory bytes, direction-table words, planning grid, planning
 * shared memory bytes, SM count, env ranges of the device step */
int smenv_launch_config(SmEnv* env, int32_t* out);
/* Measurement mode: with enable != 0 every smenv_step brackets each of its kernels with CUDA events on the caller's
 * stream and synchronises at the end of the step (so it is for measurement passes, not for the timed rollout).
 * smenv_kernel_times returns the accumulated milliseconds per SmKernel and the number of steps accumulated. */
int smenv_kernel_timing(SmEnv* env, int enable);
int smenv_kernel_times(SmEnv* env, double* ms_out /* SM_K_COUNT */, int* steps_out, int reset);
/*
 * Networks in the step loop (safe_motions_base.py:1498-1603, actions.py:303-340): batched inference on the tensor
 * cores.  which: SM_NET_RISK = risk(obs, action) -> [0, 1]; SM_NET_BACKUP = backup policy, obs -> action mean.
 * dims = { n_in, N_1 .. N_n_tc, n_out }: n_tc hidden Dense layers (widths 16, 32, 48, 64, 128, 192, 256 or 512) and
 * one output Dense layer (n_out <= 16; SM_NET_HUMAN: the human's stochastic policy, means and log-std outputs,
 * ctlp.py:4647-4762; SM_NET_AGENT: the policy that acts in the env, see smenv_step_agent).  weights (host, float32,
 * Keras layout): per layer kernel [in][out] row-major followed by its bias.  hidden_act: 0 selu, 1 swish; out_act:
 * 0 sigmoid, 1 tanh.
 */
enum SmNet { SM_NET_RISK = 0, SM_NET_BACKUP = 1, SM_NET_HUMAN = 2, SM_NET_AGENT = 3, SM_NET_COUNT = 4 };
int smenv_mlp_load(SmEnv* env, int which, int n_tc, const int32_t* dims, int hidden_act, int out_act,
                   const float* weights);
/* out[n][out_stride] = net([in0 row, in1 row]) for n rows; all device pointers (in1 may be NULL with in1_w = 0).  Every
 * output of the network is written: SM_ERR_ARG if out_stride is smaller than its output count. */
int smenv_mlp_forward(SmEnv* env, int which, const float* in0, int in0_w, const float* in1, int in1_w, float* out,
                      int out_stride, int n, SmStream stream);
/* Input and output widths of the loaded network `which` (either pointer may be NULL); SM_ERR_STATE if none is loaded. */
int smenv_mlp_shape(SmEnv* env, int which, int* n_in, int* n_out);
/* Risk gate on buf->actions in place: risk(obs, action) >= threshold replaces the env's action by the backup policy's
 * (obs = buf->obs, the observation the action was computed from).  risk_out [N] / risky_out [N] may be NULL.
 * SM_ERR_STATE if the loaded risk network is a state network (see smenv_set_risk_next_state). */
int smenv_risk_gate(SmEnv* env, const SmBuffers* buf, float threshold, float* risk_out, uint8_t* risky_out,
                    SmStream stream);
/* Risk gate inside the step (actions.py:303-340): with threshold >= 0 every smenv_step / smenv_step_random /
 * smenv_step_host first rates buf->actions with the risk network on buf->obs and executes the backup policy's action
 * in the envs rated >= threshold.  buf->actions keeps the proposed action (the action punishment of the reward is
 * computed from it, safe_motions_base.py:1066); info slots SM_INFO_RISKY_ACTION / RISK / FIRST_RISKY_STEP report the
 * gate.  Needs both networks (smenv_mlp_load).  threshold < 0 switches the gate off (default).  The risk network's input
 * width, recorded by smenv_mlp_load, tells its kind: the risk observation followed by the action (a state-action network,
 * which the network gate needs) or the risk observation alone (a state network, which smenv_set_risk_next_state needs);
 * switching the gate on with the other kind returns SM_ERR_STATE (the look-ahead does not consult the network). */
int smenv_set_risk_gate(SmEnv* env, float threshold);
/* How the gate inside the step decides (risk_state_config 4, RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP_AND_BACKUP_TRAJECTORY,
 * safe_motions_base.py:1520-1592).  backup_steps = 0: by the risk network (default).  backup_steps = K > 0: by look-ahead:
 * per env range, before the real step, the range's state is copied into shadow buffers owned by the library, the shadow
 * episode clock is set to 0, and K + 1 steps without auto reset run on the copy: the proposed buf->actions, then K times
 * the backup policy's action (tensor cores, tanh mean head) for the shadow observation.  Sub-step i uses step counter
 * s + i (s = the real step's; the Human scene draws its policy noise from it, so that sub-step 0 equals the real step when
 * the action is kept).  An env is risky exactly when some sub-step ends its episode for a reason other than
 * SM_TERM_TRAJECTORY_LENGTH; the risk network is not consulted, so the threshold does not change the decision.  Risky envs
 * execute the backup policy's action for the real observation as with the network gate (float32 with smenv_set_gate_exact);
 * SM_INFO_RISK reports 0 or 1.  Applies only while the gate is on (smenv_set_risk_gate).  In the measurement mode the
 * sub-steps run untimed before the timed real step; smenv_counters includes their work.  The shadow buffers are allocated
 * by the first call with K > 0 (or smenv_set_risk_next_state) and freed by smenv_destroy.  SM_ERR_STATE if the backup
 * policy is not loaded or the next-state check is on. */
int smenv_set_risk_lookahead(SmEnv* env, int backup_steps);
/* The gate rates the simulated next state (risk_state_config 3, RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP) with a state
 * risk network, whose input is the risk observation alone.  enable = 1: per env range, before the real step, the range's
 * state is copied into the shadow buffers (those of the look-ahead) with its episode clock as it is, and one step without
 * auto reset runs the proposed buf->actions on the copy with the real step's counter (in the Human scene the human's policy
 * noise is that of the real step).  The risk is the state network's rating of the shadow's risk observation (tensor cores;
 * with smenv_set_gate_exact the rows within the band of the threshold re-rated in float32), set to 1 where the simulated
 * step ended its episode for a reason other than SM_TERM_TRAJECTORY_LENGTH (a kept action never ends its own step in a
 * collision).  risk >= threshold executes the backup policy's action for the real observation as with the network gate;
 * SM_INFO_RISK reports the risk.  Applies only while the gate is on (smenv_set_risk_gate).  In the measurement mode the
 * simulated step runs untimed before the timed real step; smenv_counters includes its work.  SM_ERR_STATE if the backup
 * policy is not loaded, the loaded risk network is not a state network or the look-ahead is on; enable = 0 with the gate
 * on and a state network loaded returns SM_ERR_STATE as well (the network gate cannot use that network). */
int smenv_set_risk_next_state(SmEnv* env, int enable);
/* Initial-backup-trajectory check of the start pool (risk_check_initial_backup_trajectory, observations.py:155-185).
 * A reset copies a start-pool entry into the env verbatim (robot and obstacle records; in the Human scene the paired human
 * start state and its stored braking trajectory), so the check is a property of the entry and runs once per entry when
 * the pool is filled.  backup_steps = K > 0: every entry is reset into the shadow buffers of smenv_set_risk_lookahead
 * (allocated here if needed) and the backup policy acts for K steps with the episode clock from 0, no auto reset and the
 * gate off; the entry fails when one of those steps ends its episode for a reason other than SM_TERM_TRAJECTORY_LENGTH.
 * The pool is checked in batches of at most num_envs entries; env i of a batch draws from the Philox streams of its pool
 * entry, with step counters of its own (the Human and Ball scenes are stochastic: a verdict is one sample).  The pool is
 * then partitioned stably -- passing entries first in their original order, failing entries after them -- and every reset
 * (smenv_reset, the auto reset of the step, the human's reset with it) draws from the passing entries only: rejection
 * sampling from the pool, with no per-step cost.  The real env's buffers, statistics and step counter are not touched.
 * The call checks the current pools if they are filled and every later smenv_fill_pools does the same; it synchronises
 * `stream` once per check.  SM_ERR_STATE without a loaded backup policy, or when no entry passes (the pool then stays in
 * its original order and resets draw from all of it).  backup_steps = 0 switches the check off: resets draw from the whole
 * pool again; the checked order stays until the next smenv_fill_pools, which restores the unchecked pool exactly. */
int smenv_set_initial_backup_check(SmEnv* env, int backup_steps, SmStream stream);
/* checked: the start-pool entries the check rated for the current pools (0 while the check is off or the pools are not
 * filled); passed: the leading entries resets draw from (the passing entries; the whole pool while the check is off). */
int smenv_initial_backup_check_counts(SmEnv* env, int* checked, int* passed);
/* Exact gate (default on): the tensor-core risk (fp16 operands) of the rows within `band` of the threshold is re-computed
 * in float32 on the CUDA cores before the decision, and the backup policy's action of the risky rows is computed in
 * float32 too, so that decisions and executed actions are those of a float32 evaluation of the shipped networks
 * (safe_motions_base.py:1597-1603, actions.py:328-333).  exact = 0: both networks on the tensor cores only.
 * band <= 0 keeps the current band (default 0.01; the fp16 error around the reference's thresholds is < 4e-3). */
int smenv_set_gate_exact(SmEnv* env, int exact, float band);
/* The loaded network `which` in float32 on the CUDA cores for n rows (parity hook of the exact gate): the first n_out
 * outputs of every row.  SM_ERR_STATE if the network is not loaded; SM_ERR_ARG if n_out exceeds its output count or
 * out_stride < n_out. */
int smenv_mlp_forward_exact(SmEnv* env, int which, const float* in0, int in0_w, const float* in1, int in1_w, float* out,
                            int out_stride, int n_out, int n, SmStream stream);
/* Writes the U(-1,1) actions smenv_step_random would use for the next step into buf->actions (so that the gate can be
 * applied to them; follow with smenv_step). */
int smenv_random_actions(SmEnv* env, const SmBuffers* buf, SmStream stream);

/* The agent: the policy that acts in the env (a task policy, or the backup policy as the agent), a Keras fcnet loaded
 * into slot SM_NET_AGENT with a tanh output layer of 2 n_joints outputs -- the means, then the log-std pre-activations t
 * (keras_fcnet_last_layer_activation.py:187-202).  smenv_set_agent_head sets the log_std_range of its head:
 * log_std = lo + (t + 1) / 2 (hi - lo); default -1.375 / 0.0 (the shipped human policy's params.json).  SM_ERR_ARG if
 * lo > hi. */
int smenv_set_agent_head(SmEnv* env, float log_std_lo, float log_std_hi);
/* One env step (as smenv_step) whose proposed actions come from the agent on buf->obs (the full observation, target-point
 * entries included).  Per env range, before everything else of the step: the agent's network on the tensor cores, then
 * its DiagGaussian head.  explore != 0: sample = mean + exp(log_std) eps, eps ~ N(0, 1) from the Philox stream (env index,
 * step counter, joint, 0xA6E7) -- the step counter is the one smenv_step_random would use -- and
 * logp = -1/2 sum eps^2 - sum log_std - n_joints/2 log(2 pi), RLlib's DiagGaussian log-likelihood of the UNCLIPPED sample
 * (summed over the joints in order, bit-reproducible).  explore = 0: sample = mean, logp = 0 (RLlib's convention for
 * explore=False).  buf->actions = clip(sample, -1, 1) (RLlib's clip_actions): with the risk gate on it is the proposal the
 * gate rates and keeps, as in smenv_step.  Optional device outputs (NULL: not written): sample_out [N][n_joints],
 * logp_out [N], dist_out [N][2 n_joints] = mean, log_std (RLlib's action_dist_inputs).  In the measurement mode the agent
 * runs untimed before the timed step.  SM_ERR_ARG if buf->obs or buf->actions is NULL; SM_ERR_STATE if no agent is
 * loaded, its input width is not the observation size or its output count is not 2 n_joints.  smenv_step_host does not
 * run the agent. */
int smenv_step_agent(SmEnv* env, const SmBuffers* buf, int auto_reset, int explore, float* sample_out, float* logp_out,
                     float* dist_out, SmStream stream);

/* Measured peaks of the FP32 and FP64 FMA pipes of `device` in TFLOP/s (a micro-benchmark of dependent-free FMA chains
 * on all SMs): the denominators of bench.py's roofline for the vector-pipe-bound kernels. */
int smenv_measure_fma_peaks(int device, double* tflops_fp32, double* tflops_fp64);

/* Host-only (no GPU needed): the support-direction table the GJK kernel would use for a convex hull of n <= 255
 * vertices (xyz, float32) at `res` cells per cube-map face edge (4, 8, 12 or 16).  Layout: cells[6 res res] = (word offset
 * of the list << 8 | candidates), then the lists (vertex indices, one byte each).  Returns the number of words, or a
 * negative status; out may be NULL to query the size.  smenv_debug_lut_cell is the cell of a direction.  Tests check
 * that the true support vertex of every direction is among the candidates of its cell. */
int smenv_debug_build_lut(const float* xyz, int n, int res, uint32_t* out, int capacity);
int smenv_debug_lut_cell(float dx, float dy, float dz, int res);

/* Bounding volumes of the human's braking-trajectory check as human_brake_plan_kernel reads them (frame coordinates,
 * margins included).  Link-group pair g: the pairs (a, b) with a in [gp_a0, gp_a0 + gp_na) on frame gp_fa and b in
 * [gp_b0, gp_b0 + gp_nb) on frame gp_fb (human frame index; -1 = world, i.e. the table).  Side A is covered by the capsule
 * of its arm frame (hf_*, arm frames 3, 4, 7, 8 in this order); side B by gp_sb / gp_srb (trunk, frame 0), by the box
 * gp_bmin / gp_bmax (table, world frame) or by its arm frame's capsule.  Against the table the kernel replaces an arm
 * capsule by two spheres of radius hf_cover_rad at 1/4 and 3/4 of its segment.  hf_rho[i][j]: a change of joint j by dq
 * moves every shape centre and both capsule end points of arm frame i by at most |dq| * hf_rho[i][j] (0 for the joints
 * that do not move the frame); the span pass inflates its volumes by these. */
typedef struct SmHumanBounds {
    int32_t n_gp;
    int32_t gp_fa[8], gp_fb[8], gp_a0[8], gp_na[8], gp_b0[8], gp_nb[8];
    float gp_ca[8][3], gp_ra[8], gp_cb[8][3], gp_rb[8];   /* bounding spheres of both sides */
    float gp_bmin[8][3], gp_bmax[8][3];                   /* box of side B */
    float gp_sa[8][6], gp_sra[8], gp_sb[8][6], gp_srb[8]; /* capsules of both sides: segment end points, radius */
    int32_t hf_s0[4], hf_sn[4];                           /* shape range of arm frame i */
    float hf_seg[4][6], hf_rad[4], hf_cover_rad[4];
    float hf_rho[4][8];
} SmHumanBounds;

/* Host-only (no GPU needed): the bounding volumes above for a scene with the human enabled, built by the same code as
 * smenv_create.  Returns SM_OK or a negative status (the scene is refused for the same reasons as by smenv_create). */
int smenv_debug_human_bounds(const SmScene* scene, SmHumanBounds* out);

/* Constants of the distance planning as distance_plan_kernel reads them, from the float32 vertices (frame coordinates).
 * Per shape: the bounding sphere (center, radius), the box of the core vertices (bmin, bmax), the vertex mean (centroid)
 * and the support-width table: the largest extent of the core about the centre in any direction of a cube-map cell
 * (cell of a direction: smenv_debug_lut_cell with res 8).  Per pair of the pair table (static pairs, self pairs, then per
 * obstacle, per mov_reward shape, per part): pair_tab = shape A | shape B << 12 | class << 24 | (B is in frame 0: box
 * bound) << 31; pair_rm[0] = sum of the margins as the centroid upper bound subtracts it, pair_rm[1] = what the sphere or
 * box lower bound subtracts.  self_query: self-collision pairs farther apart are pruned. */
#define SM_PLAN_HWIDTH_CELLS 384   /* 6 cube-map faces x 8 x 8 cells */
#define SM_PLAN_MAX_PAIRS 512
typedef struct SmPlanBounds {
    int32_t n_shapes, n_pairs_fixed, n_pairs;
    double self_query;
    float center[SM_MAX_SHAPES][3], radius[SM_MAX_SHAPES];
    float bmin[SM_MAX_SHAPES][3], bmax[SM_MAX_SHAPES][3], centroid[SM_MAX_SHAPES][3];
    uint32_t pair_tab[SM_PLAN_MAX_PAIRS];
    float pair_rm[SM_PLAN_MAX_PAIRS][2];
    float hwidth[SM_MAX_SHAPES][SM_PLAN_HWIDTH_CELLS];
} SmPlanBounds;

/* Host-only (no GPU needed): the constants above for a scene, built by the same code as smenv_create.  Returns SM_OK or a
 * negative status (the scene is refused for the same reasons as by smenv_create). */
int smenv_debug_plan_bounds(const SmScene* scene, SmPlanBounds* out);

/* Debug: trace of one GJK call between shapes ia and ib for one env state given on the host (trace: 32 x 8 floats per
 * iteration = simplex size, |v|^2, v.w, support ids, v; result: distance, iterations, then the 9 robot frames). */
int smenv_debug_gjk(SmEnv* env, const double* kin_host, const double* obst_host, int ia, int ib, float upper,
                    float* trace_host, float* result_host);

#ifdef __cplusplus
}
#endif
#endif /* SMENV_H */
