// smenv_device.cuh -- device-side building blocks of the env-step kernels (sm_100a).
//
// Layout of the work: ONE WARP PER ENVIRONMENT.
//   * float64 joint-space maths (safe range, action mapping, interpolation, motor tracking) runs on lanes 0..n_joints-1
//     with explicit round-to-nearest intrinsics (no FMA contraction), so the joint trajectory is bit-identical to a
//     strict IEEE evaluation on the host;
//   * float32 geometry (forward kinematics, GJK) is warp-cooperative: the 32 lanes split the hull vertices of a
//     support search (vertices live in shared memory as float4) and reduce with one REDUX + ballot;
//   * the 24 physics sub-steps of one env step are mapped to lanes for the broad phase (lane k = sub-step k).
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "../../include/smenv.h"

#define FULL 0xffffffffu
#define SM_BIG 1.0e6

// ------------------------------------------------------------------------------------------------------------------
// scene constants on the device
// ------------------------------------------------------------------------------------------------------------------
struct DevShape {
    int frame, off, cnt, link;
    float margin, cx, cy, cz, radius;
    float bmin[3], bmax[3];  // axis-aligned box of the core vertices in frame coordinates
    float gx, gy, gz;        // centroid of the vertices: a point inside the hull (upper bounds of pair distances)
    int lut;                 // word offset of the shape's support-direction table in DevScene.lut, -1 = none
    int hw;                  // offset of the shape's support-width table in DevScene.hwidth (6 R R floats)
};

// Support-direction table ("LUT") of a hull: the unit sphere of directions is cut into 6 * SM_LUT_RES^2 cube-map
// cells; per cell the table lists every vertex that is the support point for SOME direction of the cell, so that a
// support query only scans that list (~20 of 252 vertices of an iiwa link).  Layout at word offset `lut`:
//   cells[6 R R]  : (word offset of the list relative to `lut`) << 8 | number of candidates
//   lists         : candidate vertex indices (local to the shape), one byte each, four per word, padded to a word
//                   boundary by repeating the last candidate
#define SM_MAX_PLAN_PAIRS 512 /* entries of the per-env pair table of the distance planning */
#ifndef SM_LUT_RES
#define SM_LUT_RES 8
#endif
#define SM_LUT_MIN_VERTS 33 /* smaller hulls are scanned directly */

// cell of direction d on a cube map with res x res cells per face
__host__ __device__ __forceinline__ int lut_cell_res(float dx, float dy, float dz, int res) {
    const float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
    int face;
    float m, u, w;
    if (ax >= ay && ax >= az) { face = dx > 0.0f ? 0 : 1; m = ax; u = dy; w = dz; }
    else if (ay >= az) { face = dy > 0.0f ? 2 : 3; m = ay; u = dz; w = dx; }
    else { face = dz > 0.0f ? 4 : 5; m = az; u = dx; w = dy; }
    const float half = 0.5f * (float)res;
    const float s = half / m;
    int iu = (int)(u * s + half), iw = (int)(w * s + half);
    iu = iu < 0 ? 0 : (iu > res - 1 ? res - 1 : iu);
    iw = iw < 0 ? 0 : (iw > res - 1 ? res - 1 : iw);
    return (face * res + iu) * res + iw;
}
__host__ __device__ __forceinline__ int lut_cell(float dx, float dy, float dz) { return lut_cell_res(dx, dy, dz, SM_LUT_RES); }
// DevShape.lut: word offset of the table | resolution code << 29: the cells per cube-map face edge are 8 (code 0), 4 (1:
// small hulls), 12 (2) or 16 (3: big hulls of scenes whose tables fit into shared memory at that resolution)
#define SM_LUT_RES_SHIFT 29
#define SM_LUT_OFF_MASK 0x1fffffff
#define SM_LUT_COARSE (1 << SM_LUT_RES_SHIFT)
#define SM_LUT_RES_COARSE 4
__host__ __device__ __forceinline__ int lut_res_of(int lut) {
    const int code = (lut >> SM_LUT_RES_SHIFT) & 3;
    return code == 0 ? SM_LUT_RES : code == 1 ? SM_LUT_RES_COARSE : code == 2 ? 12 : 16;
}
__host__ __device__ __forceinline__ int lut_code_of(int res) { return res == SM_LUT_RES ? 0 : res == SM_LUT_RES_COARSE ? 1 : res == 12 ? 2 : 3; }

// limits of one set of joints: the robot's, or the human's (nested env, ctlp.py:4647-4959)
struct JointLim {
    double pos_lo[SM_MAX_JOINTS], pos_hi[SM_MAX_JOINTS], vel_max[SM_MAX_JOINTS], acc_max[SM_MAX_JOINTS],
        jerk_max[SM_MAX_JOINTS];
    // 1 / (jerk_max ts) and 1 / (2 acc_max), rounded up: the conservative position-bound filter multiplies instead of
    // dividing (pos_bound_inactive; a filter, not part of any result)
    double inv_jts[SM_MAX_JOINTS], inv_2a[SM_MAX_JOINTS];
};

// the human obstacle (include/smenv.h SmHuman) as the kernels use it
#define SM_HGROUPS 5 /* human link groups of the coarse tests: trunk, upper arm / forearm + hand of each arm */
struct DevHuman {
    int enabled, n_joints, check_braking, brake_checks, n_brake_pairs, shape_off, n_arm_shapes, n_shapes;
    int initial_braking_trajectory;
    int joint_parent[SM_HUMAN_JOINTS];
    float baseR[9], baset[3];
    float jR[SM_HUMAN_JOINTS][9], jt[SM_HUMAN_JOINTS][3], jaxis[SM_HUMAN_JOINTS][3];
    JointLim lim;
    double brake_safety, brake_timeout, tp_radius, log_std_lo, log_std_hi;
    double tp_box_min[3], tp_box_max[3], tp_rel_min[3], tp_rel_max[3];
    double brake_t[8];                 // np.linspace(ts / C, ts, C) of the braking-trajectory check (ctlp.py:3166-3168)
    float tp_local[2][3];
    float tp_rho[2][4];                // bound on |d target link point of arm r / d q_(4 r + i)|
    const short* brake_pairs;          // device [n_brake_pairs][2]
    const float* contact_thresh;       // device [SM_MAX_HLINKS][SM_MAX_MOV_ROBOT]
    unsigned char shape_link[64];
    // link groups: the shapes of one human frame (frames 0, 3, 4, 7, 8 carry shapes), bounding sphere in frame coordinates
    int grp_frame[SM_HGROUPS], grp_off[SM_HGROUPS], grp_cnt[SM_HGROUPS];   // shape ranges are contiguous per group
    float grp_c[SM_HGROUPS][3], grp_r[SM_HGROUPS];
    float grp_rho[SM_HGROUPS][SM_HUMAN_JOINTS];   // bound on |d group centre / d q_j|
    float contact_thresh_max;
    float trunk_wmin[3], trunk_wmax[3];   // world box of the shapes in the base frame (the trunk does not move), margins included
    // braking-trajectory check: the pair list is sorted by (frame of A, frame of B); one entry per such link-group pair
    // with the bounding spheres of its two sides (frame coordinates; B in the world frame 0 is the table: its box is used)
    int n_gp;
    int gp_fa[8], gp_fb[8], gp_off[8], gp_cnt[8];
    float gp_ca[8][3], gp_ra[8], gp_cb[8][3], gp_rb[8];
    float gp_bmin[8][3], gp_bmax[8][3];   // B in frame 0: axis-aligned box of its core vertices (+ margin)
    // capsules (segment + radius, frame coordinates, margins included) around the two sides: the arm groups are long and
    // thin, a capsule is several times tighter than their bounding sphere
    float gp_sa[8][6], gp_sra[8], gp_sb[8][6], gp_srb[8];
    // the pairs of a link-group pair are the cross product of two contiguous shape ranges (checked by smenv_create)
    int gp_a0[8], gp_na[8], gp_b0[8], gp_nb[8];
    // arm frames 3, 4, 7, 8 (index 0..3): their contiguous shape range and a capsule around all of it (frame coordinates)
    int hf_s0[4], hf_sn[4];
    float hf_seg[4][6], hf_rad[4];
    float hf_rho[4][SM_HUMAN_JOINTS];     // bound on |d point of arm frame i / d q_j| over its shape centres and capsule ends
    double start_box_min[3], start_box_max[3], kinematic_sampling_probability, stay_in_state_probability,
        min_start_static, min_start_self, tp_min_static, tp_min_self;
};

struct DevScene {
    int n_joints, substeps, contact_stride, limit_velocity, limit_position;
    int joint_parent[SM_MAX_JOINTS];
    float jR[SM_MAX_JOINTS][9], jt[SM_MAX_JOINTS][3], jaxis[SM_MAX_JOINTS][3];
    int jr_identity;   // bit j: the fixed rotation of joint j is exactly the identity (all iiwa joints: rpy = 0)
    union {
        struct {
            double pos_lo[SM_MAX_JOINTS], pos_hi[SM_MAX_JOINTS], vel_max[SM_MAX_JOINTS], acc_max[SM_MAX_JOINTS],
                jerk_max[SM_MAX_JOINTS];
        };
        JointLim lim;   // the same five arrays as one record
    };
    double ts, action_mapping_factor, track_kp, track_vel;
    double sub_t[33];  // np.linspace(ts / S, ts, S)[k - 1] at index k (actions.py:420-421), computed on the host
    int n_shapes, n_verts;
    DevShape shapes[SM_MAX_SHAPES];
    int n_static_pairs, n_self_pairs, n_mov_reward, n_mov_contact;
    int contact_frame_start[SM_MAX_JOINTS + 2];  // mov_contact slots sorted by frame: slots of frame f
    short static_pairs[SM_MAX_PAIRS][2], self_pairs[SM_MAX_PAIRS][2];
    short mov_reward[SM_MAX_MOV_ROBOT], mov_contact[SM_MAX_MOV_ROBOT];
    int n_obstacles;
    int obst_kind[SM_MAX_OBSTACLES], obst_shape_off[SM_MAX_OBSTACLES], obst_shape_cnt[SM_MAX_OBSTACLES];
    float obst_center[SM_MAX_OBSTACLES][3], obst_radius[SM_MAX_OBSTACLES];
    float contact_thresh[SM_MAX_OBSTACLES][SM_MAX_MOV_ROBOT];
    float contact_thresh_max[SM_MAX_OBSTACLES];
    float obst_bmin[SM_MAX_OBSTACLES][3], obst_bmax[SM_MAX_OBSTACLES][3];  // box of all parts (cores + margins), body frame
    float obst_center_norm[SM_MAX_OBSTACLES];              // |obst_center|: sphere about the body origin instead
    float contact_rho[SM_MAX_MOV_ROBOT][SM_MAX_JOINTS];    // bound on |d centre(slot) / d q_j| (coarse contact phase)
    int planet_steps, planet_shift, obs_planet_size;
    const float4* planet_pos[SM_MAX_OBSTACLES];   // xyz, w unused
    const float4* planet_quat[SM_MAX_OBSTACLES];  // xyzw
    const double* planet_local_xy;
    double planet_obs_half[2];
    double ball_obs_pos_min[3], ball_obs_pos_max[3], ball_obs_vel_min[3], ball_obs_vel_max[3];
    double ball_active_xy;
    double static_cap, moving_query, collision_dist;
    double self_query;   // self-collision distances above it cannot change reward or termination: such pairs are pruned and
                         // the class reports the cap (min(static_cap, reward distance of the self-collision term))
    double w_self, w_static, w_moving, d_self, d_static, d_moving, w_low_acc, thr_low_acc, w_low_vel, thr_low_vel;
    int punish_action, terminate_self, terminate_static, terminate_moving;
    double action_thresh, action_max_punishment, termination_bonus, early_termination_punishment, reward_scale;
    int episode_steps, obs_size;
    // sampling
    double start_box_min[3], start_box_max[3];
    float target_offset[3], target_R[9], target_t[3];
    double kinematic_sampling_probability, stay_in_state_probability, min_start_distance;
    double ball_sphere_center[3], ball_sphere_radius, ball_height_min, ball_height_max, ball_angle_min, ball_angle_max;
    double ball_speed, ball_radius, ball_high_angle_probability;
    double ball_target_box_min[3], ball_target_box_max[3], ball_invalid_min[3], ball_invalid_max[3];
    double ball_final_min[3], ball_final_max[3], plane_z;
    int ball_check_invalid, ball_random_initial, has_table;
    double min_start_self, ball_target_min_static, ball_target_min_self;
    const float4* verts;  // device, n_verts
    // pair list of the distance planning: static pairs, self pairs, then (observed link shape x obstacle part) per
    // moving obstacle; entry = shape A | shape B << 12 | class << 24
    int n_pairs_fixed, n_pairs;
    uint32_t pair_tab[SM_MAX_PLAN_PAIRS];
    float2 pair_rm[SM_MAX_PLAN_PAIRS];   // host copies for the SceneImage (layout: smenv_geom.cuh)
    // support-width tables: per shape and cube-map cell an upper bound of h(d) = max_v (v - centre) . d over the unit
    // directions d of the cell.  centre distance - h_A(d) - h_B(-d) along the line of centres is a lower bound of the
    // pair distance that is far tighter than bounding spheres for elongated hulls (planning kernels).
    // target points of the reaching task (include/smenv.h)
    int use_target_points, tp_normalize, obs_add_tp_pos, obs_add_tp_rel, start_at_rest;
    double tp_radius, tp_bonus, tp_reward_factor, tp_box_min[3], tp_box_max[3], tp_rel_min[3], tp_rel_max[3];
    double tp_min_static, tp_min_self;
    float tp_local[3];               // target link point in the frame of the last joint
    float tp_rho[SM_MAX_JOINTS];     // bound on |d target link point / d q_j|
    const uint4* scene_img;  // device image of the tables every geometry CTA stages into shared memory (SceneImage)
    const float* hwidth;  // device
    const uint32_t* lut;  // device, n_lut_words (support-direction tables of all shapes that have one)
    int n_lut_words;
    DevHuman hu;
};

// the library is one translation unit (smenv.cu), so the constant-memory scene is defined here
__constant__ DevScene c_sc;

// ------------------------------------------------------------------------------------------------------------------
// mbarrier / 1-D bulk TMA helpers (sm_90+ PTX): one thread issues cp.async.bulk copies that complete on an mbarrier
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}\n"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}


// ------------------------------------------------------------------------------------------------------------------
// strict IEEE float64 helpers: never contracted into FMA, same rounding as the host evaluating one operation at a time
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double xadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double xmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xdiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double xsqrt(double a) { return __dsqrt_rn(a); }

// ------------------------------------------------------------------------------------------------------------------
// 1. safe acceleration range (actions.py:97-106, :206-211 -> klimits.PosVelJerkLimitation; model in DESIGN.md)
// ------------------------------------------------------------------------------------------------------------------
enum { CODE_VEL_HI = 1, CODE_VEL_LO = 2, CODE_POS_HI = 4, CODE_POS_LO = 8, CODE_ACC = 16 };

// largest next-knot acceleration that keeps the velocity peak under vmax when braking as hard as allowed afterwards
__device__ __noinline__ double vel_upper(double v0, double a0, double vmax, double J, double A, double ts) {
    double c = xsub(xadd(v0, xmul(xmul(a0, ts), 0.5)), vmax);
    if (c > 0.0) {
        double den = xsub(vmax, v0);
        if (a0 <= 0.0 || den <= 0.0) return -SM_BIG;
        return xsub(a0, xdiv(xmul(xmul(a0, a0), ts), xmul(2.0, den)));
    }
    double a1u = xmul(J, xsub(xsqrt(xsub(xmul(xmul(ts, ts), 0.25), xdiv(xmul(2.0, c), J))), xmul(ts, 0.5)));
    double JT = xmul(J, ts);
    double delta = xsub(JT, A);
    if (delta <= 0.0) return a1u;
    double n = xsub(ceil(xdiv(a1u, JT)), 1.0);
    if (n < 0.0) n = 0.0;
    double x = xsub(a1u, xmul(n, JT));
    if (x >= delta) return a1u;
    double C = xadd(c, xmul(xmul(xmul(xmul(JT, ts), n), xadd(n, 1.0)), 0.5));
    double D = xmul(ts, xadd(n, 0.5));
    double qa = xadd(D, xmul(ts, 0.5)), qb = xadd(C, xmul(D, A)), qc = xmul(C, A);
    x = xdiv(xsub(xsqrt(xsub(xmul(qb, qb), xmul(xmul(4.0, qa), qc))), qb), xmul(2.0, qa));
    return xadd(xmul(n, JT), x);
}

// highest position reached when the next knot acceleration is a1 and the hardest admissible braking follows; with
// DERIV also its derivative with respect to a1 (the state derivatives ride along the simulated profile; an interior
// peak is a stationary point of the position, so its derivative is taken at fixed tau)
template <bool DERIV>
__device__ __forceinline__ double pos_peak_impl(double p, double v, double a, double a1, double J, double A, double ts,
                                                double& dbest) {
    double best = p;
    double an = a1;
    double dp = 0.0, dv = 0.0, da = 0.0, dan = 1.0;
    dbest = 0.0;
    for (int it = 0; it < 16; ++it) {
        double j = xdiv(xsub(an, a), ts);
        double dj = DERIV ? xdiv(xsub(dan, da), ts) : 0.0;
        double tau = -1.0;
        if (j == 0.0) {
            if (a < 0.0 && v > 0.0) tau = xdiv(-v, a);
        } else {
            double disc = xsub(xmul(a, a), xmul(xmul(2.0, j), v));
            if (disc >= 0.0) {
                double s = xsqrt(disc);
                if (a <= 0.0) {
                    if (xsub(s, a) > 0.0) tau = xdiv(xmul(2.0, v), xsub(s, a));
                } else {
                    tau = xdiv(xsub(-a, s), j);
                }
            }
        }
        if (tau > 0.0 && tau <= ts) {
            // p + v*tau + 0.5*a*tau*tau + (j*tau*tau*tau)/6.0, left to right
            double pk = xadd(xadd(xadd(p, xmul(v, tau)), xmul(xmul(xmul(0.5, a), tau), tau)),
                             xdiv(xmul(xmul(xmul(j, tau), tau), tau), 6.0));
            if (pk > best) {
                best = pk;
                if (DERIV)
                    dbest = xadd(xadd(xadd(dp, xmul(dv, tau)), xmul(xmul(xmul(0.5, da), tau), tau)),
                                 xdiv(xmul(xmul(xmul(dj, tau), tau), tau), 6.0));
            }
        }
        double pn = xadd(xadd(p, xmul(v, ts)), xmul(xmul(xadd(xdiv(a, 3.0), xdiv(an, 6.0)), ts), ts));
        double vn = xadd(v, xmul(xmul(xadd(a, an), ts), 0.5));
        if (DERIV) {
            double dpn = xadd(xadd(dp, xmul(dv, ts)), xmul(xmul(xadd(xdiv(da, 3.0), xdiv(dan, 6.0)), ts), ts));
            double dvn = xadd(dv, xmul(xmul(xadd(da, dan), ts), 0.5));
            dp = dpn; dv = dvn; da = dan;
        }
        p = pn; v = vn; a = an;
        if (p > best) { best = p; if (DERIV) dbest = dp; }
        if (a <= -A) {
            if (v > 0.0) {
                double pk = xadd(p, xdiv(xmul(v, v), xmul(2.0, A)));
                if (pk > best) { best = pk; if (DERIV) dbest = xadd(dp, xdiv(xmul(v, dv), A)); }
            }
            break;
        }
        if (v <= 0.0 && a <= 0.0) break;
        an = xsub(a, xmul(J, ts));
        if (an < -A) { an = -A; dan = 0.0; }
    }
    return best;
}
__device__ __noinline__ double pos_peak(double p, double v, double a, double a1, double J, double A, double ts) {
    double d;
    return pos_peak_impl<false>(p, v, a, a1, J, A, ts, d);
}
__device__ __noinline__ double pos_peak_d(double p, double v, double a, double a1, double J, double A, double ts,
                                          double& dbest) {
    return pos_peak_impl<true>(p, v, a, a1, J, A, ts, dbest);
}

// pos_upper in two halves (the same operations in the same order): the first evaluation decides whether the bound is
// active at all, the second half is the iterative solve.  joint_heavy_kernel runs the halves in separate phases so
// that the solve executes with densely packed lanes.
__device__ __forceinline__ double pos_upper_first(double p, double v, double a, double pmax, double hi, double J,
                                                  double A, double ts) {
    return xsub(pos_peak(p, v, a, hi, J, A, ts), pmax);
}
// Acceptance window of the position-bound solve: a safe a1 (peak <= pmax) whose peak comes within this many rad of the
// limit ends the search.
#define SM_POS_SOLVE_TOL 1e-10
__device__ __noinline__ double pos_upper_rest(double p, double v, double a, double pmax, double lo, double hi, double J,
                                              double A, double ts, double fr);

__device__ __noinline__ double pos_upper(double p, double v, double a, double pmax, double lo, double hi, double J, double A,
                            double ts) {
    double fr = pos_upper_first(p, v, a, pmax, hi, J, A, ts);
    if (fr <= 0.0) return SM_BIG;
    return pos_upper_rest(p, v, a, pmax, lo, hi, J, A, ts, fr);
}

// The peak is an increasing, piecewise smooth, mostly convex function of a1: safeguarded Newton with the exact
// derivative, aimed at the middle of the acceptance window and started from the secant of the bracket; a step that
// leaves the bracket (flat stretches, kinks) is replaced by a bisection.  Mean 5 evaluations, at most 11 seen (a regula
// falsi needed 8 on average and up to 26; joint_solve_kernel runs 32 solves per warp in lockstep, so the longest one
// sets the time).
__device__ __noinline__ double pos_upper_rest(double p, double v, double a, double pmax, double lo, double hi, double J,
                                              double A, double ts, double fr) {
    double fl = xsub(pos_peak(p, v, a, lo, J, A, ts), pmax);
    if (fl > 0.0) return fl > 1e-6 ? -SM_BIG : lo;
    double xl = lo, xr = hi;
    double x = xsub(xr, xdiv(xmul(fr, xsub(xr, xl)), xsub(fr, fl)));
    if (!(x > xl && x < xr)) x = xmul(0.5, xadd(xl, xr));
    for (int it = 0; it < 40; ++it) {
        double df;
        double f = xsub(pos_peak_d(p, v, a, x, J, A, ts, df), pmax);
        if (f <= 0.0 && f > -SM_POS_SOLVE_TOL) return x;
        if (f <= 0.0) xl = x; else xr = x;
        if (xsub(xr, xl) <= 1e-9) break;
        double xn = xl;
        if (df > 0.0) xn = xsub(x, xdiv(xadd(f, 0.5 * SM_POS_SOLVE_TOL), df));
        if (!(xn > xl && xn < xr)) xn = xmul(0.5, xadd(xl, xr));
        x = xn;
    }
    return xl;
}

__device__ __forceinline__ void clamp_range(double& lo, double& hi, double blo, double bhi, int code_hi, int code_lo,
                                            int& code) {
    double nhi = hi < bhi ? hi : bhi;
    double nlo = lo > blo ? lo : blo;
    if (nhi < lo) { if (xsub(lo, nhi) > 1e-6) code |= code_hi; nhi = lo; }
    if (nlo > hi) { if (xsub(nlo, hi) > 1e-6) code |= code_lo; nlo = hi; }
    if (nlo > nhi) { if (xsub(nlo, nhi) > 1e-6) code |= code_hi | code_lo; nlo = nhi; }
    lo = nlo; hi = nhi;
}

// Conservative test "the position bound of pos_upper is inactive": true only if pos_peak(p, v, a, a1 = hi) is
// certainly below pmax, in which case pos_upper returns SM_BIG after its first evaluation and the whole iterative
// solve can be skipped without changing a bit of the result.  Bound on the braking trajectory pos_peak simulates:
//   interval 1:  p(t) <= p + v+ ts + m0 ts^2 / 2,  v1 <= v + m0 ts            (m0 = max(a, a1, 0))
//   ramp to -A:  n = ceil((a1+ + A) / (J ts)) + 1 intervals with acceleration <= a1+
//   velocity along the profile <= vp = min(v1 + a1+ n ts, 1.001 V + 1e-6)     (the velocity clamp already applied
//                                                                              to hi guarantees the second term)
//   then constant -A: stopping distance <= vp^2 / (2A)
// Everything is rounded up by a 1e-6 rad slack; plain double arithmetic (this is a filter, not part of the result).
__device__ __forceinline__ bool pos_bound_inactive(double p, double v, double a, double a1, double pmax, double inv_jts,
                                                   double inv_2a, double A, double V, double ts, bool vel_guaranteed) {
    const double m0 = fmax(fmax(a, a1), 0.0), a1p = fmax(a1, 0.0), vp0 = fmax(v, 0.0);
    const double n = ceil((a1p + A) * inv_jts) + 1.0;    // inv_jts >= 1 / (J ts): n is not below the exact count
    double w = fmax(v + m0 * ts, 0.0) + a1p * n * ts;
    if (vel_guaranteed) w = fmin(w, 1.001 * V + 1e-6);
    w = fmax(w, vp0);
    const double bound = p + vp0 * ts + 0.5 * m0 * ts * ts + w * n * ts + w * w * inv_2a;
    return bound + 1e-6 < pmax;
}

// Cheap part of the range: jerk, acceleration and velocity bounds.  Returns through need_pos whether one of the two
// position bounds may be active (then safe_range_joint has to run the iterative solve).
__device__ __forceinline__ void safe_range_light(const JointLim& L, int j, double p, double v, double a, double& lo,
                                                 double& hi, int& code, bool& need_pos) {
    double ts = c_sc.ts, J = L.jerk_max[j], A = L.acc_max[j], V = L.vel_max[j];
    code = 0;
    lo = xsub(a, xmul(J, ts)); hi = xadd(a, xmul(J, ts));
    if (lo < -A) lo = -A;
    if (hi > A) hi = A;
    if (lo > hi) {
        code |= CODE_ACC;
        if (a > 0.0) lo = hi; else hi = lo;
    }
    if (c_sc.limit_velocity) {
        double bhi = vel_upper(v, a, V, J, A, ts);
        double blo = -vel_upper(-v, -a, V, J, A, ts);
        clamp_range(lo, hi, blo, bhi, CODE_VEL_HI, CODE_VEL_LO, code);
    }
    need_pos = false;
    if (c_sc.limit_position) {
        const bool vg = c_sc.limit_velocity && code == 0 && fabs(v) <= V;
        need_pos = !(pos_bound_inactive(p, v, a, hi, L.pos_hi[j], L.inv_jts[j], L.inv_2a[j], A, V, ts, vg) &&
                     pos_bound_inactive(-p, -v, -a, -lo, -L.pos_lo[j], L.inv_jts[j], L.inv_2a[j], A, V, ts, vg));
    }
}
__device__ __forceinline__ void safe_range_light(int j, double p, double v, double a, double& lo, double& hi, int& code,
                                                 bool& need_pos) {
    safe_range_light(c_sc.lim, j, p, v, a, lo, hi, code, need_pos);
}

__device__ void safe_range_joint(const JointLim& L, int j, double p, double v, double a, double& out_lo, double& out_hi,
                                 int& out_code) {
    double ts = c_sc.ts, J = L.jerk_max[j], A = L.acc_max[j], V = L.vel_max[j];
    int code = 0;
    double lo = xsub(a, xmul(J, ts)), hi = xadd(a, xmul(J, ts));
    if (lo < -A) lo = -A;
    if (hi > A) hi = A;
    if (lo > hi) {
        code |= CODE_ACC;
        if (a > 0.0) lo = hi; else hi = lo;
    }
    if (c_sc.limit_velocity) {
        double bhi = vel_upper(v, a, V, J, A, ts);
        double blo = -vel_upper(-v, -a, V, J, A, ts);
        clamp_range(lo, hi, blo, bhi, CODE_VEL_HI, CODE_VEL_LO, code);
    }
    if (c_sc.limit_position) {
        double bhi = pos_upper(p, v, a, L.pos_hi[j], lo, hi, J, A, ts);
        double blo = -pos_upper(-p, -v, -a, -L.pos_lo[j], -hi, -lo, J, A, ts);
        clamp_range(lo, hi, blo, bhi, CODE_POS_HI, CODE_POS_LO, code);
    }
    out_lo = lo; out_hi = hi; out_code = code;
}
__device__ __forceinline__ void safe_range_joint(int j, double p, double v, double a, double& out_lo, double& out_hi,
                                                 int& out_code) {
    safe_range_joint(c_sc.lim, j, p, v, a, out_lo, out_hi, out_code);
}

// actions.py:268-280
__device__ __forceinline__ double map_action(double u, double lo, double hi) {
    if (c_sc.action_mapping_factor != 1.0) {
        double mf = xmul(0.5, xadd(c_sc.action_mapping_factor, 1.0));
        double diff = xsub(hi, lo);
        hi = xadd(lo, xmul(mf, diff));
        lo = xadd(lo, xmul(xsub(1.0, mf), diff));
    }
    return xadd(lo, xmul(xmul(0.5, xadd(u, 1.0)), xsub(hi, lo)));
}

// np.linspace(ts / S, ts, S)[k-1]  (actions.py:420-421)
__device__ __forceinline__ double substep_time(int k) {
    int S = c_sc.substeps;
    if (S <= 1 || k == S) return c_sc.ts;
    double start = xdiv(c_sc.ts, (double)S);
    double step = xdiv(xsub(c_sc.ts, start), (double)(S - 1));
    return xadd(start, xmul((double)(k - 1), step));
}

// actions.py:468-487
__device__ __forceinline__ void interpolate(double q0, double v0, double a0, double a1, double t, double& q,
                                            double& v, double& a) {
    double jerk = xdiv(xsub(a1, a0), c_sc.ts);
    a = xadd(a0, xmul(jerk, t));
    v = xadd(xadd(v0, xmul(a0, t)), xmul(xmul(xmul(0.5, jerk), t), t));
    q = xadd(xadd(xadd(q0, xmul(v0, t)), xmul(xmul(xmul(0.5, a0), t), t)),
             xmul(xmul(xmul(xmul(1.0 / 6.0, jerk), t), t), t));
}

// ------------------------------------------------------------------------------------------------------------------
// 2. Philox4x32-10 counter-based RNG (Salmon et al., SC'11)
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01f(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ double u01d(uint32_t hi, uint32_t lo) {
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) * (1.0 / 9007199254740992.0);
}

// One joint of the DiagGaussian head of a Keras-fcnet policy (keras_fcnet_last_layer_activation.py:187-202): the tanh
// output t of the log-std column is remapped to log_std = lo + (t + 1) / 2 * span (span = hi - lo, the log_std_range of
// params.json), eps ~ N(0, 1) by Box-Muller from the first two words of a Philox draw; returns the unclipped sample
// mean + exp(log_std) * eps.  Shared by the human's policy and the agent (the human's actions depend on its exact form).
__device__ __forceinline__ float diag_gaussian_sample(float mean, float t, float lo, float span, uint4 r, float& log_std,
                                                      float& eps) {
    log_std = lo + 0.5f * (t + 1.0f) * span;
    const float u1 = fmaxf(u01f(r.x), 5.9604645e-8f), u2 = u01f(r.y);
    eps = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);   // Box-Muller
    return mean + expf(log_std) * eps;
}

// per-warp sampling stream: every draw advances the counter; all lanes get the same numbers
struct Rng {
    uint32_t k0, k1, c0, c1, n;
    __device__ Rng(uint64_t seed, uint32_t a, uint32_t b) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), c0(a), c1(b), n(0) {}
    __device__ uint4 next4() { return philox(c0, c1, n++, 0x5afe, k0, k1); }
    __device__ double uniform() { uint4 r = next4(); return u01d(r.x, r.y); }
    __device__ double uniform(double lo, double hi) { return lo + (hi - lo) * uniform(); }
};

