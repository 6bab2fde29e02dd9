// smenv_human.cuh -- the Human scene (Human, ctlp.py:4647-4959): a nested SafeMotionsEnv(robot_scene = 9) moves the two
// arms of a human next to the robot (description/urdf/human.urdf:140-416, trained_networks/human_network/params.json).
//
// Per step of the main env, in launch order (smenv.cu step_range):
//   mlp_kernel (SM_NET_HUMAN)      the human's policy 38 -> 256 -> 128 -> 16 on the tensor cores        (smenv_mlp.cuh)
//   human_action_kernel            stochastic head: mean + exp(log_std) * eps, Philox normal noise, clipped
//                                  (keras_fcnet_last_layer_activation.py:187-202; explore = True, ctlp.py:4701)
//   joint_kernel .. joint_final    safe range of the 8 human joints and the mapped acceleration (set = 1, deferred advance)
//   human_brake_traj_kernel        braking trajectory that would follow the step, in joint space
//                                  (ctlp.py:3155-3207, :3467-3507; utils/braking_trajectory_generator.py:44-93)
//   human_brake_plan_kernel        span pass: one FK per run of HBP_SPAN poses, volumes inflated by the joint motion
//                                  inside the run; then the per-pose pass over the runs it could not clear: FK of
//                                  every such pose, bounding-volume culling -> GJK_BRAKE items
//   gjk_kernel                     "closer than the safety distance?" per item                             (smenv_gjk.cuh)
//   human_advance_kernel           adapt_action bookkeeping (ctlp.py:3055-3153, :3000-3024), 24 setpoints + tracked pose
//   human_outcome_kernel           target point reached? (ctlp.py:2787-2821), new knot bookkeeping, new target point from
//                                  the pool, observation of the nested env (observations.py:313-351)
//   hcontact_coarse / _plan        contacts robot <-> human at the 24 tracked sub-step poses -> GJK_CONTACT items
//                                  (ctlp.py:2613-2615, :4888-4898)
// The distance planning and the finish kernel of the main env take the human's frames / kinematic observation from the
// records written here.
#pragma once
#include "smenv_pools.cuh"
#include "smenv_step.cuh"

struct HumanArgs {
    SmBuffers buf;
    int n, env_base;
    uint32_t k0, k1, step_counter;
    uint32_t step_offset;      // added to *step_ptr: sub-step i of the look-ahead (smenv_set_risk_lookahead) draws with s + i
    const uint32_t* step_ptr;  // if set, the step counter is read from device memory instead (graph replays of the host step)
    const float* policy_out;   // [n][16] outputs of the human's policy (tanh), NULL: buf.hactions come from the caller
    double* range;             // [n][8][4] lo, hi, mapped acceleration of every human joint (joint kernels, deferred)
    double* bacc;              // [n][SM_HBRAKE_STEPS][8] braking accelerations of the trajectory under check
    float* poses;              // [n][SM_HBRAKE_POSES][8] poses the check visits
    int* binfo;                // [n][4] braking steps k, poses, timeout, reserved
    int* units;                // [0] = count, [1..] = hbp_unit(env, first pose, poses): the spans of poses the braking-trajectory
                               // check has to test (human_brake_plan_kernel<true>), or the single poses (<false>)
    int* fine;                 // [0] = count, [1..] = hbp_unit(env, pose, 1): the poses of the spans the span pass could not clear
    float* hscratch;           // [n][SM_SCRATCH_FLOATS] sub-step poses of the human (tracked, setpoints)
    const float* scratch;      // [n][SM_SCRATCH_FLOATS] sub-step poses of the robot
    GjkItem* items;
    int* item_count;
    int capacity;
    int* overflow;
    unsigned* res;             // [n][SM_RES_STRIDE]
    const double* target_pool; // [2][target_pool_n][4] target points per arm
    int target_pool_n;
    const double* start_pool;  // [start_pool_n][SM_HPOOL_STRIDE] start states of the nested env
    int start_pool_n;
    const double* pool_brake;  // [start_pool_n][SM_HBRAKE_STEPS][8] initial braking trajectory of every start state, NULL: computed
    const int* pool_bcount;    // [start_pool_n] its number of steps
    int* cwork;                // contact planning: [0] = count, [1..] = env * 8 + span
    const uint8_t* mask;       // reset: envs to reset (NULL = by done flag / all)
    unsigned long long* counters;
    const int* entry;          // reset: [n] pool entry of env i (the pool check, smenv_set_initial_backup_check), NULL: drawn
};

// ------------------------------------------------------------------------------------------------------------------
// the human's stochastic policy head (keras_fcnet_last_layer_activation.py:187-202; RLlib clips actions to [-1, 1])
// ------------------------------------------------------------------------------------------------------------------
__global__ void human_action_kernel(HumanArgs A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int env = t >> 3, j = t & 7;
    if (env >= A.n) return;
    const float* o = A.policy_out + (size_t)env * 16;
    const float mean = o[j], t_log_std = o[8 + j];
    const uint32_t step = A.step_ptr ? __ldg(A.step_ptr) + A.step_offset : A.step_counter;
    const uint4 r = philox((uint32_t)(env + A.env_base), step, (uint32_t)j, 0x4057u, A.k0, A.k1);
    float log_std, eps;
    const float sample = diag_gaussian_sample(mean, t_log_std, (float)c_sc.hu.log_std_lo,
                                              (float)(c_sc.hu.log_std_hi - c_sc.hu.log_std_lo), r, log_std, eps);
    A.buf.hactions[(size_t)env * SM_HUMAN_JOINTS + j] = fminf(1.0f, fmaxf(-1.0f, sample));
}

// ------------------------------------------------------------------------------------------------------------------
// braking trajectory of the nested env in joint space: thread = (env, joint), the eight lanes of an env in lockstep
// ------------------------------------------------------------------------------------------------------------------
// BrakingTrajectoryGenerator.get_braking_acceleration for one joint: the next acceleration from which the acceleration
// can be ramped back to zero at full jerk, in whole time steps, so that velocity and acceleration reach zero together
// (same operations as brake_target of the oracle)
__device__ __forceinline__ double brake_target(double v, double a, double J, double Am, double ts) {
    const double s0 = xadd(v, xmul(xmul(a, ts), 0.5));
    const double sg = s0 < 0.0 ? -1.0 : 1.0;
    const double S = sg * s0, r = xmul(J, ts);
    double a1 = 0.0;
#pragma unroll 1
    for (int n = 1; n <= 8; ++n) {
        const double dn = (double)n;
        a1 = xdiv(xadd(S, xmul(xmul(xmul(xmul(ts, r), dn), xsub(dn, 1.0)), 0.5)), xmul(dn, ts));
        if (a1 <= xmul(dn, r)) break;
    }
    a1 = -sg * a1;
    double lo = xsub(a, xmul(J, ts)), hi = xadd(a, xmul(J, ts));
    if (lo < -Am) lo = -Am;
    if (hi > Am) hi = Am;
    if (lo > hi) { if (a > 0.0) lo = hi; else hi = lo; }
    if (a1 < lo) a1 = lo;
    if (a1 > hi) a1 = hi;
    return a1;
}

// _compute_braking_acceleration for one joint (ctlp.py:3495-3507): brake_target clipped to the full safe range, which is
// evaluated lazily like the oracle's human_braking_acceleration (the iterative position bounds only if the braking profile
// that follows the clipped value would leave a position limit)
__device__ __forceinline__ double human_braking_acceleration(const JointLim& L, int j, double p, double v, double a, bool small_j) {
    const double ts = c_sc.ts, J = L.jerk_max[j], Am = L.acc_max[j];
    double lo, hi;
    int code;
    bool need_pos;
    safe_range_light(L, j, p, v, a, lo, hi, code, need_pos);
    const double e0 = small_j ? 0.0 : brake_target(v, a, J, Am, ts);
    double e = e0;
    if (e < lo) e = lo;
    if (e > hi) e = hi;
    if (need_pos) {
        const double V = L.vel_max[j];
        const bool ok_hi = pos_bound_inactive(p, v, a, e, L.pos_hi[j], L.inv_jts[j], L.inv_2a[j], Am, V, ts, false) ||
                           xsub(pos_peak(p, v, a, e, J, Am, ts), L.pos_hi[j]) <= 0.0;
        const bool ok_lo = pos_bound_inactive(-p, -v, -a, -e, -L.pos_lo[j], L.inv_jts[j], L.inv_2a[j], Am, V, ts, false) ||
                           xsub(pos_peak(-p, -v, -a, -e, J, Am, ts), -L.pos_lo[j]) <= 0.0;
        if (!(ok_hi && ok_lo)) {
            safe_range_joint(L, j, p, v, a, lo, hi, code);
            e = e0;
            if (e < lo) e = lo;
            if (e > hi) e = hi;
        }
    }
    return e;
}

#ifndef HBP_SPAN
#define HBP_SPAN 3   /* consecutive poses of a braking trajectory the span pass of human_brake_plan_kernel tests at once */
#endif
static_assert(HBP_SPAN >= 1 && HBP_SPAN <= 8, "the unit word holds the pose count of a span in 3 bits");
static_assert(SM_HBRAKE_POSES <= 128, "the unit word holds the first pose of a span in 7 bits");
// unit of the braking-trajectory geometry pass: env in the upper 22 bits, n - 1 in bits 7..9, the first pose in bits 0..6
#define HBP_MAX_ENVS (1 << 22)
__host__ __device__ __forceinline__ int hbp_unit(int env, int p0, int n) {
    return (int)(((unsigned)env << 10) | ((unsigned)(n - 1) << 7) | (unsigned)p0);
}

#ifndef HBT_MIN_BLOCKS
#define HBT_MIN_BLOCKS 8   /* resident CTAs per SM the register allocation aims for: 64 registers and 220 B of spill, but 32
                              warps instead of 16 hide the FP64 latency chains (Human step 1547 -> 1483 us; 5, 6: no gain, 10, 12: worse) */
#endif
__global__ void __launch_bounds__(128, HBT_MIN_BLOCKS) human_brake_traj_kernel(HumanArgs A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int env_raw = t >> 3, j = t & 7;
    const bool valid = env_raw < A.n;
    const size_t env = valid ? (size_t)env_raw : (size_t)(A.n - 1);
    const JointLim& L = c_sc.hu.lim;
    const double ts = c_sc.ts, J = L.jerk_max[j], Am = L.acc_max[j];
    const int C = c_sc.hu.brake_checks;
    const double* kin = A.buf.hkin + env * SM_KIN_STRIDE;
    double q = kin[j], v = kin[8 + j], as = kin[16 + j], ae = A.range[(env * 8 + j) * 4 + 2];
    float* poses = A.poses + env * SM_HBRAKE_POSES * 8;
    double* bacc = A.bacc + env * SM_HBRAKE_STEPS * 8;
    int k = 0, np = 0, timeout = 0;
    bool done = !valid || !c_sc.hu.check_braking;
    const int gsh = lane & 24;   // first lane of this env's group of eight
#pragma unroll 1
    while (true) {
        double pend = q, vend = v;
        bool small_j = true;
        if (!done) {
#pragma unroll 1
            for (int m = 1; m <= C; ++m) {   // poses of this step (ctlp.py:3166-3178)
                double pm, vv, aa;
                interpolate(q, v, as, ae, c_sc.hu.brake_t[m], pm, vv, aa);
                if (np + m - 1 < SM_HBRAKE_POSES) poses[(np + m - 1) * 8 + j] = (float)pm;
                pend = pm;
            }
            np += C;
            if ((double)k * ts > c_sc.hu.brake_timeout) { timeout = 1; done = true; }   // ctlp.py:3471-3473
            else {
                double qq, aa;
                interpolate(q, v, as, ae, ts, qq, vend, aa);
                small_j = fabs(vend) < 0.01 && fabs(ae) < 0.01;
            }
        }
        // robot_stopped: every joint of the env slow and without acceleration (braking_trajectory_generator.py:45-47)
        const unsigned sm_all = __ballot_sync(FULL, done || small_j);
        const bool stopped = ((sm_all >> gsh) & 0xffu) == 0xffu;
        if (!done) {
            if (stopped) done = true;
            else {
                const double e = human_braking_acceleration(L, j, pend, vend, ae, small_j);
                if (k < SM_HBRAKE_STEPS) bacc[k * 8 + j] = e;
                ++k;
                q = pend; v = vend; as = ae; ae = e;
            }
        }
        if (__all_sync(FULL, done)) break;
    }
    const int npc = valid ? (np < SM_HBRAKE_POSES ? np : SM_HBRAKE_POSES) : 0;   // the same in the eight lanes of the env
    const int nsp = (npc + HBP_SPAN - 1) / HBP_SPAN;
    int base = 0;
    if (valid && j == 0) {
        int* bi = A.binfo + env * 4;
        bi[0] = k; bi[1] = npc; bi[2] = timeout; bi[3] = 0;
        A.res[env * SM_RES_STRIDE + GJK_BRAKE] = SM_RES_NO_CONTACT;
        if (A.counters && npc > 0) {
            atomicAdd(&A.counters[16], (unsigned long long)npc);
            atomicAdd(&A.counters[18], (unsigned long long)nsp);
        }
        if (nsp > 0) base = atomicAdd(A.units, nsp);
    }
    if (t == 0) A.fine[0] = 0;   // the span pass of this step fills the per-pose list afresh
    base = __shfl_sync(FULL, base, lane & 24);
    for (int s = j; s < nsp; s += 8) {   // one unit per span of up to HBP_SPAN consecutive poses for the geometry pass
        const int p0 = s * HBP_SPAN, n = npc - p0 < HBP_SPAN ? npc - p0 : HBP_SPAN;
        A.units[1 + base + s] = hbp_unit((int)env, p0, n);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// geometry of the braking-trajectory check: ONE THREAD PER POSE (the span pass lists them).  Serial forward
// kinematics of the two arms; as soon as a frame is known, the bounding-sphere centres of its shapes and the end points
// of its bounding capsule go to the thread's column of a shared-memory table -- every later test reads points by
// (uniform) index from there, no transform is applied twice.  Then the link-group pairs of get_minimum_distance
// (ctlp.py:3282-3374: table x forearm / hand, forearm / hand x other arm, forearm / hand x body / head): a capsule test
// per group pair, and inside a surviving group pair the sphere bound of every convex pair (the pairs of a group pair
// are the cross product of two shape ranges, smenv_create checks it) and the separating-axis bound of the distance
// planning for what is left.  A pair that may be closer than the safety distance becomes a GJK_BRAKE item carrying
// the pose number.  The trunk does not move: its shapes' world centres are computed once per CTA.
// In front of it runs the same kernel as a span pass (SPAN = true): one thread per run of up to HBP_SPAN consecutive poses
// of an env, the FK of the middle pose, the arm frames' volumes grown by how far their points can move inside the run, the
// same capsule tests and sphere bounds; no axis bound, no items.  The poses of a run with a sphere-bound survivor are
// listed for the per-pose pass.  A cleared run has no survivor at any of its poses, so the two passes emit the items the
// per-pose pass alone would.
// ------------------------------------------------------------------------------------------------------------------
// squared distance between the segments [p1, q1] and [p2, q2] (Ericson, Real-Time Collision Detection, 5.1.9)
__device__ __forceinline__ float segment_dist2(V3 p1, V3 q1, V3 p2, V3 q2) {
    const V3 d1 = q1 - p1, d2 = q2 - p2, r = p1 - p2;
    const float a = dot(d1, d1), e = dot(d2, d2), f = dot(d2, r);
    float s, t;
    if (a <= 1e-12f && e <= 1e-12f) return dot(r, r);
    if (a <= 1e-12f) { s = 0.f; t = fminf(fmaxf(f / e, 0.f), 1.f); }
    else {
        const float c = dot(d1, r);
        if (e <= 1e-12f) { t = 0.f; s = fminf(fmaxf(-c / a, 0.f), 1.f); }
        else {
            const float b = dot(d1, d2), den = a * e - b * b;
            s = den > 1e-12f ? fminf(fmaxf((b * f - c * e) / den, 0.f), 1.f) : 0.f;
            t = (b * s + f) / e;
            if (t < 0.f) { t = 0.f; s = fminf(fmaxf(-c / a, 0.f), 1.f); }
            else if (t > 1.f) { t = 1.f; s = fminf(fmaxf((b - c) / a, 0.f), 1.f); }
        }
    }
    const V3 c1 = p1 + s * d1, c2 = p2 + t * d2, dd = c1 - c2;
    return dot(dd, dd);
}

#define HBP_THREADS 128
#ifndef HBP_INTERLEAVE
#define HBP_INTERLEAVE 0   /* the FK chains of the two arms written side by side (experiment) */
#endif
#ifndef HBP_UNROLL_NEAR
#define HBP_UNROLL_NEAR 0  /* capsule tests of the link-group pairs unrolled (experiment) */
#endif
#define HBP_MAX_TRUNK 32
// dynamic shared memory: point table [n_arm_shapes + 8][3][HBP_THREADS] | trunk spheres [HBP_MAX_TRUNK] float4 |
// world capsules of the trunk sides of the group pairs [8][8] | radius + margin of the arm shapes [32]
static size_t human_plan_smem_bytes(int n_arm_shapes) {
    return (size_t)(n_arm_shapes + 8) * 3 * HBP_THREADS * sizeof(float) + HBP_MAX_TRUNK * sizeof(float4) + (64 + 32) * sizeof(float);
}
// radius of the two spheres at 1/4 and 3/4 of a capsule's segment (length len) that stand in for the capsule (radius ra)
// in the test against the table's box: ra + len / 4, since a point of an end cap lies within ra of the segment's end and
// that end within len / 4 of the nearer centre (sqrt(ra^2 + (len / 4)^2) covers the cylinder only: the capsule's segment
// is pulled in by its radius, so vertices do lie in the caps).  Host and device: smenv_debug_human_bounds exports it.
__host__ __device__ __forceinline__ float table_cover_radius(float ra, float len) { return ra + 0.25f * len; }
__device__ __forceinline__ int hbp_frame_index(int f) { return f == 3 ? 0 : f == 4 ? 1 : f == 7 ? 2 : 3; }
__device__ __forceinline__ void hbp_pick(int f, const Xf& F3, const Xf& F4, const Xf& F7, const Xf& F8, const Xf& B,
                                         const Xf& world, Xf& out) {
    out = f < 0 ? world : f == 0 ? B : f == 3 ? F3 : f == 4 ? F4 : f == 7 ? F7 : F8;
}

template <bool SPAN>
__global__ void __launch_bounds__(HBP_THREADS) human_brake_plan_kernel(HumanArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n_units = A.units[0];
    if (blockIdx.x * HBP_THREADS >= n_units) return;
    const int tid = threadIdx.x, lane = tid & 31;
    const int nas = c_sc.hu.n_arm_shapes, soff = c_sc.hu.shape_off;
    float* P = reinterpret_cast<float*>(smem_raw) + tid;                    // this thread's column: P[(slot * 3 + k) * HBP_THREADS]
    float4* TC = reinterpret_cast<float4*>(smem_raw + (size_t)(nas + 8) * 3 * HBP_THREADS * sizeof(float));
    float* GC = reinterpret_cast<float*>(TC + HBP_MAX_TRUNK);
    float* RM = GC + 64;
    const float safety = (float)c_sc.hu.brake_safety;
    Xf world, B;
    xf_identity(world);
    human_base(B);
    const int n_trunk = c_sc.hu.n_shapes - nas;
    if (tid < n_trunk) {
        const DevShape& sh = c_sc.shapes[soff + nas + tid];
        const V3 c = xf_apply(B, sh.cx, sh.cy, sh.cz);
        TC[tid] = make_float4(c.x, c.y, c.z, sh.radius + sh.margin);
    }
    if (tid < nas && tid < 32) RM[tid] = c_sc.shapes[soff + tid].radius + c_sc.shapes[soff + tid].margin;
    if (tid < c_sc.hu.n_gp && c_sc.hu.gp_fb[tid] == 0) {
        const float* sb = c_sc.hu.gp_sb[tid];
        const V3 b0 = xf_apply(B, sb[0], sb[1], sb[2]), b1 = xf_apply(B, sb[3], sb[4], sb[5]);
        GC[8 * tid] = b0.x; GC[8 * tid + 1] = b0.y; GC[8 * tid + 2] = b0.z;
        GC[8 * tid + 3] = b1.x; GC[8 * tid + 4] = b1.y; GC[8 * tid + 5] = b1.z;
    }
    __syncthreads();
    auto put = [&](int slot, V3 v) {
        P[(slot * 3 + 0) * HBP_THREADS] = v.x; P[(slot * 3 + 1) * HBP_THREADS] = v.y; P[(slot * 3 + 2) * HBP_THREADS] = v.z;
    };
    auto get = [&](int slot) {
        return mk(P[(slot * 3 + 0) * HBP_THREADS], P[(slot * 3 + 1) * HBP_THREADS], P[(slot * 3 + 2) * HBP_THREADS]);
    };
    auto frame_points = [&](const Xf& F, int fi) {   // shapes and capsule of arm frame fi (uniform loop bounds)
        const int s0 = c_sc.hu.hf_s0[fi], s1 = s0 + c_sc.hu.hf_sn[fi];
#pragma unroll 1
        for (int sI = s0; sI < s1; ++sI) put(sI - soff, xf_apply(F, c_sc.shapes[sI].cx, c_sc.shapes[sI].cy, c_sc.shapes[sI].cz));
        const float* sg = c_sc.hu.hf_seg[fi];
        put(nas + 2 * fi, xf_apply(F, sg[0], sg[1], sg[2]));
        put(nas + 2 * fi + 1, xf_apply(F, sg[3], sg[4], sg[5]));
    };
    unsigned n_bounds = 0;   // sphere bounds of convex pairs evaluated by this thread (counted in the measurement mode)
    unsigned n_fine = 0;     // span pass: poses this warp passed on to the per-pose pass (lane 31 counts)
#pragma unroll 1
    for (int u0 = blockIdx.x * HBP_THREADS; u0 < n_units; u0 += gridDim.x * HBP_THREADS) {
        __syncwarp();   // lanes leave the pair loops of the previous pose at different times
        const int u = u0 + tid;
        const bool valid = u < n_units;   // the loops below are uniform over the warp: idle lanes run them on the last pose
        const unsigned unit = (unsigned)A.units[1 + (valid ? u : n_units - 1)];
        const int env = (int)(unit >> 10), p = (int)(unit & 127u);
        const int np = SPAN ? (int)((unit >> 7) & 7u) + 1 : 1;
        const float4* row = reinterpret_cast<const float4*>(A.poses + ((size_t)env * SM_HBRAKE_POSES + p + (np - 1) / 2) * 8);
        const float4 r0 = row[0], r1 = row[1];
        // span pass: the forward kinematics of the middle pose stands for the span; every point of arm frame i lies within
        // e_i of where it is at any pose of the span (sum_j max_p |q_p,j - q_mid,j| hf_rho[i][j]), so every volume of
        // the frame grows by e_i.  A span without a sphere-bound survivor has none at any of its poses.
        float e_f[4] = {0.f, 0.f, 0.f, 0.f};
        if constexpr (SPAN) {
            const float4* row0 = reinterpret_cast<const float4*>(A.poses + ((size_t)env * SM_HBRAKE_POSES + p) * 8);
            float dq[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
            for (int i = 0; i < np; ++i) {
                const float4 a = row0[2 * i], b = row0[2 * i + 1];
                dq[0] = fmaxf(dq[0], fabsf(a.x - r0.x)); dq[1] = fmaxf(dq[1], fabsf(a.y - r0.y));
                dq[2] = fmaxf(dq[2], fabsf(a.z - r0.z)); dq[3] = fmaxf(dq[3], fabsf(a.w - r0.w));
                dq[4] = fmaxf(dq[4], fabsf(b.x - r1.x)); dq[5] = fmaxf(dq[5], fabsf(b.y - r1.y));
                dq[6] = fmaxf(dq[6], fabsf(b.z - r1.z)); dq[7] = fmaxf(dq[7], fabsf(b.w - r1.w));
            }
#pragma unroll
            for (int fi = 0; fi < 4; ++fi) {
                float e = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) e = fmaf(dq[j], c_sc.hu.hf_rho[fi][j], e);
                e_f[fi] = e * (1.0f + 1e-5f) + 1e-5f;
            }
        }
        // inflation of arm frame fi (uniform index: selects, no local memory)
        auto infl = [&](int fi) { return fi == 0 ? e_f[0] : fi == 1 ? e_f[1] : fi == 2 ? e_f[2] : e_f[3]; };
        // frames that carry shapes of the check: upper arm (3 / 7) and forearm + hand (4 / 8) of both arms
        Xf F3, F4, F7, F8;
#if HBP_INTERLEAVE
        {   // the two arms are independent chains: written side by side so that their latencies overlap
            Xf Fa = B, Fb = B;
            human_chain_step(Fa, 0, r0.x); human_chain_step(Fb, 4, r1.x);
            human_chain_step(Fa, 1, r0.y); human_chain_step(Fb, 5, r1.y);
            human_chain_step(Fa, 2, r0.z); human_chain_step(Fb, 6, r1.z);
            F3 = Fa; F7 = Fb;
            human_chain_step(Fa, 3, r0.w); human_chain_step(Fb, 7, r1.w);
            F4 = Fa; F8 = Fb;
            frame_points(F3, 0); frame_points(F7, 2); frame_points(F4, 1); frame_points(F8, 3);
        }
#else
        {
            Xf F = B;
            human_chain_step(F, 0, r0.x); human_chain_step(F, 1, r0.y); human_chain_step(F, 2, r0.z);
            F3 = F;
            frame_points(F3, 0);
            human_chain_step(F, 3, r0.w);
            F4 = F;
            frame_points(F4, 1);
            F = B;
            human_chain_step(F, 4, r1.x); human_chain_step(F, 5, r1.y); human_chain_step(F, 6, r1.z);
            F7 = F;
            frame_points(F7, 2);
            human_chain_step(F, 7, r1.w);
            F8 = F;
            frame_points(F8, 3);
        }
#endif
        // capsule tests of all link-group pairs first (independent of each other: unrolled, no branches between them)
        unsigned near = 0u;
#if HBP_UNROLL_NEAR
#pragma unroll
#else
#pragma unroll 1
#endif
        for (int g = 0; g < 8; ++g) {
            if (g >= c_sc.hu.n_gp) continue;
            const int fa = c_sc.hu.gp_fa[g], fb = c_sc.hu.gp_fb[g];
            const int fia = hbp_frame_index(fa);
            const V3 a0 = get(nas + 2 * fia), a1 = get(nas + 2 * fia + 1);
            const float ra = SPAN ? c_sc.hu.hf_rad[fia] + infl(fia) : c_sc.hu.hf_rad[fia];
            bool near_g;
            if (fb < 0) {    // the table's box against two spheres that cover the capsule of side A
                const V3 dl = a1 - a0;
                const float l = table_cover_radius(ra, sqrtf(dot(dl, dl))) * (1.0f + 1e-5f) + safety + 1e-5f;
                near_g = box_dist2(a0 + 0.25f * dl, c_sc.hu.gp_bmin[g], c_sc.hu.gp_bmax[g]) <= l * l ||
                         box_dist2(a0 + 0.75f * dl, c_sc.hu.gp_bmin[g], c_sc.hu.gp_bmax[g]) <= l * l;
            } else {         // capsules of both sides: the arm groups are long and thin
                V3 b0, b1;
                float rb;
                if (fb == 0) {
                    b0 = mk(GC[8 * g], GC[8 * g + 1], GC[8 * g + 2]); b1 = mk(GC[8 * g + 3], GC[8 * g + 4], GC[8 * g + 5]);
                    rb = c_sc.hu.gp_srb[g];
                } else {
                    const int fib = hbp_frame_index(fb);
                    b0 = get(nas + 2 * fib); b1 = get(nas + 2 * fib + 1);
                    rb = SPAN ? c_sc.hu.hf_rad[fib] + infl(fib) : c_sc.hu.hf_rad[fib];
                }
                const float l = ra + rb + safety * (1.0f + 1e-5f) + 1e-5f;
                near_g = segment_dist2(a0, a1, b0, b1) <= l * l;
            }
            near |= (near_g ? 1u : 0u) << g;
        }
        if (!valid) near = 0u;
        bool flag = false;   // span pass: some pair of the span survives its sphere bound
#pragma unroll 1
        for (int g = 0; g < c_sc.hu.n_gp; ++g) {
            __syncwarp();
            if (!((near >> g) & 1u) || flag) continue;
            const int fa = c_sc.hu.gp_fa[g], fb = c_sc.hu.gp_fb[g];
            const int sa0 = c_sc.hu.gp_a0[g], sa1 = sa0 + c_sc.hu.gp_na[g];
            const int sb0 = c_sc.hu.gp_b0[g], nb = c_sc.hu.gp_nb[g];
            const float eb = SPAN && fb > 0 ? infl(hbp_frame_index(fb)) : 0.f;   // trunk and table do not move
            if (!SPAN) n_bounds += (unsigned)((sa1 - sa0) * nb);
#pragma unroll 1
            for (int ia = sa0; ia < sa1; ++ia) {
                const V3 ca = get(ia - soff);
                const float la = SPAN ? RM[ia - soff] + safety + infl(hbp_frame_index(fa)) : RM[ia - soff] + safety;
                // sphere bound of the nb pairs (ia, sb0 + k): bit k of `hits` = the pair goes on to the axis bound
                unsigned hits = 0u;
                if (fb < 0) {              // the table: sphere against its axis-aligned box
#pragma unroll 1
                    for (int k = 0; k < nb; ++k) {
                        const DevShape& SB = c_sc.shapes[sb0 + k];
                        const float l = la + SB.margin;
                        hits |= (box_dist2(ca, SB.bmin, SB.bmax) <= l * l * (1.0f + 1e-5f) ? 1u : 0u) << k;
                    }
                } else if (fb == 0) {      // the trunk: constant spheres
                    const float4* tc = TC + (sb0 - soff - nas);
#pragma unroll 4
                    for (int k = 0; k < nb; ++k) {
                        const float4 t = tc[k];
                        const float dx = t.x - ca.x, dy = t.y - ca.y, dz = t.z - ca.z, l = la + t.w;
                        hits |= (fmaf(dx, dx, fmaf(dy, dy, dz * dz)) <= l * l * (1.0f + 1e-5f) ? 1u : 0u) << k;
                    }
                } else {                   // the other arm
                    const int slot0 = sb0 - soff;
#pragma unroll 4
                    for (int k = 0; k < nb; ++k) {
                        const V3 d = get(slot0 + k) - ca;
                        const float l = SPAN ? la + RM[slot0 + k] + eb : la + RM[slot0 + k];
                        hits |= (dot(d, d) <= l * l * (1.0f + 1e-5f) ? 1u : 0u) << k;
                    }
                }
                if constexpr (SPAN) {
                    if (hits) { flag = true; break; }
                } else {
                    while (hits) {             // rare: the frames are picked out of the registers only here
                        const int ib = sb0 + __ffs(hits) - 1;
                        hits &= hits - 1u;
                        Xf TA, TB;
                        hbp_pick(fa, F3, F4, F7, F8, B, world, TA);
                        hbp_pick(fb, F3, F4, F7, F8, B, world, TB);
                        const DevShape& SA = c_sc.shapes[ia];
                        const DevShape& SB = c_sc.shapes[ib];
                        const V3 d = xf_apply(TB, SB.cx, SB.cy, SB.cz) - ca;
                        if (axis_lower_bound_d(SA, SB, TA, TB, d) <= safety) {
                            const int idx = atomicAdd(A.item_count, 1);
                            if (idx < A.capacity) write_item(A.items + idx, env, ia, ib, GJK_BRAKE, p + 1, safety, TA, TB);
                            else atomicAdd(A.overflow, 1);
                        }
                    }
                }
            }
        }
        if constexpr (SPAN) {   // every pose of an uncleared span goes to the per-pose pass, warp-aggregated
            const int cnt = valid && flag ? np : 0;
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int x = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += x;
            }
            const int total = __shfl_sync(FULL, incl, 31);
            if (total) {
                int base = 0;
                if (lane == 31) { base = atomicAdd(A.fine, total); n_fine += (unsigned)total; }
                base = __shfl_sync(FULL, base, 31) + incl - cnt;
                for (int i = 0; i < cnt; ++i) A.fine[1 + base + i] = hbp_unit(env, p + i, 1);
            }
        }
    }
    if (A.counters && n_bounds) atomicAdd(&A.counters[17], (unsigned long long)n_bounds);
    if (A.counters && n_fine) atomicAdd(&A.counters[19], (unsigned long long)n_fine);
}

// observation of the nested env (observations.py:313-351 with two arms and alternating target points): entries spread over
// `stride` lanes
__device__ __forceinline__ void write_human_observation(float* hobs, const double* hk, const double* hs, int lane, int stride) {
    const JointLim& L = c_sc.hu.lim;
#pragma unroll 1
    for (int i = lane; i < SM_HOBS_STRIDE; i += stride) {
        double val = 0.0;
        if (i < 24) {
            const int grp = i >> 3, j = i & 7;
            const double x = hk[grp * 8 + j];
            val = grp == 0 ? normalize_mm(x, L.pos_lo[j], L.pos_hi[j]) : xdiv(x, grp == 1 ? L.vel_max[j] : L.acc_max[j]);
        } else if (i < 30) {
            const int r = (i - 24) / 3, c = (i - 24) % 3;
            const double* tp = hs + 12 * r;
            if (tp[SM_TP_ACTIVE] != 0.0) val = normalize_mm(tp[SM_TP_POS + c], c_sc.hu.tp_box_min[c], c_sc.hu.tp_box_max[c]);
        } else if (i < 36) {
            const int r = (i - 30) / 3, c = (i - 30) % 3;
            const double* tp = hs + 12 * r;
            if (tp[SM_TP_ACTIVE] != 0.0)
                val = normalize_mm(xsub(tp[SM_TP_POS + c], tp[SM_TP_LINK_POS + c]), c_sc.hu.tp_rel_min[c], c_sc.hu.tp_rel_max[c]);
        } else if (i < 38) {
            val = hs[12 * (i - 36) + SM_TP_ACTIVE] != 0.0 ? 1.0 : 0.0;
        }
        hobs[i] = clip1(val);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// outcome of the nested env's step: 8 lanes per env (the second half of human_advance_kernel).  Lanes 0 / 1 take the link
// points of the two arms at the new knot; if the active arm's point is close enough to its target for a sub-step to have
// reached it (how far every joint strays from the knot inside the step comes from the lanes that just integrated it), lane
// i checks sub-steps i, i + 8, i + 16 (ctlp.py:2787-2821; target link point of the sub-step's setpoint pose); then
// get_target_point_observation (ctlp.py:2210-2271) and the observation.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void human_outcome(const HumanArgs& A, size_t env, bool valid, int lane,
                                              float dq_lane /* how far joint (lane & 7) strays from the new knot in the step */,
                                              double q0, double v0, double a0, double a1 /* the step of joint (lane & 7) */) {
    const int sl = lane & 7;
    const unsigned gmask = 0xffu << (lane & 24);
    const int S = c_sc.substeps;
    double* hs = A.buf.hstate + env * SM_HSTATE_STRIDE;
    const double* hk = A.buf.hkin + env * SM_KIN_STRIDE;
    int active = -1;
    if (hs[SM_TP_ACTIVE] != 0.0) active = 0;
    else if (hs[12 + SM_TP_ACTIVE] != 0.0) active = 1;
    // link points of both arms at the new knot (the setpoint pose of the last sub-step)
    V3 lp = mk(0.f, 0.f, 0.f);
    if (sl < 2) {
        Xf F;
        human_base(F);
#pragma unroll 1
        for (int i = 0; i < 4; ++i) human_chain_step(F, 4 * sl + i, (float)hk[4 * sl + i]);
        lp = xf_apply(F, c_sc.hu.tp_local[sl][0], c_sc.hu.tp_local[sl][1], c_sc.hu.tp_local[sl][2]);
    }
    bool hit = false;
    {
        // every sub-step's link point lies within infl of the new knot's: sum_i max_k |q_i(k) - q_i(S)| rho_i; only an
        // env whose knot point is that close to the target runs the forward kinematics of the sub-steps
        const int arm = active >= 0 ? active : 0, src = (lane & 24) | arm;
        const V3 lpa = mk(__shfl_sync(FULL, lp.x, src), __shfl_sync(FULL, lp.y, src), __shfl_sync(FULL, lp.z, src));
        float infl = 1e-5f;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            infl = fmaf(__shfl_sync(FULL, dq_lane, (lane & 24) | (4 * arm + i)), c_sc.hu.tp_rho[arm][i], infl);
        if (active >= 0) {
            const double* tp = hs + 12 * active;
            const V3 T = mk((float)tp[SM_TP_POS], (float)tp[SM_TP_POS + 1], (float)tp[SM_TP_POS + 2]);
            const V3 e1 = lpa - T;
            if (sqrtf(dot(e1, e1)) - infl < (float)c_sc.hu.tp_radius) {   // uniform over the eight lanes of the env
                // the step of the four joints of the active arm, from the lanes that own them (the setpoints are not stored)
                double jq[4], jv[4], ja[4], ja1[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int from = (lane & 24) | (4 * arm + i);
                    jq[i] = __shfl_sync(gmask, q0, from); jv[i] = __shfl_sync(gmask, v0, from);
                    ja[i] = __shfl_sync(gmask, a0, from); ja1[i] = __shfl_sync(gmask, a1, from);
                }
                Xf B;
                human_base(B);
#pragma unroll 1
                for (int k = sl; k < S; k += 8) {
                    Xf F = B;
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        human_chain_step(F, 4 * active + i, (float)joint_setpoint_at(jq[i], jv[i], ja[i], ja1[i], k + 1));
                    const V3 e = xf_apply(F, c_sc.hu.tp_local[active][0], c_sc.hu.tp_local[active][1], c_sc.hu.tp_local[active][2]) - T;
                    if (sqrtf(dot(e, e)) < (float)c_sc.hu.tp_radius) hit = true;
                }
            }
        }
    }
    const bool reached = (__ballot_sync(FULL, hit) & gmask) != 0u;
    const double draws = hs[SM_HS_DRAWS];
    __syncwarp();
    if (valid && sl < 2) {   // lane r owns the record of arm r
        double* tp = hs + 12 * sl;
        tp[SM_TP_LINK_POS] = (double)lp.x; tp[SM_TP_LINK_POS + 1] = (double)lp.y; tp[SM_TP_LINK_POS + 2] = (double)lp.z;
        bool act = tp[SM_TP_ACTIVE] != 0.0;
        tp[SM_HTP_REACHED] = 0.0;
        if (reached && sl == active) {         // ctlp.py:2806-2811
            act = false;
            tp[SM_TP_REACHED_N] += 1.0;
        }
        const bool sample_new = reached && sl == (active + 1) % 2;   // alternating target points (ctlp.py:2815-2817)
        if (sample_new && A.target_pool_n > 0) {                      // _add_target_point from the device pool
            const uint4 r = philox((uint32_t)(env + A.env_base), (uint32_t)draws, 0x7A28u, 3u, A.k0, A.k1);
            const double* e = A.target_pool + ((size_t)sl * A.target_pool_n + (r.x % (uint32_t)A.target_pool_n)) * 4;
            tp[SM_TP_POS] = e[0]; tp[SM_TP_POS + 1] = e[1]; tp[SM_TP_POS + 2] = e[2];
            act = true;
            tp[SM_TP_INIT_DIST] = nan("");
        } else if (sample_new) {
            tp[SM_HTP_SAMPLE_NEW] = 1.0;   // no pool: the caller injects the next target point (parity protocol)
        }
        tp[SM_TP_ACTIVE] = act ? 1.0 : 0.0;
        if (act) {
            const double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
                         dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
            tp[SM_TP_LAST_DIST] = sqrt(dx * dx + dy * dy + dz * dz);
            if (isnan(tp[SM_TP_INIT_DIST])) tp[SM_TP_INIT_DIST] = tp[SM_TP_LAST_DIST];
        }
        if (sample_new && A.target_pool_n > 0) hs[SM_HS_DRAWS] = draws + 1.0;
        __threadfence_block();
    }
    __syncwarp();
    if (valid) write_human_observation(A.buf.hobs + env * SM_HOBS_STRIDE, hk, hs, sl, 8);
}

// ------------------------------------------------------------------------------------------------------------------
// adapt_action (ctlp.py:3055-3153) + get_braking_acceleration (:3000-3024), then the 24 setpoints and the tracked pose of
// the human (Human.prepare_sim_step ctlp.py:4850-4860; robot_scene_base.py:789-837): thread = (env, joint); then the outcome
// ------------------------------------------------------------------------------------------------------------------
#ifndef HADV_MIN_BLOCKS
#define HADV_MIN_BLOCKS 4   /* resident CTAs per SM the register allocation aims for (3, 5, 6: 1491 / 1482 / 1485 us against 1480) */
#endif
__global__ void __launch_bounds__(256, HADV_MIN_BLOCKS) human_advance_kernel(HumanArgs A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int env_raw = t >> 3, j = t & 7;
    const bool valid = env_raw < A.n;
    const size_t env = valid ? (size_t)env_raw : (size_t)(A.n - 1);
    double* kin = A.buf.hkin + env * SM_KIN_STRIDE;
    double* hs = A.buf.hstate + env * SM_HSTATE_STRIDE;
    double* hb = A.buf.hbrake + env * SM_HBRAKE_STEPS * 8;
    const int* bi = A.binfo + env * 4;
    double a1 = A.range[(env * 8 + j) * 4 + 2];
    const int count = (int)hs[SM_HS_BRAKE_COUNT];
    int braked = 0, new_count = count;
    // `valid`: the lanes past the last env alias its record and must not shift its stored trajectory a second time
    if (valid && c_sc.hu.check_braking) {
        const bool execute = A.res[env * SM_RES_STRIDE + GJK_BRAKE] != SM_RES_NO_CONTACT || bi[2] != 0;
        if (execute) {   // the stored braking trajectory is executed instead of the action
            braked = 1;
            if (count > 0) {
                a1 = hb[j];
#pragma unroll 1
                for (int i = 0; i + 1 < count; ++i) hb[i * 8 + j] = hb[(i + 1) * 8 + j];
                new_count = count - 1;
            } else {
                a1 = 0.0;
            }
        } else {         // the checked trajectory becomes the valid one (ctlp.py:3096-3119)
            int k = bi[0];
            if (k > SM_HBRAKE_STEPS) k = SM_HBRAKE_STEPS;
            const double* src = A.bacc + env * SM_HBRAKE_STEPS * 8;
#pragma unroll 1
            for (int i = 0; i < k; ++i) hb[i * 8 + j] = src[i * 8 + j];
            new_count = k;
        }
    }
    const double q = kin[j], v = kin[8 + j], a = kin[16 + j], qa = kin[24 + j];
    const double steps = hs[SM_HS_STEPS];
    __syncwarp();   // every lane of the env has read the record before lane 0 rewrites it
    float dq = 0.f;
    if (valid) {
        joint_advance_a1(kin, A.hscratch + env * SM_SCRATCH_FLOATS, j, q, v, a, qa, a1, 0.87, false, c_sc.hu.lim.jerk_max[j], &dq);
        if (j == 0) {
            hs[SM_HS_BRAKE_COUNT] = (double)new_count;
            hs[SM_HS_BRAKED] = (double)braked;
            hs[SM_HS_STEPS] = steps + 1.0;
        }
    }
    __syncwarp();   // the new knot and the sub-step setpoints of the env are visible to its eight lanes
    human_outcome(A, env, valid, threadIdx.x & 31, dq, q, v, a, a1);
}

// ------------------------------------------------------------------------------------------------------------------
// contacts robot <-> human in the simulation client (Human.check_if_object_is_colliding, ctlp.py:4888-4898): both bodies
// at their motor-tracked poses of the 24 sub-steps.  Coarse phase as for planets / balls (smenv_plan.cuh): 8 threads per
// env, each clears a span of 3 sub-steps with one forward kinematics of both bodies; link spheres are inflated by what
// the joints move inside the span.  Spans that cannot be cleared go to the fine planning (one lane per sub-step).
// ------------------------------------------------------------------------------------------------------------------
#ifndef HCC_MIN_BLOCKS
#define HCC_MIN_BLOCKS 4   /* resident CTAs per SM the register allocation aims for: 64 registers instead of 75 (Human step
                              1485 -> 1469 us) */
#endif
__global__ void __launch_bounds__(256, HCC_MIN_BLOCKS) hcontact_coarse_kernel(HumanArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SceneSmem* smp = reinterpret_cast<SceneSmem*>(smem_raw);
    for (int i = threadIdx.x; i < (int)(sizeof(SceneSmem) / 16); i += blockDim.x)
        reinterpret_cast<uint4*>(smp)[i] = __ldg(c_sc.scene_img + i);
    __syncthreads();
    const SceneSmem& sm = *smp;
    const int tid = threadIdx.x, lane = tid & 31;
    const int t = blockIdx.x * blockDim.x + tid;
    const int env = t / SM_COARSE_LANES, c = t % SM_COARSE_LANES;
    const int S = c_sc.substeps;
    const int span = (S + SM_COARSE_LANES - 1) / SM_COARSE_LANES;
    bool flag = false;
    if (env < A.n && c_sc.contact_stride > 0 && c * span < S &&
        A.buf.obst[(size_t)env * SM_OBST_STRIDE + SM_OB_LATCH] == 0.0) {
        const int k0 = c * span, k1 = k0 + span < S ? k0 + span : S;
        const int kc = (k0 + k1 - 1) >> 1;
        const float* scr = A.scratch + (size_t)env * SM_SCRATCH_FLOATS;
        const float* hscr = A.hscratch + (size_t)env * SM_SCRATCH_FLOATS;
        float dq[SM_MAX_JOINTS], dh[SM_HUMAN_JOINTS], hq[SM_HUMAN_JOINTS];
#pragma unroll
        for (int j = 0; j < 8; ++j) { dq[j] = 0.f; dh[j] = 0.f; hq[j] = hscr[kc * SM_MAX_JOINTS + j]; }
#pragma unroll 1
        for (int k = k0; k < k1; ++k)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                dq[j] = fmaxf(dq[j], fabsf(scr[k * SM_MAX_JOINTS + j] - scr[kc * SM_MAX_JOINTS + j]));
                dh[j] = fmaxf(dh[j], fabsf(hscr[k * SM_MAX_JOINTS + j] - hq[j]));
            }
        // human group spheres at the middle pose, inflated by the motion of the human inside the span
        V3 gc[SM_HGROUPS];
        float gr[SM_HGROUPS];
        {
            Xf hfr[SM_MAX_OBST_FRAMES];
            human_fk_serial(hq, hfr);
#pragma unroll
            for (int g = 0; g < SM_HGROUPS; ++g) {
                gc[g] = xf_apply(hfr[c_sc.hu.grp_frame[g]], c_sc.hu.grp_c[g][0], c_sc.hu.grp_c[g][1], c_sc.hu.grp_c[g][2]);
                float infl = 1e-5f;
#pragma unroll
                for (int j = 0; j < 8; ++j) infl = fmaf(dh[j], c_sc.hu.grp_rho[g][j], infl);
                gr[g] = c_sc.hu.grp_r[g] + infl + c_sc.hu.contact_thresh_max;
            }
        }
        Xf F;
        xf_identity(F);
#pragma unroll 1
        for (int f = 0; f <= c_sc.n_joints && !flag; ++f) {
            if (f > 0) fk_chain_step(sm, F, f - 1, scr[kc * SM_MAX_JOINTS + f - 1]);
#pragma unroll 1
            for (int slot = c_sc.contact_frame_start[f]; slot < c_sc.contact_frame_start[f + 1]; ++slot) {
                const DevShape& sh = sm.shapes[sm.mov_contact[slot]];
                const V3 ctr = xf_apply(F, sh.cx, sh.cy, sh.cz);
                float infl = 1e-5f;
#pragma unroll
                for (int j = 0; j < SM_MAX_JOINTS; ++j) infl = fmaf(dq[j], c_sc.contact_rho[slot][j], infl);
                const float rr = sh.radius + sh.margin + infl;
#pragma unroll
                for (int g = 0; g < SM_HGROUPS; ++g) {
                    if (c_sc.hu.grp_cnt[g] == 0) continue;
                    if (c_sc.hu.grp_frame[g] == 0) {   // the trunk stands still: its world box instead of a sphere
                        const float lim = rr + c_sc.hu.contact_thresh_max;
                        if (box_dist2(ctr, c_sc.hu.trunk_wmin, c_sc.hu.trunk_wmax) <= lim * lim) flag = true;
                        continue;
                    }
                    const V3 e = ctr - gc[g];
                    const float lim = rr + gr[g];
                    if (dot(e, e) <= lim * lim) flag = true;
                }
            }
        }
    }
    const unsigned fm = __ballot_sync(FULL, flag);
    if (fm) {
        int base = 0;
        if (lane == __ffs(fm) - 1) base = atomicAdd(A.cwork, __popc(fm));
        base = __shfl_sync(FULL, base, __ffs(fm) - 1);
        if (flag) A.cwork[1 + base + __popc(fm & ((1u << lane) - 1u))] = t;
        if (A.counters && lane == __ffs(fm) - 1) atomicAdd(&A.counters[5], (unsigned long long)__popc(fm));
    }
}

// fine contact planning over the listed spans: one lane per sub-step; robot link spheres against the human's link groups,
// then against every part's sphere and box, then the separating-axis bound; survivors become contact items
#ifndef HCP_MIN_BLOCKS
#define HCP_MIN_BLOCKS 1   /* resident CTAs per SM the register allocation aims for (4: 64 registers, 1486 -> 1498 us: worse) */
#endif
__global__ void __launch_bounds__(SM_WARPS_PER_BLOCK * 32, HCP_MIN_BLOCKS) hcontact_plan_kernel(HumanArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n_units = A.cwork[0];
    const int span = (c_sc.substeps + SM_COARSE_LANES - 1) / SM_COARSE_LANES;
    const int upw = 32 / span;
    if (blockIdx.x * SM_WARPS_PER_BLOCK * upw >= n_units) return;
    SceneSmem* smp = reinterpret_cast<SceneSmem*>(smem_raw);
    for (int i = threadIdx.x; i < (int)(sizeof(SceneSmem) / 16); i += blockDim.x)
        reinterpret_cast<uint4*>(smp)[i] = __ldg(c_sc.scene_img + i);
    __syncthreads();
    const SceneSmem& sm = *smp;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = c_sc.substeps, stride = c_sc.contact_stride;
    const int lu = lane / span, i = lane - lu * span;
    unsigned n_flag = 0;
#pragma unroll 1
    for (int ub = (blockIdx.x * SM_WARPS_PER_BLOCK + warp) * upw; ub < n_units; ub += gridDim.x * SM_WARPS_PER_BLOCK * upw) {
        const int u = ub + lu;
        if (u >= n_units || lu >= upw) continue;
        const int unit = A.cwork[1 + u];
        const int env = unit / SM_COARSE_LANES, k = (unit % SM_COARSE_LANES) * span + i;   // 0-based sub-step
        if (k >= S || ((k + 1) % stride) != 0) continue;
        const float* qrow = A.scratch + (size_t)env * SM_SCRATCH_FLOATS + k * SM_MAX_JOINTS;
        const float* hrow = A.hscratch + (size_t)env * SM_SCRATCH_FLOATS + k * SM_MAX_JOINTS;
        Xf hfr[SM_MAX_OBST_FRAMES];
        {
            float hq[SM_HUMAN_JOINTS];
#pragma unroll
            for (int j = 0; j < 8; ++j) hq[j] = hrow[j];
            human_fk_serial(hq, hfr);
        }
        Xf F;
        xf_identity(F);
#pragma unroll 1
        for (int f = 0; f <= c_sc.n_joints; ++f) {
            if (f > 0) fk_chain_step(sm, F, f - 1, qrow[f - 1]);
#pragma unroll 1
            for (int slot = c_sc.contact_frame_start[f]; slot < c_sc.contact_frame_start[f + 1]; ++slot) {
                const int ia = sm.mov_contact[slot];
                const DevShape& sh = sm.shapes[ia];
                const V3 cw = xf_apply(F, sh.cx, sh.cy, sh.cz);
                const float rr = sh.radius + sh.margin;
#pragma unroll 1
                for (int g = 0; g < SM_HGROUPS; ++g) {
                    const Xf& TB = hfr[c_sc.hu.grp_frame[g]];
                    const V3 gcw = xf_apply(TB, c_sc.hu.grp_c[g][0], c_sc.hu.grp_c[g][1], c_sc.hu.grp_c[g][2]);
                    const V3 dd = cw - gcw;
                    const float lim = rr + c_sc.hu.grp_r[g] + c_sc.hu.contact_thresh_max;
                    if (c_sc.hu.grp_cnt[g] == 0) continue;
                    if (c_sc.hu.grp_frame[g] == 0) {
                        const float lb = rr + c_sc.hu.contact_thresh_max;
                        if (box_dist2(cw, c_sc.hu.trunk_wmin, c_sc.hu.trunk_wmax) > lb * lb) continue;
                    } else if (dot(dd, dd) > lim * lim) continue;
                    const V3 cl = xf_rot_t(TB, mk(cw.x - TB.t[0], cw.y - TB.t[1], cw.z - TB.t[2]));   // in the group's frame
#pragma unroll 1
                    for (int s = c_sc.hu.grp_off[g]; s < c_sc.hu.grp_off[g] + c_sc.hu.grp_cnt[g]; ++s) {
                        const DevShape& ps = sm.shapes[c_sc.hu.shape_off + s];
                        const float th = __ldg(c_sc.hu.contact_thresh + c_sc.hu.shape_link[s] * SM_MAX_MOV_ROBOT + slot);
                        const V3 e = mk(cl.x - ps.cx, cl.y - ps.cy, cl.z - ps.cz);
                        const float l2 = rr + ps.radius + ps.margin + th;
                        const float l3 = (rr + ps.margin + th) * (1.0f + 1e-6f) + 1e-6f;
                        if (dot(e, e) <= l2 * l2 && box_dist2(cl, ps.bmin, ps.bmax) <= l3 * l3 &&
                            axis_lower_bound(sh, ps, F, TB) <= th) {
                            const int idx = atomicAdd(A.item_count, 1);
                            if (idx < A.capacity) write_item(A.items + idx, env, ia, c_sc.hu.shape_off + s, GJK_CONTACT, k + 1, th, F, TB);
                            else atomicAdd(A.overflow, 1);
                            ++n_flag;
                        }
                    }
                }
            }
        }
    }
    if (A.counters && n_flag) atomicAdd(&A.counters[6], (unsigned long long)n_flag);
}

// ------------------------------------------------------------------------------------------------------------------
// start of an episode of the nested env: from the pool (reset / auto reset: envs with `done` set, or masked) or injected
// (parity protocol).  One thread per env.
// ------------------------------------------------------------------------------------------------------------------
// The eight lanes of an env (sl = lane & 7) start its nested episode together: lane j copies joint j, lanes 0 / 1 take the
// link point of arm 0 / 1, lane `active_arm` sets up the first target point, then every lane writes its share of the
// observation.  All eight lanes call (inactive groups skip the stores).
__device__ __forceinline__ void human_episode_start(bool active, int sl, unsigned gmask, double* hk, double* hs, double* hb,
                                                    float* hobs, const double* q, const double* v, const double* a,
                                                    const double* first_target, int active_arm, double draws) {
    (void)hb;   // the stored braking trajectory is empty (count 0) or set by the caller: nothing to clear
    if (active) {
        const double dt = xdiv(c_sc.ts, (double)c_sc.substeps), tvdt = xmul(0.87, dt);
        hk[sl] = q[sl]; hk[8 + sl] = v[sl]; hk[16 + sl] = a[sl];
        hk[24 + sl] = xadd(q[sl], xmul(tvdt, v[sl]));   // as the robot: one stepSimulation with the start state as target
#pragma unroll
        for (int i = sl; i < SM_HSTATE_STRIDE; i += 8) hs[i] = 0.0;
    }
    __syncwarp(gmask);
    if (active && sl < 2) {   // link point of arm sl
        Xf F;
        human_base(F);
#pragma unroll 1
        for (int i = 0; i < 4; ++i) human_chain_step(F, 4 * sl + i, (float)q[4 * sl + i]);
        const V3 p = xf_apply(F, c_sc.hu.tp_local[sl][0], c_sc.hu.tp_local[sl][1], c_sc.hu.tp_local[sl][2]);
        double* tp = hs + 12 * sl;
        tp[SM_TP_LINK_POS] = (double)p.x; tp[SM_TP_LINK_POS + 1] = (double)p.y; tp[SM_TP_LINK_POS + 2] = (double)p.z;
        if (sl == active_arm) {
            tp[SM_TP_POS] = first_target[0]; tp[SM_TP_POS + 1] = first_target[1]; tp[SM_TP_POS + 2] = first_target[2];
            tp[SM_TP_ACTIVE] = 1.0;
            const double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
                         dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
            tp[SM_TP_LAST_DIST] = tp[SM_TP_INIT_DIST] = sqrt(dx * dx + dy * dy + dz * dz);
        }
    }
    if (active && sl == 2) hs[SM_HS_DRAWS] = draws;
    __syncwarp(gmask);
    if (active) write_human_observation(hobs, hk, hs, sl, 8);
}

// the human part of the main env's observation: Human.kinematic_observation (observations.py:100-110, :294-307)
__device__ __forceinline__ void copy_human_kinematic_obs(float* obs, const float* hobs, int sl = 0, int stride = 1) {
    const int off = c_sc.obs_size - 3 * SM_HUMAN_JOINTS;
    for (int i = sl; i < 3 * SM_HUMAN_JOINTS; i += stride) obs[off + i] = hobs[i];
}

// ObstacleWrapperBase.reset with compute_initial_braking_trajectory (ctlp.py:1120-1139): the stored braking trajectory
// starts as the accelerations that brake from the start state; the position handed to the range computation is not
// advanced along it (as in the reference).  The eight lanes of an env, lane j = joint j, all lanes of the warp call.
__device__ __forceinline__ int human_initial_braking_steps(double* hb, double q, double v, double a, bool active, int lane) {
    const JointLim& L = c_sc.hu.lim;
    const int j = lane & 7, gsh = lane & 24;
    const double ts = c_sc.ts;
    int k = 0;
    bool done = !active || !c_sc.hu.check_braking || !c_sc.hu.initial_braking_trajectory;
#pragma unroll 1
    while (true) {
        if (!done && ((double)(k - 1) * ts > c_sc.hu.brake_timeout || k >= SM_HBRAKE_STEPS)) done = true;
        const bool small_j = fabs(v) < 0.01 && fabs(a) < 0.01;
        const unsigned sm_all = __ballot_sync(FULL, done || small_j);
        if (!done && ((sm_all >> gsh) & 0xffu) == 0xffu) done = true;
        if (!done) {
            const double e = human_braking_acceleration(L, j, q, v, a, small_j);
            hb[k * 8 + j] = e;
            ++k;
            double qq, vv, aa;
            interpolate(q, v, a, e, ts, qq, vv, aa);
            v = vv; a = e;
        }
        if (__all_sync(FULL, done)) break;
    }
    return k;
}
__device__ __forceinline__ void human_initial_braking(double* hs, double* hb, double q, double v, double a, bool active,
                                                      int lane) {
    const int k = human_initial_braking_steps(hb, q, v, a, active, lane);
    if (active && (lane & 7) == 0) hs[SM_HS_BRAKE_COUNT] = (double)k;
}
// the same for every entry of the start pool, once per pool fill: a reset then copies the stored trajectory
__global__ void __launch_bounds__(256) human_pool_braking_kernel(const double* pool, int n, double* pool_brake, int* pool_bcount) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, j = t & 7;
    const int e_raw = t >> 3;
    const bool active = e_raw < n;
    const size_t e = active ? (size_t)e_raw : (size_t)(n - 1);
    const double* st = pool + e * SM_HPOOL_STRIDE;
    const int k = human_initial_braking_steps(pool_brake + e * SM_HBRAKE_STEPS * 8, st[j], st[8 + j], st[16 + j], active, lane);
    if (active && j == 0) pool_bcount[e] = k;
}

__global__ void __launch_bounds__(256) human_set_state_kernel(HumanArgs A, const double* hq, const double* hv,
                                                              const double* ha, const double* first_target,
                                                              const int32_t* active_arm) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, j = t & 7;
    const int env_raw = t >> 3;
    const bool active = env_raw < A.n && !(A.mask && !A.mask[env_raw]);
    const size_t env = env_raw < A.n ? (size_t)env_raw : (size_t)(A.n - 1);
    const unsigned gmask = 0xffu << (lane & 24);
    human_episode_start(active, j, gmask, A.buf.hkin + env * SM_KIN_STRIDE, A.buf.hstate + env * SM_HSTATE_STRIDE,
                        A.buf.hbrake + env * SM_HBRAKE_STEPS * 8, A.buf.hobs + env * SM_HOBS_STRIDE, hq + env * 8,
                        hv + env * 8, ha + env * 8, first_target + env * 3, active_arm ? active_arm[env] : 0, 1.0);
    __syncwarp(gmask);
    if (active && A.buf.obs) copy_human_kinematic_obs(A.buf.obs + env * c_sc.obs_size, A.buf.hobs + env * SM_HOBS_STRIDE, j, 8);
    __syncwarp();
    human_initial_braking(A.buf.hstate + env * SM_HSTATE_STRIDE, A.buf.hbrake + env * SM_HBRAKE_STEPS * 8, hq[env * 8 + j],
                          hv[env * 8 + j], ha[env * 8 + j], active, lane);
}

// reset of the nested env from the pools.  by_done != 0: the envs whose `done` flag the finish kernel just set (auto
// reset; the robot's record was re-initialised there with pool entry `reset_count - 1`, the human takes the same entry:
// the robot's start pose was sampled clear of that human pose); else the masked envs (smenv_reset, after reset_kernel).
// Eight lanes per env.
__global__ void __launch_bounds__(256) human_reset_kernel(HumanArgs A, int by_done) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, j = t & 7;
    const int env_raw = t >> 3;
    bool active = env_raw < A.n && A.start_pool_n > 0;
    const size_t env = env_raw < A.n ? (size_t)env_raw : (size_t)(A.n - 1);
    if (active) active = by_done ? A.buf.done[env] != 0 : !(A.mask && !A.mask[env]);
    const int4 ep = *reinterpret_cast<const int4*>(A.buf.episode + 4 * env);
    const uint4 r = philox((uint32_t)(env + A.env_base), (uint32_t)(ep.y - 1), 0x5E7u, 1u, A.k0, A.k1);   // the robot's draw
    const uint32_t pick = A.entry ? (uint32_t)A.entry[env] : r.x % (uint32_t)(A.start_pool_n > 0 ? A.start_pool_n : 1);
    const double* e = A.start_pool + (size_t)pick * SM_HPOOL_STRIDE;
    {
        const unsigned gmask = 0xffu << (lane & 24);
        const uint4 r2 = philox((uint32_t)(env + A.env_base), (uint32_t)(ep.y - 1), 0x5E8u, 4u, A.k0, A.k1);
        const int arm = (int)(r2.x & 1u);                          // np.random.randint(0, num_robots) (ctlp.py:1037-1038)
        double ft[3] = {0.3, 0.0, 0.4};
        if (active && A.target_pool_n > 0) {
            const double* tp = A.target_pool + ((size_t)arm * A.target_pool_n + (r2.y % (uint32_t)A.target_pool_n)) * 4;
            ft[0] = tp[0]; ft[1] = tp[1]; ft[2] = tp[2];
        }
        human_episode_start(active, j, gmask, A.buf.hkin + env * SM_KIN_STRIDE, A.buf.hstate + env * SM_HSTATE_STRIDE,
                            A.buf.hbrake + env * SM_HBRAKE_STEPS * 8, A.buf.hobs + env * SM_HOBS_STRIDE, e, e + 8, e + 16, ft,
                            arm, 1.0);
        __syncwarp(gmask);
        if (active && A.buf.obs)
            copy_human_kinematic_obs(A.buf.obs + env * c_sc.obs_size, A.buf.hobs + env * SM_HOBS_STRIDE, j, 8);
    }
    __syncwarp();
    if (A.pool_brake) {   // the braking trajectory of a pool entry does not depend on the env: stored with the pool
        if (active) {
            const size_t entry = pick;
            const int k = c_sc.hu.check_braking && c_sc.hu.initial_braking_trajectory ? A.pool_bcount[entry] : 0;
            const double* src = A.pool_brake + entry * SM_HBRAKE_STEPS * 8;
            double* hb = A.buf.hbrake + env * SM_HBRAKE_STEPS * 8;
#pragma unroll 1
            for (int i = 0; i < k; ++i) hb[i * 8 + j] = src[i * 8 + j];
            if (j == 0) A.buf.hstate[env * SM_HSTATE_STRIDE + SM_HS_BRAKE_COUNT] = (double)k;
        }
        return;
    }
    human_initial_braking(A.buf.hstate + env * SM_HSTATE_STRIDE, A.buf.hbrake + env * SM_HBRAKE_STEPS * 8,
                          active ? e[j] : 0.0, active ? e[8 + j] : 0.0, active ? e[16 + j] : 0.0, active, lane);
}

// ------------------------------------------------------------------------------------------------------------------
// pools of the nested env (device-side rejection sampling with Philox streams, one warp per entry):
//   start states   get_starting_point_joint_pos_vel_acc with always_use_collision_avoidance_starting_point_sampling
//                  (ctlp.py:1461-1656; Human.__init__ ctlp.py:4723-4729): a random pose with both hands inside the box
//                  and the clearances of the nested env, then with probability p a random feasible (v, a) per joint,
//                  else a random walk with random actions that stops with probability 0.3 per step
//   target points  _add_target_point(robot = r) (ctlp.py:1658-1676): the link point of a random pose of arm r
// Not reproduced: the torque check of the pose sampler (Bullet dynamics) and the braking-trajectory check along the random
// walk; a target point is sampled with the other arm hanging down instead of at its current pose (DESIGN.md).
// ------------------------------------------------------------------------------------------------------------------
// clearance of the human pose whose frames are in W.obx: pairs of the braking-trajectory check; arm_only >= 0 restricts
// them to shapes of arm `arm_only` (frames 101 + 4 r .. 104 + 4 r), the trunk and the table
__device__ __noinline__ bool human_pose_is_free(const float4* verts, const SceneSmem& sm, WarpScratch& W, float thr_static,
                                                float thr_self, int arm_only, int lane) {
    const int np = c_sc.hu.n_brake_pairs;
#pragma unroll 1
    for (int base = 0; base < np; base += 32) {
        const int i = base + lane;
        bool cand = false;
        int ia = 0, ib = 0;
        float thr = 0.f;
        if (i < np) {
            ia = c_sc.hu.brake_pairs[2 * i]; ib = c_sc.hu.brake_pairs[2 * i + 1];
            const int fa = sm.shapes[ia].frame - 100, fb = sm.shapes[ib].frame;
            thr = fb == 0 ? thr_static : thr_self;
            bool use = true;
            if (arm_only >= 0) {
                const bool a_ok = fa >= 1 + 4 * arm_only && fa <= 4 + 4 * arm_only;
                const bool b_ok = fb == 0 || fb == 100 || (fb - 100 >= 1 + 4 * arm_only && fb - 100 <= 4 + 4 * arm_only);
                use = a_ok && b_ok;
            }
            cand = use && pair_lower_bound(sm, ia, ib, W.fr, W.obx) < thr;
        }
        unsigned mask = __ballot_sync(FULL, cand);
#pragma unroll 1
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            const int qa = __shfl_sync(FULL, ia, src), qb = __shfl_sync(FULL, ib, src);
            const float t = __shfl_sync(FULL, thr, src);
            const float d = pair_distance(verts, sm, qa, qb, W.fr, W.obx, t + 0.005f, -1.f, lane, nullptr);
            if (d < t) return false;
        }
    }
    return true;
}

// check_braking_trajectory_method for a candidate start state (ctlp.py:1527-1544): brake from (q, v, a) and check every
// visited pose; lanes 0..7 hold the joints.  true = the braking trajectory is free of collisions and ends at rest.
__device__ __noinline__ bool human_start_state_can_brake(double q, double v, double a, const float4* verts,
                                                         const SceneSmem& sm, WarpScratch& W, int lane) {
    const JointLim& L = c_sc.hu.lim;
    const int j = lane & 7;
    const bool jl = lane < SM_HUMAN_JOINTS;
    const double ts = c_sc.ts, J = L.jerk_max[j], Am = L.acc_max[j];
    const float safety = (float)c_sc.hu.brake_safety;
    double as = a, ae = a;
    {   // _compute_braking_acceleration at the start state
        const bool small0 = fabs(v) < 0.01 && fabs(a) < 0.01;
        if (__all_sync(FULL, !jl || small0)) return true;
        double lo = 0.0, hi = 0.0;
        int code = 0;
        if (jl) safe_range_joint(L, j, q, v, a, lo, hi, code);
        double e = brake_target(v, a, J, Am, ts);
        if (small0) e = 0.0;
        ae = fmin(fmax(e, lo), hi);
    }
#pragma unroll 1
    for (int k = 0; k < 24; ++k) {
        double pend = q;
#pragma unroll 1
        for (int m = 1; m <= c_sc.hu.brake_checks; ++m) {
            double pm, vv, aa;
            interpolate(q, v, as, ae, c_sc.hu.brake_t[m], pm, vv, aa);
            human_fk_scan((float)pm, W.obx, lane);
            const bool free_pose = human_pose_is_free(verts, sm, W, safety, safety, -1, lane);
            __syncwarp();
            if (!free_pose) return false;
            pend = pm;
        }
        if ((double)k * ts > c_sc.hu.brake_timeout) return false;
        double qq, vend, aa;
        interpolate(q, v, as, ae, ts, qq, vend, aa);
        const bool small_j = fabs(vend) < 0.01 && fabs(ae) < 0.01;
        if (__all_sync(FULL, !jl || small_j)) return true;
        double lo = 0.0, hi = 0.0;
        int code = 0;
        if (jl) safe_range_joint(L, j, pend, vend, ae, lo, hi, code);
        double e = brake_target(vend, ae, J, Am, ts);
        if (small_j) e = 0.0;
        e = fmin(fmax(e, lo), hi);
        q = pend; v = vend; as = ae; ae = e;
    }
    return false;
}

struct HumanPoolArgs {
    double* start_pool;
    int start_pool_n;
    double* target_pool;   // [2][target_pool_n][4]
    int target_pool_n;
    uint32_t k0, k1;
};

__global__ void __launch_bounds__(SM_WARPS_PER_BLOCK * 32) fill_human_pool_kernel(HumanPoolArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemLayout Lm = block_prologue(smem_raw, true);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpScratch& W = Lm.scratch[warp];
    const SceneSmem& sm = Lm.bs->scene;
    const float4* verts = Lm.verts;
    const JointLim& L = c_sc.hu.lim;
    const int j = lane & 7;
    const bool jl = lane < SM_HUMAN_JOINTS;
    if (lane == 0) xf_identity(W.fr[0]);
    __syncwarp();
    const int total = A.start_pool_n + 2 * A.target_pool_n;
#pragma unroll 1
    for (int e = blockIdx.x * SM_WARPS_PER_BLOCK + warp; e < total; e += gridDim.x * SM_WARPS_PER_BLOCK) {
        Rng rng(key64(A.k0, A.k1), (uint32_t)e, 0x4A11u);
        if (e >= A.start_pool_n) {   // ---------------- a target point of arm r
            const int r = (e - A.start_pool_n) / A.target_pool_n, slot = (e - A.start_pool_n) % A.target_pool_n;
            V3 p = mk(0.f, 0.f, 0.f);
#pragma unroll 1
            for (int attempt = 0; attempt < 25000; ++attempt) {
                double ql = 0.0;
#pragma unroll 1
                for (int jj = 0; jj < 4; ++jj) {
                    const double u = rng.uniform(L.pos_lo[4 * r + jj], L.pos_hi[4 * r + jj]);
                    if (j == 4 * r + jj) ql = u;
                }
                human_fk_scan((float)ql, W.obx, lane);
                p = human_link_point(W.obx, r);
                bool ok = p.x >= c_sc.hu.tp_box_min[0] && p.x <= c_sc.hu.tp_box_max[0] && p.y >= c_sc.hu.tp_box_min[1] &&
                          p.y <= c_sc.hu.tp_box_max[1] && p.z >= c_sc.hu.tp_box_min[2] && p.z <= c_sc.hu.tp_box_max[2];
                if (ok) ok = human_pose_is_free(verts, sm, W, (float)c_sc.hu.tp_min_static, (float)c_sc.hu.tp_min_self, r, lane);
                __syncwarp();
                if (ok) break;
            }
            if (lane == 0) {
                double* o = A.target_pool + ((size_t)r * A.target_pool_n + slot) * 4;
                o[0] = (double)p.x; o[1] = (double)p.y; o[2] = (double)p.z; o[3] = 0.0;
            }
            __syncwarp();
            continue;
        }
        // ---------------- a start state
        double q = 0.0, v = 0.0, a = 0.0;
        uint32_t lane_ctr = 0;
#pragma unroll 1
        for (int outer = 0; outer < 1000; ++outer) {
#pragma unroll 1
            for (int attempt = 0; attempt < 100000; ++attempt) {
#pragma unroll 1
                for (int jj = 0; jj < SM_HUMAN_JOINTS; ++jj) {
                    const double u = rng.uniform(L.pos_lo[jj], L.pos_hi[jj]);
                    if (j == jj) q = u;
                }
                human_fk_scan((float)q, W.obx, lane);
                bool ok = true;
#pragma unroll 1
                for (int r = 0; r < 2; ++r) {
                    const V3 p = human_link_point(W.obx, r);
                    ok = ok && p.x >= c_sc.hu.start_box_min[0] && p.x <= c_sc.hu.start_box_max[0] && p.y >= c_sc.hu.start_box_min[1] &&
                         p.y <= c_sc.hu.start_box_max[1] && p.z >= c_sc.hu.start_box_min[2] && p.z <= c_sc.hu.start_box_max[2];
                }
                if (ok) ok = human_pose_is_free(verts, sm, W, (float)c_sc.hu.min_start_static, (float)c_sc.hu.min_start_self, -1, lane);
                __syncwarp();
                if (ok) break;
            }
            v = 0.0; a = 0.0;
            if (rng.uniform() < c_sc.hu.kinematic_sampling_probability) {   // ctlp.py:1494-1556
                bool found = false;
                if (jl) {
#pragma unroll 1
                    for (int iv = 0; iv < 5 && !found; ++iv) {
                        const uint4 r = philox((uint32_t)e, 0x7000u + lane_ctr++, (uint32_t)lane, 0x4A12u, A.k0, A.k1);
                        const double vj = L.vel_max[j] * (2.0 * u01d(r.x, r.y) - 1.0);
#pragma unroll 1
                        for (int ia = 0; ia < 10 && !found; ++ia) {
                            const uint4 r2 = philox((uint32_t)e, 0x7000u + lane_ctr++, (uint32_t)lane, 0x4A13u, A.k0, A.k1);
                            const double aj = L.acc_max[j] * (2.0 * u01d(r2.x, r2.y) - 1.0);
                            double lo, hi;
                            int code;
                            safe_range_joint(L, j, q, vj, aj, lo, hi, code);
                            if (code == 0) { found = true; v = vj; a = aj; }
                        }
                    }
                }
                if (!__all_sync(FULL, !jl || found)) continue;
                // the state must be able to brake without a collision (ctlp.py:1527-1544)
                if (!c_sc.hu.check_braking || human_start_state_can_brake(q, v, a, verts, sm, W, lane)) break;
                continue;
            }
            // random walk from rest with random actions (ctlp.py:1558-1654); the braking-trajectory method is applied to
            // the state the walk ends in instead of to every step
#pragma unroll 1
            for (int step = 0; step < 64; ++step) {
                if (rng.uniform() < c_sc.hu.stay_in_state_probability) break;
                const uint4 r = philox((uint32_t)e, 0x7000u + lane_ctr++, (uint32_t)lane, 0x4A14u, A.k0, A.k1);
                if (jl) {
                    double lo, hi, qe, ve, as_;
                    int code;
                    safe_range_joint(L, j, q, v, a, lo, hi, code);
                    const double un = 2.0 * u01d(r.x, r.y) - 1.0;
                    const double a1 = lo + 0.5 * (un + 1.0) * (hi - lo);
                    interpolate(q, v, a, a1, c_sc.ts, qe, ve, as_);
                    q = qe; v = ve; a = a1;
                }
            }
            if (!c_sc.hu.check_braking || human_start_state_can_brake(q, v, a, verts, sm, W, lane)) break;
        }
        if (jl) {
            double* o = A.start_pool + (size_t)e * SM_HPOOL_STRIDE;
            o[j] = q; o[8 + j] = v; o[16 + j] = a; o[24 + j] = 0.0;
        }
        __syncwarp();
    }
}
