// smenv_pools.cuh -- device-side rejection sampling of start states and ball launches (one warp per pool entry),
// reset, and the parity hooks.
//
// Restates, with Philox streams instead of the global np.random stream (safe_motions_base.py:1704-1710):
//   * get_starting_point_joint_pos_vel_acc / _get_collision_free_robot_position   ctlp.py:1461-1656, :1980-2138
//   * Planet.reset (collision-free random phase)                                   ctlp.py:4470-4501
//   * _add_moving_object / _get_moving_object_release_point / Ball.__init__        ctlp.py:1723-1954, :4010-4101
//   * the random initial ball time of ObstacleWrapperSim.reset                     ctlp.py:1090-1111
// The torque check of the reference's pose sampler (one Bullet stepSimulation, ctlp.py:2091-2111) needs rigid-body
// dynamics and is not reproduced (DESIGN.md, deviations).
#pragma once
#include "smenv_kernels.cuh"

struct PoolArgs {
    double* start_pool;
    int start_pool_n;
    double* ball_pool;
    int ball_pool_n;
    uint32_t k0, k1;
    const double* hstart_pool;   // Human scene: start states of the nested env, entry e pairs with start-pool entry e
};
#define SM_HPOOL_STRIDE 32     /* doubles per entry of the human start pool: q[8] v[8] a[8] spare[8] */

__device__ __forceinline__ uint64_t key64(uint32_t k0, uint32_t k1) { return ((uint64_t)k1 << 32) | k0; }

// static / self clearance of the pose whose frames are in W.fr (ctlp.py:2140-2208): query distance thr + 0.005,
// violated if d < thr
__device__ __noinline__ bool pose_is_free(const float4* verts, const SceneSmem& sm, WarpScratch& W, float thr_static,
                                          float thr_self, int lane) {
    float cap = thr_static + 0.005f;
    float d = min_pairs(verts, sm, 0, sm.static_pairs, nullptr, c_sc.n_static_pairs, 1, 0, cap, cap, W.fr, W.obx, lane,
                        nullptr);
    if (d < thr_static) return false;
    cap = thr_self + 0.005f;
    d = min_pairs(verts, sm, 0, sm.self_pairs, nullptr, c_sc.n_self_pairs, 1, 0, cap, cap, W.fr, W.obx, lane, nullptr);
    return !(d < thr_self);
}

// Random joint vector with the target point inside the box and the static / self distances above the thresholds
// (_get_collision_free_robot_position, ctlp.py:1980-2138).  Lane j gets q_j; frames are left in W.fr.
__device__ __noinline__ double sample_free_pose(Rng& rng, const float4* verts, const SceneSmem& sm, WarpScratch& W,
                                                const double* box_min, const double* box_max, float thr_static,
                                                float thr_self, V3& target, int lane) {
    const int nj = c_sc.n_joints, j = lane & 7;
    const float ox = c_sc.target_t[0] + c_sc.target_R[0] * c_sc.target_offset[0] +
                     c_sc.target_R[1] * c_sc.target_offset[1] + c_sc.target_R[2] * c_sc.target_offset[2];
    const float oy = c_sc.target_t[1] + c_sc.target_R[3] * c_sc.target_offset[0] +
                     c_sc.target_R[4] * c_sc.target_offset[1] + c_sc.target_R[5] * c_sc.target_offset[2];
    const float oz = c_sc.target_t[2] + c_sc.target_R[6] * c_sc.target_offset[0] +
                     c_sc.target_R[7] * c_sc.target_offset[1] + c_sc.target_R[8] * c_sc.target_offset[2];
    int attempts = 0;
    double ql = 0.0;
#pragma unroll 1
    while (true) {
        ++attempts;
#pragma unroll 1
        for (int jj = 0; jj < nj; ++jj) {  // np.random.uniform(lower, upper) (ctlp.py:2035-2037)
            double r = rng.uniform(c_sc.pos_lo[jj], c_sc.pos_hi[jj]);
            if (j == jj) ql = r;
        }
        frames_from_q64(sm, ql, W.fr, lane);
        target = xf_apply(W.fr[nj], ox, oy, oz);
        bool ok = target.x >= box_min[0] && target.x <= box_max[0] && target.y >= box_min[1] &&
                  target.y <= box_max[1] && target.z >= box_min[2] && target.z <= box_max[2];  // ctlp.py:2054-2061
        if (ok) ok = pose_is_free(verts, sm, W, thr_static, thr_self, lane);
        __syncwarp();
        if (ok || attempts >= 100000) break;
    }
    return ql;
}

// Ball.get_target_height_time (ctlp.py:4346-4361); NaN if the height is never reached
__device__ __noinline__ double target_height_time(double h0, double vz, double h) {
    const double g = 9.81;
    double sq = vz * vz + 2.0 * g * (h0 - h);
    if (sq >= 0.0) {
        double t = (vz + sqrt(sq)) / g;
        if (t > 0.0) return t;
    }
    return nan("");
}

__global__ void __launch_bounds__(SM_WARPS_PER_BLOCK * 32) fill_ball_pool_kernel(PoolArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemLayout L = block_prologue(smem_raw, true);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpScratch& W = L.scratch[warp];
    const SceneSmem& sm = L.bs->scene;
    const float4* verts = L.verts;
    const double g = 9.81, spd = c_sc.ball_speed, rad = c_sc.ball_radius;
    const double upd = c_sc.ts / (double)c_sc.substeps;
#pragma unroll 1
    for (int e = blockIdx.x * SM_WARPS_PER_BLOCK + warp; e < A.ball_pool_n; e += gridDim.x * SM_WARPS_PER_BLOCK) {
        Rng rng(key64(A.k0, A.k1), (uint32_t)e, 0xBA11u);
        double rel[3] = {0, 0, 0}, vel[3] = {0, 0, 1}, nmax = 0.0, nhit = 0.0;
#pragma unroll 1
        for (int attempt = 0; attempt < 25000; ++attempt) {
            // release point on the sphere segment (ctlp.py:1943-1952)
            double h = rng.uniform(c_sc.ball_height_min, c_sc.ball_height_max);
            double rr = sqrt(c_sc.ball_sphere_radius * c_sc.ball_sphere_radius - h * h);
            double ang = rng.uniform(c_sc.ball_angle_min, c_sc.ball_angle_max);
            rel[0] = c_sc.ball_sphere_center[0] + rr * cos(ang);
            rel[1] = c_sc.ball_sphere_center[1] + rr * sin(ang);
            rel[2] = c_sc.ball_sphere_center[2] + h;
            // aim at the target point of a random collision-free robot pose (ctlp.py:1782-1790)
            V3 tgt;
            sample_free_pose(rng, verts, sm, W, c_sc.ball_target_box_min, c_sc.ball_target_box_max,
                             (float)c_sc.ball_target_min_static, (float)c_sc.ball_target_min_self, tgt, lane);
            double dx = (double)tgt.x - rel[0], dy = (double)tgt.y - rel[1], dh = (double)tgt.z - rel[2];
            double dxy = sqrt(dx * dx + dy * dy);
            double num = spd * spd * spd * spd - g * (g * dxy * dxy + 2.0 * dh * spd * spd);  // ctlp.py:1797
            bool valid = num >= 0.0 && dxy > 0.0;
            if (valid) {
                bool high = rng.uniform() <= c_sc.ball_high_angle_probability;
                double theta = atan((spd * spd + (high ? 1.0 : -1.0) * sqrt(num)) / (g * dxy));
                vel[2] = spd * sin(theta);
                vel[0] = spd * cos(theta) * dx / dxy;
                vel[1] = spd * cos(theta) * dy / dxy;
            }
            if (valid && c_sc.ball_check_invalid) {  // ctlp.py:1813-1848
                double tt = target_height_time(rel[2], vel[2], c_sc.ball_invalid_max[2] + rad);
                double tb = target_height_time(rel[2], vel[2], c_sc.ball_invalid_min[2] + rad);
                double xt = rel[0] + vel[0] * tt, yt = rel[1] + vel[1] * tt;
                double xb = rel[0] + vel[0] * tb, yb = rel[1] + vel[1] * tb;
                bool in_top = !isnan(tt) && xt >= c_sc.ball_invalid_min[0] && xt <= c_sc.ball_invalid_max[0] &&
                              yt >= c_sc.ball_invalid_min[1] && yt <= c_sc.ball_invalid_max[1];
                bool in_bot = !isnan(tb) && xb >= c_sc.ball_invalid_min[0] && xb <= c_sc.ball_invalid_max[0] &&
                              yb >= c_sc.ball_invalid_min[1] && yb <= c_sc.ball_invalid_max[1];
                if (in_top || in_bot) valid = false;
            }
            double final_t = nan("");
            if (valid) {  // Ball.get_final_ball_position (ctlp.py:4304-4344): straight-line exit of the box, or floor
#pragma unroll 1
                for (int i = 0; i < 2; ++i) {
                    int ia = (i + 1) % 3, ib = (i + 2) % 3;
                    if (vel[i] != 0.0) {
#pragma unroll 1
                        for (int mm = 0; mm < 2; ++mm) {
                            double bound = mm == 0 ? c_sc.ball_final_min[i] : c_sc.ball_final_max[i];
                            double t = (bound - rel[i]) / vel[i];
                            double pa = rel[ia] + vel[ia] * t, pb = rel[ib] + vel[ib] * t;
                            if (pa >= c_sc.ball_final_min[ia] && pa <= c_sc.ball_final_max[ia] &&
                                pb >= c_sc.ball_final_min[ib] && pb <= c_sc.ball_final_max[ib]) {
                                if (isnan(final_t) || t > final_t) final_t = t;
                            }
                        }
                    }
                }
                double mht = target_height_time(rel[2], vel[2], c_sc.ball_final_min[2]);
                if (!isnan(mht) && (isnan(final_t) || mht < final_t)) final_t = mht;
                if (isnan(final_t)) valid = false;  // the reference raises here; resample instead
            }
            if (valid) {
                nmax = floor(final_t / upd);  // ctlp.py:4101
                bool table = false;
                if (c_sc.has_table) {  // ctlp.py:1889-1904
                    double ht = target_height_time(rel[2], vel[2], rad);
                    double px = rel[0] + vel[0] * ht, py = rel[1] + vel[1] * ht;
                    if (px >= -0.6 && px <= 0.6 && py >= -0.8 && py <= 0.8) {
                        nhit = rint(ht / upd) - 1.0;
                        table = true;
                    }
                }
                if (!table) {  // ctlp.py:1906-1915
                    double ht = target_height_time(rel[2], vel[2], c_sc.plane_z + rad);
                    nhit = rint(ht / upd) - 1.0;
                }
                break;
            }
        }
        // initial orientation: rotation taking +z onto the flight direction, as euler angles (ctlp.py:4029-4034)
        double n = sqrt(vel[0] * vel[0] + vel[1] * vel[1] + vel[2] * vel[2]);
        double bx = vel[0] / n, by = vel[1] / n, bz = vel[2] / n;
        double kk = 1.0 / (1.0 + bz);
        double e0 = atan2(by, bz), e1 = -asin(fmax(-1.0, fmin(1.0, bx))), e2 = atan2(-bx * by * kk, 1.0 - bx * bx * kk);
        double omega = rng.uniform(0.0, 2.0 * 3.14159265358979323846);  // ctlp.py:4056-4057
        if (lane == 0) {
            double* o = A.ball_pool + (size_t)e * SM_BALL_STRIDE;
            o[0] = rel[0]; o[1] = rel[1]; o[2] = rel[2];
            o[3] = vel[0]; o[4] = vel[1]; o[5] = vel[2];
            o[6] = e0; o[7] = e1; o[8] = e2;
            o[9] = omega; o[10] = nmax; o[11] = nhit;
        }
    }
}

__global__ void __launch_bounds__(SM_WARPS_PER_BLOCK * 32) fill_start_pool_kernel(PoolArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemLayout L = block_prologue(smem_raw, true);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpScratch& W = L.scratch[warp];
    const SceneSmem& sm = L.bs->scene;
    const float4* verts = L.verts;
    const int nj = c_sc.n_joints, j = lane & 7, S = c_sc.substeps;
    const bool jl = lane < nj;
    const float thr_s = (float)c_sc.min_start_distance, thr_self = (float)c_sc.min_start_self;
    const double dt = xdiv(c_sc.ts, (double)S), tvdt = xmul(c_sc.track_vel, dt);
    const int kind = c_sc.n_obstacles > 0 ? c_sc.obst_kind[0] : SM_OBST_NONE;
#pragma unroll 1
    for (int e = blockIdx.x * SM_WARPS_PER_BLOCK + warp; e < A.start_pool_n; e += gridDim.x * SM_WARPS_PER_BLOCK) {
        Rng rng(key64(A.k0, A.k1), (uint32_t)e, 0x51A7u);
        double q = 0.0, v = 0.0, a = 0.0;
        uint32_t lane_ctr = 0;
        if (kind == SM_OBST_HUMAN && A.hstart_pool) {   // the human of this pool entry, at its start pose
            human_fk_scan((float)A.hstart_pool[(size_t)e * SM_HPOOL_STRIDE + (lane & 7)], W.obx, lane);
        }
#pragma unroll 1
        for (int hretry = 0; hretry < 200; ++hretry) {
#pragma unroll 1
        for (int outer = 0; outer < 1000; ++outer) {
            V3 tgt;
            q = sample_free_pose(rng, verts, sm, W, c_sc.start_box_min, c_sc.start_box_max, thr_s, thr_self, tgt, lane);
            v = 0.0; a = 0.0;
            if (c_sc.start_at_rest) break;   // not collision_avoidance_mode: the pose at rest (ctlp.py:1461-1500)
            if (rng.uniform() < c_sc.kinematic_sampling_probability) {
                // per joint: up to 5 velocities x 10 accelerations with violation code 0 (ctlp.py:1503-1525)
                bool found = false;
                if (jl) {
#pragma unroll 1
                    for (int iv = 0; iv < 5 && !found; ++iv) {
                        uint4 r = philox((uint32_t)e, 0x7000u + lane_ctr++, (uint32_t)lane, 0x51A8u, A.k0, A.k1);
                        double vj = c_sc.vel_max[j] * (2.0 * u01d(r.x, r.y) - 1.0);
#pragma unroll 1
                        for (int ia = 0; ia < 10 && !found; ++ia) {
                            uint4 r2 = philox((uint32_t)e, 0x7000u + lane_ctr++, (uint32_t)lane, 0x51A9u, A.k0, A.k1);
                            double aj = c_sc.acc_max[j] * (2.0 * u01d(r2.x, r2.y) - 1.0);
                            double lo, hi;
                            int code;
                            safe_range_joint(j, q, vj, aj, lo, hi, code);
                            if (code == 0) { found = true; v = vj; a = aj; }
                        }
                    }
                }
                if (__all_sync(FULL, !jl || found)) break;
                continue;  // some joint found no feasible (v, a): new pose (ctlp.py:1547-1556)
            }
            // random walk from rest with random actions (ctlp.py:1558-1654); h0 = oldest ... h2 = newest state
            double hq0 = q, hq1 = q, hq2 = q, hv0 = 0, hv1 = 0, hv2 = 0, ha0 = 0, ha1 = 0, ha2 = 0;
            int len = 1;
#pragma unroll 1
            while (true) {
                if (rng.uniform() < c_sc.stay_in_state_probability) { q = hq2; v = hv2; a = ha2; break; }
                double lo = 0.0, hi = 0.0, qe = hq2, ve = hv2, ae = ha2;
                int code;
                uint4 r = philox((uint32_t)e, 0x7000u + lane_ctr++, (uint32_t)lane, 0x51AAu, A.k0, A.k1);
                if (jl) {
                    safe_range_joint(j, hq2, hv2, ha2, lo, hi, code);
                    double un = 2.0 * u01d(r.x, r.y) - 1.0;
                    double a1 = lo + 0.5 * (un + 1.0) * (hi - lo);  // denormalize (ctlp.py:1577-1578)
                    double as_;
                    interpolate(hq2, hv2, ha2, a1, c_sc.ts, qe, ve, as_);
                    ae = a1;
                }
                frames_from_q64(sm, qe, W.fr, lane);
                bool free_pose = pose_is_free(verts, sm, W, thr_s, thr_self, lane);
                __syncwarp();
                if (free_pose) {
                    hq0 = hq1; hv0 = hv1; ha0 = ha1;
                    hq1 = hq2; hv1 = hv2; ha1 = ha2;
                    hq2 = qe; hv2 = ve; ha2 = ae;
                    ++len;
                } else {  // collision: one of the three latest states (ctlp.py:1638-1648)
                    int m = len < 3 ? len : 3;
                    int sel = 1 + (int)(rng.next4().x % (uint32_t)m);
                    q = sel == 1 ? hq2 : sel == 2 ? hq1 : hq0;
                    v = sel == 1 ? hv2 : sel == 2 ? hv1 : hv0;
                    a = sel == 1 ? ha2 : sel == 2 ? ha1 : ha0;
                    break;
                }
            }
            break;
        }
        // ---------------- obstacles at reset
        frames_from_q64(sm, q, W.fr, lane);
        if (kind != SM_OBST_HUMAN || !A.hstart_pool) break;
        {   // "Collision with human." (ctlp.py:2113-2121): the start pose keeps the minimum distance to the human
            const float thr = (float)c_sc.min_start_distance;
            const float d = min_pairs(verts, sm, 1, nullptr, sm.mov_reward, c_sc.n_mov_reward * c_sc.obst_shape_cnt[0],
                                      c_sc.obst_shape_cnt[0], c_sc.obst_shape_off[0], thr + 0.005f, thr + 0.005f, W.fr, W.obx,
                                      lane, nullptr);
            __syncwarp();
            if (!(d < thr)) break;
        }
        }
        double ob = 0.0;
        if (kind == SM_OBST_PLANET) {  // Planet.reset: random phase without contact (ctlp.py:4470-4501)
            int idx = 0;
#pragma unroll 1
            for (int t = 0; t < 1000; ++t) {
                idx = (int)(rng.next4().x % (uint32_t)c_sc.planet_steps);
                if (lane < c_sc.n_obstacles) planet_pose(lane, idx, W.obx2[lane]);
                __syncwarp();
                bool hit = false;
                for (int o = 0; o < c_sc.n_obstacles && !hit; ++o)
                    hit = contact_exists(verts, sm, o, W.fr, W.obx2, lane, nullptr);
                __syncwarp();
                if (!hit) break;
            }
            // the first obstacle_wrapper.update after the reset advances the planets once (ctlp.py:2626-2629)
            if (lane == SM_OB_INDEX) ob = (double)((idx + 1) % c_sc.planet_steps);
        } else if (kind == SM_OBST_BALL && A.ball_pool_n > 0) {
            const double* b = A.ball_pool + (size_t)(rng.next4().x % (uint32_t)A.ball_pool_n) * SM_BALL_STRIDE;
            if (lane < 10) W.ob[SM_OB_BALL_P0 + lane] = b[lane];
            __syncwarp();
            double nmax = b[10], nhit = b[11];
            double n0 = 0.0;
            if (c_sc.ball_random_initial) {  // ctlp.py:1090-1111
                double mc = nhit < nmax ? nhit : nmax;
                int max_ts = (int)floor(mc / (double)S);
                if (max_ts < 0) max_ts = 0;
#pragma unroll 1
                for (int t = 0; t < 1000; ++t) {
                    n0 = (double)((int)(rng.next4().x % (uint32_t)(max_ts + 1)) * S);
                    if (lane == 0) ball_pose(W.ob, n0 * dt, W.obx2[0]);
                    __syncwarp();
                    bool hit = contact_exists(verts, sm, 0, W.fr, W.obx2, lane, nullptr);
                    __syncwarp();
                    if (!hit) break;
                }
            }
            if (lane == SM_OB_INDEX) ob = n0;
            if (lane >= SM_OB_BALL_P0 && lane < SM_OB_BALL_P0 + 10) ob = b[lane - SM_OB_BALL_P0];
            if (lane == SM_OB_BALL_T) ob = xmul(n0, dt);  // set_position_update_step_counter (ctlp.py:4257-4259)
            if (lane == SM_OB_BALL_ACTIVE) ob = 1.0;
            if (lane == SM_OB_BALL_NMAX) ob = nmax;
            if (lane == SM_OB_BALL_NHIT) ob = nhit;
        }
        // ---------------- write the entry: kin record (q, v, a, q_act) + obstacle record
        double qact = xadd(q, xmul(tvdt, v));  // pose after the reset's stepSimulation (safe_motions_base.py:973-978)
        double qq = shfl_d(q, j), vv = shfl_d(v, j), aa = shfl_d(a, j), tt = shfl_d(qact, j);
        int grp = lane >> 3;
        double* o = A.start_pool + (size_t)e * SM_POOL_STRIDE;
        o[lane] = j < nj ? (grp == 0 ? qq : grp == 1 ? vv : grp == 2 ? aa : tt) : 0.0;
        if (lane < SM_OBST_STRIDE) o[SM_KIN_STRIDE + lane] = ob;
        __syncwarp();
    }
}

// reset of the masked envs from the start pool + first observation (observations.py:144-187)
struct ResetArgs {
    SmBuffers buf;
    int n;
    const uint8_t* mask;
    const double* start_pool;
    int start_pool_n;
    const double* target_pool;
    int target_pool_n;
    uint32_t k0, k1;
    const int* entry;   // [n] pool entry of env i (the pool check, smenv_set_initial_backup_check), NULL: drawn
};

// injected first target points (parity protocol) or, with first_target == NULL, draws from the pool
__global__ void target_init_kernel(SmBuffers buf, int n, const double* first_target, const uint8_t* mask,
                                   const double* pool, int pool_n, uint32_t k0, uint32_t k1) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= n || !buf.target || (mask && !mask[env])) return;
    double* tp = buf.target + (size_t)env * SM_TP_STRIDE;
    target_episode_start(tp, buf.kin + (size_t)env * SM_KIN_STRIDE, first_target ? first_target + 3 * (size_t)env : nullptr,
                         pool, pool_n, env, k0, k1);
}

// target points of the reaching task: the target link point of a random collision-free pose inside the target box
// (_add_target_point, ctlp.py:1658-1676 -> _get_collision_free_robot_position); the torque check of the sampler is
// not reproduced (DESIGN.md)
__global__ void __launch_bounds__(SM_WARPS_PER_BLOCK * 32) fill_target_pool_kernel(double* pool, int pool_n, uint32_t k0,
                                                                                    uint32_t k1) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemLayout L = block_prologue(smem_raw, true);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpScratch& W = L.scratch[warp];
#pragma unroll 1
    for (int e = blockIdx.x * SM_WARPS_PER_BLOCK + warp; e < pool_n; e += gridDim.x * SM_WARPS_PER_BLOCK) {
        Rng rng(key64(k0, k1), (uint32_t)e, 0x7A27u);
        V3 tgt;
        sample_free_pose(rng, L.verts, L.bs->scene, W, c_sc.tp_box_min, c_sc.tp_box_max, (float)c_sc.tp_min_static,
                         (float)c_sc.tp_min_self, tgt, lane);
        if (lane == 0) {
            double* o = pool + (size_t)e * 4;
            o[0] = (double)tgt.x; o[1] = (double)tgt.y; o[2] = (double)tgt.z; o[3] = 0.0;
        }
        __syncwarp();
    }
}
__global__ void __launch_bounds__(256) reset_kernel(ResetArgs A) {
    const int lane = threadIdx.x & 31;
    const int env = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (env >= A.n) return;
    if (A.mask && !A.mask[env]) return;
    int4 ep = *reinterpret_cast<const int4*>(A.buf.episode + 4 * (size_t)env);
    uint4 r = philox((uint32_t)env, (uint32_t)ep.y, 0x5E7u, 1u, A.k0, A.k1);
    const uint32_t pick = A.entry ? (uint32_t)A.entry[env] : r.x % (uint32_t)A.start_pool_n;
    const double* e = A.start_pool + (size_t)pick * SM_POOL_STRIDE;
    A.buf.kin[(size_t)env * SM_KIN_STRIDE + lane] = e[lane];
    if (lane < SM_OBST_STRIDE) A.buf.obst[(size_t)env * SM_OBST_STRIDE + lane] = e[SM_KIN_STRIDE + lane];
    if (lane == 0) {
        *reinterpret_cast<int4*>(A.buf.episode + 4 * (size_t)env) = make_int4(0, ep.y + 1, ep.z, 0);
        A.buf.ep_return[env] = 0.0;
        if (A.buf.done) A.buf.done[env] = 0;
    }
    double* tp = (c_sc.use_target_points && A.buf.target) ? A.buf.target + (size_t)env * SM_TP_STRIDE : nullptr;
    if (tp) {
        if (lane == 0) target_episode_start(tp, e, nullptr, A.target_pool, A.target_pool_n, env, A.k0, A.k1);
        __syncwarp();
    }
    write_observation(A.buf.obs + (size_t)env * c_sc.obs_size, e, e + SM_KIN_STRIDE, tp, lane, 32,
                      A.buf.hobs ? A.buf.hobs + (size_t)env * SM_HOBS_STRIDE : nullptr);
}

// ---------------- the initial-backup-trajectory check of the start pool (smenv_set_initial_backup_check)
__global__ void pool_entry_kernel(int* entry, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) entry[i] = i;
}

// Stable partition of the pool by verdict: dest[e] is the new position of entry e, the passing entries (verdict 0) first
// and the failing ones after them, each in their original order; *passed is the number of passing entries.  One CTA:
// every thread counts a contiguous run of entries, a scan over the runs gives each run its first positions.
#define SM_PARTITION_THREADS 1024
__global__ void __launch_bounds__(SM_PARTITION_THREADS) pool_partition_kernel(const float* verdict, int n, int* dest,
                                                                              int* passed) {
    __shared__ int s_scan[SM_PARTITION_THREADS];
    const int t = threadIdx.x;
    const int per = (n + SM_PARTITION_THREADS - 1) / SM_PARTITION_THREADS;
    const int e0 = min(n, t * per), e1 = min(n, e0 + per);
    int cnt = 0;
#pragma unroll 1
    for (int e = e0; e < e1; ++e) cnt += verdict[e] == 0.0f;
    s_scan[t] = cnt;
    __syncthreads();
#pragma unroll 1
    for (int off = 1; off < SM_PARTITION_THREADS; off <<= 1) {   // inclusive scan of the run counts
        const int v = t >= off ? s_scan[t - off] : 0;
        __syncthreads();
        s_scan[t] += v;
        __syncthreads();
    }
    const int total = s_scan[SM_PARTITION_THREADS - 1];
    int before = s_scan[t] - cnt;   // passing entries before entry e
#pragma unroll 1
    for (int e = e0; e < e1; ++e) dest[e] = verdict[e] == 0.0f ? before++ : total + (e - before);
    if (t == 0) *passed = total;
}

// dst[dest[e]] = src[e] for the n records of `stride` elements of a pool array
template <typename T>
__global__ void pool_scatter_kernel(const T* __restrict__ src, T* __restrict__ dst, const int* __restrict__ dest, int n,
                                    int stride) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * stride) return;
    const size_t e = i / stride, k = i % stride;
    dst[(size_t)dest[e] * stride + k] = src[i];
}

// observation only (after smenv_set_state)
__global__ void __launch_bounds__(256) observation_kernel(SmBuffers buf, int n) {
    const int lane = threadIdx.x & 31;
    const int env = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (env >= n) return;
    write_observation(buf.obs + (size_t)env * c_sc.obs_size, buf.kin + (size_t)env * SM_KIN_STRIDE,
                      buf.obst + (size_t)env * SM_OBST_STRIDE,
                      (c_sc.use_target_points && buf.target) ? buf.target + (size_t)env * SM_TP_STRIDE : nullptr, lane, 32,
                      buf.hobs ? buf.hobs + (size_t)env * SM_HOBS_STRIDE : nullptr);
}

// ---------------- parity hooks: pieces of the step on caller-supplied states
__global__ void safe_range_kernel(const double* kin, double* lo, double* hi, int32_t* code, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int env = i >> 3, j = i & 7;
    if (env >= n || j >= c_sc.n_joints) return;
    const double* k = kin + (size_t)env * SM_KIN_STRIDE;
    double l, h;
    int c;
    // same two-path evaluation as the step: the light path with the conservative position filter, the full
    // iterative solve only where the filter cannot rule the position bounds out
    bool need_pos;
    safe_range_light(j, k[j], k[8 + j], k[16 + j], l, h, c, need_pos);
    if (need_pos) safe_range_joint(j, k[j], k[8 + j], k[16 + j], l, h, c);
    lo[env * SM_MAX_JOINTS + j] = l;
    hi[env * SM_MAX_JOINTS + j] = h;
    code[env * SM_MAX_JOINTS + j] = c;
}

__global__ void __launch_bounds__(SM_WARPS_PER_BLOCK * 32)
distances_kernel(const double* kin, const double* obst, float* d_static, float* d_self, float* d_moving, int n) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemLayout L = block_prologue(smem_raw, true);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpScratch& W = L.scratch[warp];
    const SceneSmem& sm = L.bs->scene;
    const int kind = c_sc.n_obstacles > 0 ? c_sc.obst_kind[0] : SM_OBST_NONE;
#pragma unroll 1
    for (int env = blockIdx.x * SM_WARPS_PER_BLOCK + warp; env < n; env += gridDim.x * SM_WARPS_PER_BLOCK) {
        if (lane < SM_OBST_STRIDE) W.ob[lane] = obst[(size_t)env * SM_OBST_STRIDE + lane];
        __syncwarp();
        frames_from_q64(sm, kin[(size_t)env * SM_KIN_STRIDE + (lane & 7)], W.fr, lane);
        if (kind == SM_OBST_PLANET && lane < c_sc.n_obstacles) planet_pose(lane, (int)W.ob[SM_OB_INDEX], W.obx[lane]);
        if (kind == SM_OBST_BALL && lane == 0) ball_pose(W.ob, W.ob[SM_OB_BALL_T], W.obx[0]);
        __syncwarp();
        float ds, dse, dm;
        all_distances(L.verts, sm, W.fr, W.obx, W.ob[SM_OB_LATCH] != 0.0,
                      kind == SM_OBST_BALL && W.ob[SM_OB_BALL_ACTIVE] == 0.0, ds, dse, dm, lane, nullptr);
        __syncwarp();
        if (lane == 0) { d_static[env] = ds; d_self[env] = dse; d_moving[env] = dm; }
    }
}

// debug hook: trace of one GJK call (8 floats per iteration: simplex size, |v|^2, v.w, support ids, v)
__global__ void __launch_bounds__(32) debug_gjk_kernel(const double* kin, const double* obst, int ia, int ib, float upper,
                                                       float* trace, float* result) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmemLayout L = block_prologue(smem_raw, true);
    const int lane = threadIdx.x & 31;
    WarpScratch& W = L.scratch[0];
    const SceneSmem& sm = L.bs->scene;
    const int kind = c_sc.n_obstacles > 0 ? c_sc.obst_kind[0] : SM_OBST_NONE;
    if (lane < SM_OBST_STRIDE) W.ob[lane] = obst[lane];
    __syncwarp();
    frames_from_q64(sm, kin[lane & 7], W.fr, lane);
    if (kind == SM_OBST_PLANET && lane < c_sc.n_obstacles) planet_pose(lane, (int)W.ob[SM_OB_INDEX], W.obx[lane]);
    if (kind == SM_OBST_BALL && lane == 0) ball_pose(W.ob, W.ob[SM_OB_BALL_T], W.obx[0]);
    __syncwarp();
    GjkCounters cnt = {0u, 0u, 0u, trace};
    float d = pair_distance(L.verts, sm, ia, ib, W.fr, W.obx, upper, -1.f, lane, &cnt);
    if (lane == 0) { result[0] = d; result[1] = (float)cnt.iters; }
    if (lane <= c_sc.n_joints) for (int i = 0; i < 12; ++i) result[4 + 12 * lane + i] = i < 9 ? W.fr[lane].r[i] : W.fr[lane].t[i - 9];
}
