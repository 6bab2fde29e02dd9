// smenv.cu -- C ABI of libsmenv.so (include/smenv.h): scene upload, pools, reset, step.  sm_100a only, no CPU path.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <algorithm>
#include <array>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

#include "smenv_pools.cuh"
#include "smenv_step.cuh"
#include "smenv_mlp.cuh"
#include "smenv_human.cuh"

static thread_local std::string g_error;
static int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}
#define CU(call)                                                                                            \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess)                                                                              \
            return fail(SM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                   \
    } while (0)

// ------------------------------------------------------------------------------------------------------------------
// Support-direction table of one hull (layout: smenv_device.cuh).  A vertex is listed for a cell if, for some sample
// direction of the cell (a (SUB x SUB) grid that includes the cell border), its support value is within
// diam * (distance to the nearest sample) of the maximum -- then it is listed for every direction of the cell it
// could win.  Float rounding of lut_cell on the device at a cell border is covered by the same slack.
// Two passes: a coarse grid (17 or 33 samples per cell edge) over all vertices gives a superset of the candidates; a
// fine grid (1 / 512 of a face edge between samples, slack eight times smaller) over that superset alone thins it to nearly
// the exact set.  The lists set the trip count of the support loop of a whole GJK warp (its longest list), so every
// listed vertex that cannot win costs time in every step: 17 -> 9 candidates on average for an iiwa link.
// SMENV_LUT_FINE=0 keeps the coarse pass only (experiments).
// ------------------------------------------------------------------------------------------------------------------
static void build_lut_uncached(const float4* v, int n, int R, std::vector<uint32_t>& out);

// tables are cached per process (keyed by the vertex bytes): every env of a scene shares the same hulls
static void build_lut(const float4* v, int n, int R, std::vector<uint32_t>& out) {
    static std::mutex mu;
    static std::map<std::string, std::vector<uint32_t>> cache;
    const std::string key = std::string(reinterpret_cast<const char*>(v), (size_t)n * sizeof(float4)) + (char)R;
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it == cache.end()) {
        std::vector<uint32_t> t;
        build_lut_uncached(v, n, R, t);
        it = cache.emplace(key, std::move(t)).first;
    }
    out.insert(out.end(), it->second.begin(), it->second.end());
}

// marks in `take` the vertices of `cand` (all n vertices if cand is NULL) that come within `slack` of the maximum for some
// sample direction of cell (face, iu, iw) on a SUB x SUB grid
static void lut_cell_pass(const float4* v, int n, const unsigned char* cand, int n_cand, int R, int face, int iu, int iw,
                          int SUB, double slack, std::vector<char>& take) {
    const int ax = face / 2, a = (ax + 1) % 3, b = (ax + 2) % 3;
    const double sgn = (face % 2 == 0) ? 1.0 : -1.0;
    const int m = cand ? n_cand : n;
    std::vector<double> dots(m);
    for (int su = 0; su < SUB; ++su)
        for (int sw = 0; sw < SUB; ++sw) {
            double d[3];
            d[ax] = sgn;
            d[a] = -1.0 + 2.0 * (iu + (double)su / (SUB - 1)) / R;
            d[b] = -1.0 + 2.0 * (iw + (double)sw / (SUB - 1)) / R;
            const double inv = 1.0 / sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
            const double dx = d[0] * inv, dy = d[1] * inv, dz = d[2] * inv;
            double mx = -1e300;
            for (int k = 0; k < m; ++k) {
                const float4& p = v[cand ? cand[k] : k];
                dots[k] = p.x * dx + p.y * dy + p.z * dz;
                if (dots[k] > mx) mx = dots[k];
            }
            for (int k = 0; k < m; ++k)
                if (mx - dots[k] <= slack) take[cand ? cand[k] : k] = 1;
        }
}

static void build_lut_uncached(const float4* v, int n, int R, std::vector<uint32_t>& out) {
    const int SUB = R >= 8 ? 17 : 33, cells = 6 * R * R;   // the same sample density on the sphere for coarse cells
    static const bool fine = !(getenv("SMENV_LUT_FINE") && atoi(getenv("SMENV_LUT_FINE")) == 0);
    static const int fine_div = getenv("SMENV_LUT_FINE_DIV") ? atoi(getenv("SMENV_LUT_FINE_DIV")) : 1024;   // samples per face edge
    const int SUB_FINE = 1 + fine_div / R;
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int i = 0; i < n; ++i) {
        const float p[3] = {v[i].x, v[i].y, v[i].z};
        for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], p[k]); hi[k] = fmaxf(hi[k], p[k]); }
    }
    const double diam = sqrt((double)(hi[0] - lo[0]) * (hi[0] - lo[0]) + (double)(hi[1] - lo[1]) * (hi[1] - lo[1]) +
                             (double)(hi[2] - lo[2]) * (hi[2] - lo[2]));
    // spacing on the cube face; the chord on the sphere is shorter
    auto slack_of = [&](int sub) { return diam * (2.0 / R / (sub - 1)) * 0.7072 * 1.05 + 1e-7; };
    std::vector<std::vector<unsigned char>> lists(cells);
    auto do_cells = [&](int c0, int c1) {
        std::vector<char> take(n), take2(n);
        std::vector<unsigned char> sup;
        for (int c = c0; c < c1; ++c) {
            const int face = c / (R * R), iu = (c / R) % R, iw = c % R;
            std::fill(take.begin(), take.end(), 0);
            lut_cell_pass(v, n, nullptr, 0, R, face, iu, iw, SUB, slack_of(SUB), take);
            if (fine) {
                sup.clear();
                for (int i = 0; i < n; ++i)
                    if (take[i]) sup.push_back((unsigned char)i);
                std::fill(take2.begin(), take2.end(), 0);
                lut_cell_pass(v, n, sup.data(), (int)sup.size(), R, face, iu, iw, SUB_FINE, slack_of(SUB_FINE), take2);
                take.swap(take2);
            }
            std::vector<unsigned char>& L = lists[c];
            for (int i = 0; i < n; ++i)
                if (take[i]) L.push_back((unsigned char)i);
        }
    };
    {   // cells are independent: a few host threads (the tables of a scene are built once per process)
        unsigned nt = std::thread::hardware_concurrency();
        nt = nt < 1 ? 1 : nt > 16 ? 16 : nt;
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; ++t)
            th.emplace_back(do_cells, (int)((long long)cells * t / nt), (int)((long long)cells * (t + 1) / nt));
        for (auto& x : th) x.join();
    }
    const size_t base = out.size();
    out.resize(base + cells);
    for (int c = 0; c < cells; ++c) {
        std::vector<unsigned char>& L = lists[c];
        size_t cnt = L.size();
        if (cnt > 255) { L.resize(255); cnt = 255; }  // cannot happen for <= 255-vertex hulls
        while (L.size() % 4) L.push_back(L.back());
        const uint32_t off = (uint32_t)(out.size() - base);
        out[base + c] = (off << 8) | (uint32_t)cnt;
        for (size_t k = 0; k < L.size(); k += 4)
            out.push_back((uint32_t)L[k] | ((uint32_t)L[k + 1] << 8) | ((uint32_t)L[k + 2] << 16) | ((uint32_t)L[k + 3] << 24));
    }
}

// support-width table of one hull about its bounding-sphere centre (layout: smenv_device.cuh), same cube-map cells and
// sampling as the direction tables; the slack covers directions between the samples
static void build_hwidth(const float4* v, int n, const float* c, float radius, std::vector<float>& out) {
    const int R = SM_LUT_RES, SUB = 17;
    const double spacing = 2.0 / R / (SUB - 1);
    const double slack = (double)radius * spacing * 0.7072 * 1.05 + 1e-6;
    for (int face = 0; face < 6; ++face) {
        const int ax = face / 2, a = (ax + 1) % 3, b = (ax + 2) % 3;
        const double sgn = (face % 2 == 0) ? 1.0 : -1.0;
        for (int iu = 0; iu < R; ++iu)
            for (int iw = 0; iw < R; ++iw) {
                double hmax = 0.0;
                for (int su = 0; su < SUB; ++su)
                    for (int sw = 0; sw < SUB; ++sw) {
                        double d[3];
                        d[ax] = sgn;
                        d[a] = -1.0 + 2.0 * (iu + (double)su / (SUB - 1)) / R;
                        d[b] = -1.0 + 2.0 * (iw + (double)sw / (SUB - 1)) / R;
                        const double nrm = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
                        double mx = -1e300;
                        for (int i = 0; i < n; ++i) {
                            const double s = ((v[i].x - c[0]) * d[0] + (v[i].y - c[1]) * d[1] + (v[i].z - c[2]) * d[2]) / nrm;
                            if (s > mx) mx = s;
                        }
                        if (mx > hmax) hmax = mx;
                    }
                out.push_back((float)((hmax + slack) * (1.0 + 1e-6)));
            }
    }
}

struct SmEnv {
    int n = 0, device = 0;
    uint64_t seed = 0;
    DevScene host_scene;  // device pointers inside
    float4* d_verts = nullptr;
    uint32_t* d_lut = nullptr;
    float* d_hwidth = nullptr;
    SceneImage* d_scene_img = nullptr;
    float4* d_ppos[SM_MAX_OBSTACLES] = {nullptr, nullptr};
    float4* d_pquat[SM_MAX_OBSTACLES] = {nullptr, nullptr};
    double* d_plocal = nullptr;
    double* d_start_pool = nullptr;
    double* d_ball_pool = nullptr;
    double* d_target_pool = nullptr;   // [target_pool_n][4] target points of the reaching task
    int target_pool_n = 0;
    int start_pool_n = 0, ball_pool_n = 0;
    bool pools_filled = false;
    unsigned long long* d_counters = nullptr;
    float* d_scratch = nullptr;  // per-env hand-over between the phase kernels of a step
    int* d_worklist = nullptr;   // [0] = GJK item counter (cleared by joint_kernel), [1] = overflowed items
    GjkItem* d_items = nullptr;  // work items of one step (smenv_plan.cuh -> smenv_gjk.cuh)
    int item_capacity = 0;
    unsigned* d_res = nullptr;   // [n][SM_RES_STRIDE] distance keys / first contact sub-step
    int* h_flag = nullptr;       // mapped pinned host word set by finish_kernel when the item buffer overflowed
    int* d_flag = nullptr;       // its device alias
    uint32_t* h_step = nullptr;  // pinned: the step counter of the host-buffer step; a captured copy node reads it at every
    uint32_t* d_step = nullptr;  // replay of the graph (a kernel argument would be frozen at capture time)
    size_t smem_bytes_gjk = 0;
    int grid_gjk = 0;
    int gjk_threads = GJK_THREADS;   // 512 when only one CTA of the GJK kernel fits on an SM
    MlpNet nets[SM_NET_COUNT];   // risk network, backup policy, human policy (smenv_mlp_load)
    bool net_loaded[SM_NET_COUNT] = {};
    std::vector<void*> net_allocs;
    float* d_risk = nullptr;     // [n] risk of the proposed action
    float* d_backup = nullptr;   // [n][MLP_MAX_OUT] action mean of the backup policy
    float* d_exec = nullptr;     // [n][n_joints] actions executed when the gate is on (smenv_set_risk_gate)
    uint8_t* d_risky = nullptr;  // [n] 1 where the gate replaced the action
    float gate_threshold = -1.0f;  // < 0: gate off
    int* d_gate_list = nullptr;    // [0..15] counters (two per env range), then [n] near-threshold rows, [n] risky rows
    int gate_exact = 1;            // re-rate near-threshold rows and compute the backup actions in float32 (smenv_set_gate_exact)
    float gate_band = 0.01f;       // |risk - threshold| below which the tensor-core risk is re-rated
    // Human scene (smenv_human.cuh)
    bool human = false;
    int human_external = 0;        // the human's actions come from buf->hactions (parity protocol)
    short* d_hpairs = nullptr;     // pair list of the braking-trajectory check
    float* d_hthresh = nullptr;    // contact thresholds per (human link, robot contact slot)
    double* d_hrange = nullptr;    // [n][8][4]
    double* d_hbacc = nullptr;     // [n][SM_HBRAKE_STEPS][8]
    float* d_hposes = nullptr;     // [n][SM_HBRAKE_POSES][8]
    int* d_hbinfo = nullptr;       // [n][4]
    int* d_hunits = nullptr;       // [0] = count, [1..] = (env << 7 | pose) units of the braking-trajectory pose checks
    float* d_hscratch = nullptr;   // [n][SM_SCRATCH_FLOATS]
    float* d_hpolicy = nullptr;    // [n][16]
    double* d_hstart_pool = nullptr;   // [start_pool_n][SM_HPOOL_STRIDE]
    double* d_hpool_brake = nullptr;   // [start_pool_n][SM_HBRAKE_STEPS][8] initial braking trajectory of every start state
    int* d_hpool_bcount = nullptr;     // [start_pool_n]
    double* d_htarget_pool = nullptr;  // [2][htarget_pool_n][4]
    int htarget_pool_n = 0;
    size_t smem_bytes_hplan = 0;
    int grid_hplan = 0;              // resident CTAs of human_brake_plan_kernel on the device
    bool time_kernels = false;   // measurement mode (smenv_kernel_timing)
    cudaEvent_t ev[SM_K_COUNT + 1] = {};
    double kernel_ms[SM_K_COUNT] = {};
    int timed_steps = 0;
    cudaStream_t chunk_streams[8] = {};  // smenv_step_host: one stream per env range in flight
    cudaEvent_t chunk_done[8] = {};
    cudaEvent_t chunk_fork = nullptr;
    cudaStream_t side_streams[8] = {};   // contact planning next to the distance planning, per env range
    cudaEvent_t side_fork[8] = {}, side_join[8] = {};
    cudaEvent_t joint_fork[8] = {}, joint_join[8] = {};   // Human scene: the robot's joint kernels next to the nested env
    cudaStream_t host_stream = nullptr;  // origin stream of the host-step graph
    cudaEvent_t host_order = nullptr;
    cudaGraphExec_t host_graph = nullptr;
    unsigned char host_graph_key[sizeof(SmBuffers) + 4 * sizeof(void*) + 8 * sizeof(int) + 32] = {};
    int host_graph_kernels = 0;
    int step_ranges = 1;         // env ranges the device step runs side by side (smenv_set_step_ranges)
    int list_layout = 1;         // number of env ranges of the last step (where the counts of the work lists sit)
    int* d_heavy = nullptr;      // [0] = count, [1..8n] = (env, joint) instances deferred to joint_heavy_kernel
    int* d_cwork = nullptr;      // [0] = count, [1..8n] = spans (env * 8 + span) the coarse contact phase could not clear
    int* d_tasks = nullptr;      // [0] = count, [1..16n] = position bounds to solve (joint_solve_kernel)
    double* d_hpar = nullptr;    // [8n][SM_HPAR] hand-over records of the deferred joints
    int* d_hheavy = nullptr;     // Human scene: the same three lists for the human's joints (its joint kernels run next to
    int* d_htasks = nullptr;     // the robot's)
    double* d_hhpar = nullptr;
    bool count = false;
    size_t smem_bytes = 0;        // kernels that stage the hull vertices
    size_t smem_bytes_broad = 0;  // contact_broad_kernel: scene tables only
    int grid = 0, grid_broad = 0, sms = 0;
    uint32_t step_counter = 0;
    unsigned long long launches = 0;
};

// The scene of the env being driven sits in constant memory (c_sc), one copy per device.  Every entry point that
// launches kernels holds the device's lock for the duration of the call (all launches are asynchronous, so calls are
// short) and, when another env's scene is loaded, waits for that env's outstanding work before replacing it: several
// envs, also on different host threads or streams, can share a device and only pay a device synchronisation when the
// driven env changes.
#define SM_MAX_DEVICES 64
static std::recursive_mutex g_dev_mu[SM_MAX_DEVICES];
static SmEnv* g_active[SM_MAX_DEVICES] = {};   // whose scene currently sits in the device's constant memory
static size_t g_smem_geom[SM_MAX_DEVICES] = {}, g_smem_gjk[SM_MAX_DEVICES] = {};  // opt-in limits set so far (never lowered)

struct DevLock {
    std::unique_lock<std::recursive_mutex> l;
    explicit DevLock(const SmEnv* env);
};

static int activate(SmEnv* env, cudaStream_t stream) {
    CU(cudaSetDevice(env->device));
    SmEnv*& active = g_active[env->device % SM_MAX_DEVICES];
    if (active != env) {
        if (active) CU(cudaDeviceSynchronize());   // kernels of the previous env may still read its scene
        CU(cudaMemcpyToSymbolAsync(c_sc, &env->host_scene, sizeof(DevScene), 0, cudaMemcpyHostToDevice, stream));
        active = env;
    }
    return SM_OK;
}

DevLock::DevLock(const SmEnv* env) : l(g_dev_mu[(env ? env->device : 0) % SM_MAX_DEVICES]) {}

extern "C" const char* smenv_last_error(void) { return g_error.c_str(); }
extern "C" int smenv_abi_version(void) { return 1; }
extern "C" int smenv_sizeof_scene(void) { return (int)sizeof(SmScene); }
extern "C" int smenv_sizeof_shape(void) { return (int)sizeof(SmShape); }

template <typename T>
static int upload(T** dst, const std::vector<T>& src) {
    CU(cudaMalloc((void**)dst, src.size() * sizeof(T)));
    CU(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return SM_OK;
}

// link-group pairs of the human's braking-trajectory check and the capsules of the arm frames (human_brake_plan_kernel):
// the pair list sorted by (frame of A, frame of B, A, B), per link-group pair the bounding volumes of both sides.  Host only,
// shared by smenv_create and smenv_debug_human_bounds; hpairs receives the sorted pair list.
static int human_brake_bounds(const SmScene* sc, DevHuman& u, std::vector<short>& hpairs) {
    const SmHuman& h = sc->human;
    std::vector<std::array<int, 4>> ps;
    for (int i = 0; i < h.n_brake_pairs; ++i) {
        const int a = h.brake_pairs[i][0], b = h.brake_pairs[i][1];
        ps.push_back({sc->shapes[a].frame, sc->shapes[b].frame, a, b});
    }
    std::sort(ps.begin(), ps.end());
    auto bound = [&](const std::vector<int>& ids, float* c, float* r, float* bmin, float* bmax) {
        float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        float mrg = 0.f;
        for (int id : ids) {
            const SmShape& sh = sc->shapes[id];
            mrg = fmaxf(mrg, (float)sh.margin);
            for (int i = sh.vert_off; i < sh.vert_off + sh.vert_cnt; ++i)
                for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], (float)sc->verts[3 * i + k]); hi[k] = fmaxf(hi[k], (float)sc->verts[3 * i + k]); }
        }
        float rad = 0.f;
        for (int k = 0; k < 3; ++k) { c[k] = 0.5f * (lo[k] + hi[k]); bmin[k] = lo[k] - mrg - 1e-6f; bmax[k] = hi[k] + mrg + 1e-6f; }
        for (int id : ids) {
            const SmShape& sh = sc->shapes[id];
            for (int i = sh.vert_off; i < sh.vert_off + sh.vert_cnt; ++i) {
                const float dx = (float)sc->verts[3 * i] - c[0], dy = (float)sc->verts[3 * i + 1] - c[1], dz = (float)sc->verts[3 * i + 2] - c[2];
                rad = fmaxf(rad, sqrtf(dx * dx + dy * dy + dz * dz));
            }
        }
        *r = rad * (1.0f + 1e-6f) + mrg + 1e-6f;
    };
    // capsule around a set of shapes: segment along the principal axis of the vertices, radius = largest distance of a
    // vertex to the segment (+ margin)
    auto capsule = [&](const std::vector<int>& ids, float* seg, float* r) {
        std::vector<std::array<double, 3>> pts;
        double mrg = 0.0;
        for (int id : ids) {
            const SmShape& sh = sc->shapes[id];
            mrg = std::max(mrg, sh.margin);
            for (int i = sh.vert_off; i < sh.vert_off + sh.vert_cnt; ++i)
                pts.push_back({sc->verts[3 * i], sc->verts[3 * i + 1], sc->verts[3 * i + 2]});
        }
        double m[3] = {0, 0, 0}, C[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
        for (auto& q : pts) for (int k = 0; k < 3; ++k) m[k] += q[k] / (double)pts.size();
        for (auto& q : pts)
            for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) C[a][b] += (q[a] - m[a]) * (q[b] - m[b]);
        double u[3] = {1.0, 0.7, 0.3};
        for (int it = 0; it < 64; ++it) {   // power iteration: dominant eigenvector of the covariance
            double w[3];
            for (int a = 0; a < 3; ++a) w[a] = C[a][0] * u[0] + C[a][1] * u[1] + C[a][2] * u[2];
            const double nrm = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
            if (nrm < 1e-30) break;
            for (int a = 0; a < 3; ++a) u[a] = w[a] / nrm;
        }
        double tmin = 1e300, tmax = -1e300;
        for (auto& q : pts) {
            const double t = (q[0] - m[0]) * u[0] + (q[1] - m[1]) * u[1] + (q[2] - m[2]) * u[2];
            tmin = std::min(tmin, t); tmax = std::max(tmax, t);
        }
        // pull the end points in by the cross-section radius (a capsule's caps cover the ends)
        double rad_line = 0.0;
        for (auto& q : pts) {
            const double t = (q[0] - m[0]) * u[0] + (q[1] - m[1]) * u[1] + (q[2] - m[2]) * u[2];
            double d2 = 0.0;
            for (int a = 0; a < 3; ++a) { const double e = q[a] - m[a] - t * u[a]; d2 += e * e; }
            rad_line = std::max(rad_line, sqrt(d2));
        }
        double t0 = tmin + rad_line, t1 = tmax - rad_line;
        if (t0 > t1) t0 = t1 = 0.5 * (tmin + tmax);
        double rad = 0.0;
        for (auto& q : pts) {
            double t = (q[0] - m[0]) * u[0] + (q[1] - m[1]) * u[1] + (q[2] - m[2]) * u[2];
            t = std::min(std::max(t, t0), t1);
            double d2 = 0.0;
            for (int a = 0; a < 3; ++a) { const double e = q[a] - m[a] - t * u[a]; d2 += e * e; }
            rad = std::max(rad, sqrt(d2));
        }
        for (int a = 0; a < 3; ++a) { seg[a] = (float)(m[a] + t0 * u[a]); seg[3 + a] = (float)(m[a] + t1 * u[a]); }
        *r = (float)(rad * (1.0 + 1e-5) + mrg + 1e-5);
    };
    int ngp = 0;
    for (size_t i = 0; i < ps.size();) {
        size_t e = i;
        while (e < ps.size() && ps[e][0] == ps[i][0] && ps[e][1] == ps[i][1]) ++e;
        if (ngp >= 8) return fail(SM_ERR_SCENE, "the human's braking-trajectory check has more than 8 link-group pairs");
        std::vector<int> ia, ib;
        for (size_t q = i; q < e; ++q) { ia.push_back(ps[q][2]); ib.push_back(ps[q][3]); }
        u.gp_fa[ngp] = ps[i][0] - 100; u.gp_fb[ngp] = ps[i][1] >= 100 ? ps[i][1] - 100 : -1;   // -1: world frame
        u.gp_off[ngp] = (int)i; u.gp_cnt[ngp] = (int)(e - i);
        {   // the device code walks a group pair as two nested shape ranges
            std::vector<int> ua(ia), ub(ib);
            std::sort(ua.begin(), ua.end()); ua.erase(std::unique(ua.begin(), ua.end()), ua.end());
            std::sort(ub.begin(), ub.end()); ub.erase(std::unique(ub.begin(), ub.end()), ub.end());
            const bool dense = ua.size() * ub.size() == e - i && ua.back() - ua.front() + 1 == (int)ua.size() &&
                               ub.back() - ub.front() + 1 == (int)ub.size();
            if (!dense)
                return fail(SM_ERR_SCENE, "the pairs of the human's braking check between two frames must be the cross "
                                          "product of two contiguous shape ranges");
            if (ub.size() > 32) return fail(SM_ERR_SCENE, "braking check: more than 32 shapes on side B of a link-group pair");
            u.gp_a0[ngp] = ua.front(); u.gp_na[ngp] = (int)ua.size();
            u.gp_b0[ngp] = ub.front(); u.gp_nb[ngp] = (int)ub.size();
        }
        float dmin[3], dmax[3];
        bound(ia, u.gp_ca[ngp], &u.gp_ra[ngp], dmin, dmax);
        bound(ib, u.gp_cb[ngp], &u.gp_rb[ngp], u.gp_bmin[ngp], u.gp_bmax[ngp]);
        capsule(ia, u.gp_sa[ngp], &u.gp_sra[ngp]);
        capsule(ib, u.gp_sb[ngp], &u.gp_srb[ngp]);
        ++ngp;
        i = e;
    }
    u.n_gp = ngp;
    // arm frames 3, 4, 7, 8: shape range and capsule (side A of every group pair is one of them)
    const int arm_frames[4] = {103, 104, 107, 108};
    for (int fi = 0; fi < 4; ++fi) {
        std::vector<int> ids;
        for (int q = 0; q < h.n_arm_shapes; ++q)
            if (sc->shapes[h.shape_off + q].frame == arm_frames[fi]) ids.push_back(h.shape_off + q);
        u.hf_s0[fi] = ids.empty() ? h.shape_off : ids.front(); u.hf_sn[fi] = (int)ids.size();
        if (!ids.empty() && ids.back() - ids.front() + 1 != (int)ids.size())
            return fail(SM_ERR_SCENE, "the shapes of a human arm frame must be contiguous");
        for (int k = 0; k < 6; ++k) u.hf_seg[fi][k] = 0.f;
        u.hf_rad[fi] = 0.f;
        if (!ids.empty()) capsule(ids, u.hf_seg[fi], &u.hf_rad[fi]);
    }
    for (int g = 0; g < ngp; ++g) {
        const int fa = u.gp_fa[g], fb = u.gp_fb[g];
        const bool arm_a = fa == 3 || fa == 4 || fa == 7 || fa == 8, arm_b = fb == 3 || fb == 4 || fb == 7 || fb == 8;
        if (!arm_a || !(arm_b || fb == 0 || fb == -1))
            return fail(SM_ERR_SCENE, "braking check: side A must be an arm frame, side B an arm frame, the trunk or the world");
        if (h.n_arm_shapes > 32) return fail(SM_ERR_SCENE, "braking check: more than 32 arm shapes");
        if (fb == 0 && (u.gp_b0[g] < h.shape_off + h.n_arm_shapes || h.n_shapes - h.n_arm_shapes > 32))
            return fail(SM_ERR_SCENE, "braking check: trunk shapes must follow the arm shapes (at most 32)");
    }
    for (auto& q : ps) { hpairs.push_back((short)q[2]); hpairs.push_back((short)q[3]); }
    return SM_OK;
}

// Constants of the distance planning (distance_plan_kernel), from the float32 vertices the kernels use: per shape the
// bounding sphere, the box of the core vertices, the centroid and the support-width table (appended to hwidth); the pair
// table with the margins and radii its bounds subtract; the self-collision query.  Fills d.shapes (all but .lut),
// d.pair_tab, d.pair_rm, d.n_pairs_fixed, d.n_pairs and d.self_query.  Host only, shared by smenv_create and
// smenv_debug_plan_bounds.
static int plan_bounds(const SmScene* sc, const std::vector<float4>& verts, DevScene& d, std::vector<float>& hwidth) {
    for (int s = 0; s < sc->n_shapes; ++s) {
        const SmShape& h = sc->shapes[s];
        DevShape& g = d.shapes[s];
        g.frame = h.frame; g.off = h.vert_off; g.cnt = h.vert_cnt; g.link = h.link;
        g.margin = (float)h.margin; g.cx = (float)h.center[0]; g.cy = (float)h.center[1]; g.cz = (float)h.center[2];
        // bounding sphere recomputed on the float32 vertices so that it certainly contains them
        float r = 0.f;
        for (int k = 0; k < 3; ++k) { g.bmin[k] = FLT_MAX; g.bmax[k] = -FLT_MAX; }
        for (int i = h.vert_off; i < h.vert_off + h.vert_cnt; ++i) {
            float dx = verts[i].x - g.cx, dy = verts[i].y - g.cy, dz = verts[i].z - g.cz;
            r = fmaxf(r, sqrtf(dx * dx + dy * dy + dz * dz));
            g.bmin[0] = fminf(g.bmin[0], verts[i].x); g.bmax[0] = fmaxf(g.bmax[0], verts[i].x);
            g.bmin[1] = fminf(g.bmin[1], verts[i].y); g.bmax[1] = fmaxf(g.bmax[1], verts[i].y);
            g.bmin[2] = fminf(g.bmin[2], verts[i].z); g.bmax[2] = fmaxf(g.bmax[2], verts[i].z);
        }
        g.radius = r * (1.0f + 1e-6f) + 1e-7f;
        double gs[3] = {0, 0, 0};
        for (int i = h.vert_off; i < h.vert_off + h.vert_cnt; ++i) { gs[0] += verts[i].x; gs[1] += verts[i].y; gs[2] += verts[i].z; }
        g.gx = (float)(gs[0] / h.vert_cnt); g.gy = (float)(gs[1] / h.vert_cnt); g.gz = (float)(gs[2] / h.vert_cnt);
        g.hw = (int)hwidth.size();
        {
            const float cc[3] = {g.cx, g.cy, g.cz};
            build_hwidth(verts.data() + h.vert_off, h.vert_cnt, cc, g.radius, hwidth);
        }
        g.lut = -1;
    }
    int np = 0;
    auto push = [&](int a, int b, int cls) {
        if (np < SM_MAX_PLAN_PAIRS) {
            const DevShape& SA = d.shapes[a];
            const DevShape& SB = d.shapes[b];
            const bool box = SB.frame == 0;
            d.pair_tab[np] = (uint32_t)a | ((uint32_t)b << 12) | ((uint32_t)cls << 24) | (box ? 0x80000000u : 0u);
            const float m = SA.margin + SB.margin;
            d.pair_rm[np] = make_float2(m * (1.0f - 1e-6f), (SA.radius + (box ? 0.f : SB.radius) + m) * (1.0f + 1e-6f));
        }
        ++np;
    };
    for (int i = 0; i < sc->n_static_pairs; ++i) push(sc->static_pairs[i][0], sc->static_pairs[i][1], 0);
    for (int i = 0; i < sc->n_self_pairs; ++i) push(sc->self_pairs[i][0], sc->self_pairs[i][1], 1);
    d.n_pairs_fixed = np;
    for (int o = 0; o < sc->n_obstacles; ++o)
        for (int r = 0; r < sc->n_mov_reward; ++r)
            for (int k = 0; k < sc->obst_shape_cnt[o]; ++k) push(sc->mov_reward[r], sc->obst_shape_off[o] + k, 2);
    d.n_pairs = np;
    if (np > SM_MAX_PLAN_PAIRS) return fail(SM_ERR_SCENE, "too many convex pairs per env for the distance planning (max 512)");
    d.self_query = std::min(sc->static_cap, std::max(sc->collision_dist, sc->w_self != 0.0 ? sc->d_self : 0.0));
    return SM_OK;
}

extern "C" int smenv_destroy(SmEnv* env);
// frees a half-built env on every early return of smenv_create
struct CreateGuard {
    SmEnv* env;
    ~CreateGuard() { if (env) smenv_destroy(env); }
};

extern "C" int smenv_create(const SmScene* sc, int num_envs, int device, uint64_t seed, SmEnv** out) {
    if (!sc || !out || num_envs <= 0) return fail(SM_ERR_ARG, "smenv_create: bad argument");
    if (sc->n_joints <= 0 || sc->n_joints > 7) return fail(SM_ERR_SCENE, "n_joints must be in 1..7");
    if (sc->substeps < 1 || sc->substeps > SM_MAX_SUB) return fail(SM_ERR_SCENE, "substeps must be in 1..32");
    if (sc->n_shapes > SM_MAX_SHAPES || sc->n_verts <= 0) return fail(SM_ERR_SCENE, "bad shape table");
    if (sc->obs_size > SM_MAX_OBS) return fail(SM_ERR_SCENE, "obs_size too large");
    for (int j = 0; j < sc->n_joints; ++j)
        if (sc->joint_parent[j] != j) return fail(SM_ERR_SCENE, "only serial kinematic chains are supported");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(SM_ERR_ARG, "smenv_create: no such CUDA device");
    CU(cudaSetDevice(device));
    if (device >= SM_MAX_DEVICES) return fail(SM_ERR_ARG, "smenv_create: device index too large");
    SmEnv* env = new SmEnv();
    CreateGuard guard{env};
    env->device = device;
    DevLock dev_lock_(env);
    env->n = num_envs;
    env->device = device;
    env->seed = seed;
    DevScene& d = env->host_scene;
    memset(&d, 0, sizeof(d));
    d.n_joints = sc->n_joints; d.substeps = sc->substeps; d.contact_stride = sc->contact_stride;
    d.limit_velocity = sc->limit_velocity; d.limit_position = sc->limit_position;
    for (int j = 0; j < SM_MAX_JOINTS; ++j) {
        d.joint_parent[j] = sc->joint_parent[j];
        for (int i = 0; i < 9; ++i) d.jR[j][i] = (float)sc->joint_R[j][i];
        {
            bool ident = true;
            for (int i = 0; i < 9; ++i) ident = ident && d.jR[j][i] == ((i % 4 == 0) ? 1.0f : 0.0f);
            if (ident) d.jr_identity |= 1 << j;
        }
        for (int i = 0; i < 3; ++i) { d.jt[j][i] = (float)sc->joint_t[j][i]; d.jaxis[j][i] = (float)sc->joint_axis[j][i]; }
        d.pos_lo[j] = sc->pos_lo[j]; d.pos_hi[j] = sc->pos_hi[j]; d.vel_max[j] = sc->vel_max[j];
        d.acc_max[j] = sc->acc_max[j]; d.jerk_max[j] = sc->jerk_max[j];
        d.lim.inv_jts[j] = sc->jerk_max[j] * sc->ts > 0.0 ? (1.0 / (sc->jerk_max[j] * sc->ts)) * (1.0 + 1e-12) : 0.0;
        d.lim.inv_2a[j] = sc->acc_max[j] > 0.0 ? (1.0 / (2.0 * sc->acc_max[j])) * (1.0 + 1e-12) : 0.0;
    }
    d.ts = sc->ts; d.action_mapping_factor = sc->action_mapping_factor; d.track_kp = sc->track_kp;
    d.track_vel = sc->track_vel;
    {  // sub-step times exactly as np.linspace(ts / S, ts, S) produces them (actions.py:420-421)
        const int S = sc->substeps;
        volatile double start = sc->ts / (double)S;
        volatile double step = S > 1 ? (sc->ts - start) / (double)(S - 1) : 0.0;
        for (int k = 1; k <= S; ++k) {
            volatile double prod = (double)(k - 1) * step;
            d.sub_t[k] = (S <= 1 || k == S) ? sc->ts : start + prod;
        }
    }
    d.n_shapes = sc->n_shapes; d.n_verts = sc->n_verts;
    std::vector<float4> verts(sc->n_verts);
    for (int i = 0; i < sc->n_verts; ++i)
        verts[i] = make_float4((float)sc->verts[3 * i], (float)sc->verts[3 * i + 1], (float)sc->verts[3 * i + 2], 0.f);
    std::vector<uint32_t> lut;
    std::vector<float> hwidth;
    if (const int rc = plan_bounds(sc, verts, d, hwidth)) return rc;
    // Support-direction tables.  The longest candidate list among the lanes of a GJK warp sets the trip count of its
    // support loop, so every hull that can have a table gets one as long as the kernel's shared-memory image (vertices +
    // tables + shapes) fits.  Candidates in order of quality, the first that fits the budget wins:
    //   hulls from 33 vertices with 8 x 8 cells per cube face, smaller hulls (from 8 vertices) with 4 x 4 -- then every lane
    //   takes the table branch instead of the warp running a table loop and a full-scan loop one after the other;
    //   the same without tables for the hulls below 33 vertices;
    //   4 x 4 cells for all hulls up to 64 vertices (Human scene: 40 human parts), with / without the small hulls;
    //   tables only from 65 / 129 / 256 vertices.
    // Budget: 113 KB if some candidate of the first four fits (two 256-thread CTAs per SM), else 220 KB (one 768-thread
    // CTA).  Measured (profiles/r02b_gjk_table_sweep.txt): finer cells for the big hulls (12 or 16 per edge) shorten the
    // lists further but cost the second CTA, or the room a planning CTA of the other env range finds next to the pair,
    // and lose: space_bm 661 us per step with 8 cells in 111 KB, 672 / 674 with 16 / 12 cells; Ball 388 (77 KB) against 402.
    // SMENV_LUT_BUDGET_KB, SMENV_LUT_BIG_RES, SMENV_LUT_TINY_MIN, SMENV_LUT_CONFIG override (experiments).
    auto build_tables = [&](int min_verts, int small_res, int tiny_min, int big_res) {
        lut.clear();
        for (int s = 0; s < sc->n_shapes; ++s) {
            const SmShape& h = sc->shapes[s];
            d.shapes[s].lut = -1;
            const bool tiny = h.vert_cnt < min_verts && h.vert_cnt >= tiny_min;
            if ((h.vert_cnt >= min_verts || tiny) && h.vert_cnt <= 255) {
                const int R = tiny ? SM_LUT_RES_COARSE : h.vert_cnt <= 64 ? small_res : big_res;
                d.shapes[s].lut = (int)lut.size() | (lut_code_of(R) << SM_LUT_RES_SHIFT);
                build_lut(verts.data() + h.vert_off, h.vert_cnt, R, lut);
            }
        }
        return gjk_smem_bytes(sc->n_verts, (int)lut.size() + 4, sc->n_shapes);
    };
    {
        const int forced_budget = getenv("SMENV_LUT_BUDGET_KB") ? atoi(getenv("SMENV_LUT_BUDGET_KB")) : 0;
        const int forced_cfg = getenv("SMENV_LUT_CONFIG") ? atoi(getenv("SMENV_LUT_CONFIG")) : -1;
        const int big = getenv("SMENV_LUT_BIG_RES") ? atoi(getenv("SMENV_LUT_BIG_RES")) : SM_LUT_RES;
        const int tiny_min = getenv("SMENV_LUT_TINY_MIN") ? atoi(getenv("SMENV_LUT_TINY_MIN")) : 8;
        const int none = 1 << 30, n_cand = 7;
        // min vertices, cells of hulls up to 64 vertices, smallest hull with a coarse table
        const int cand[n_cand][3] = {{33, 8, tiny_min}, {33, 8, none}, {33, 4, tiny_min}, {33, 4, none},
                                     {65, 8, none}, {129, 8, none}, {256, 8, none}};
        bool placed = false;
        for (int pass = 0; pass < 2 && !placed; ++pass) {
            const size_t budget = (size_t)(forced_budget ? forced_budget : pass == 0 ? 113 : 220) * 1024;
            for (int ci = 0; ci < (pass == 0 ? 4 : n_cand) && !placed; ++ci) {
                if (forced_cfg >= 0 && ci != forced_cfg) continue;
                placed = build_tables(cand[ci][0], cand[ci][1], cand[ci][2], big) <= budget;
            }
        }
        if (!placed) build_tables(cand[n_cand - 1][0], cand[n_cand - 1][1], cand[n_cand - 1][2], SM_LUT_RES);
    }
    d.n_static_pairs = sc->n_static_pairs; d.n_self_pairs = sc->n_self_pairs;
    d.n_mov_reward = sc->n_mov_reward; d.n_mov_contact = sc->n_mov_contact;
    for (int i = 0; i < SM_MAX_PAIRS; ++i)
        for (int k = 0; k < 2; ++k) {
            d.static_pairs[i][k] = (short)sc->static_pairs[i][k];
            d.self_pairs[i][k] = (short)sc->self_pairs[i][k];
        }
    for (int i = 0; i < SM_MAX_MOV_ROBOT; ++i) { d.mov_reward[i] = (short)sc->mov_reward[i]; d.mov_contact[i] = (short)sc->mov_contact[i]; }
    {  // contact slots must be sorted by frame for the per-lane broad phase
        int f = 0;
        d.contact_frame_start[0] = 0;
        for (int slot = 0; slot < sc->n_mov_contact; ++slot) {
            int fr = sc->shapes[sc->mov_contact[slot]].frame;
            if (fr < f || fr > sc->n_joints) { return fail(SM_ERR_SCENE, "mov_contact must be sorted by frame"); }
            while (f < fr) d.contact_frame_start[++f] = slot;
        }
        while (f <= sc->n_joints) d.contact_frame_start[++f] = sc->n_mov_contact;
    }
    d.n_obstacles = sc->n_obstacles;
    for (int o = 0; o < SM_MAX_OBSTACLES; ++o) {
        d.obst_kind[o] = sc->obst_kind[o]; d.obst_shape_off[o] = sc->obst_shape_off[o];
        d.obst_shape_cnt[o] = sc->obst_shape_cnt[o];
        for (int i = 0; i < 3; ++i) d.obst_center[o][i] = (float)sc->obst_center[o][i];
        d.obst_radius[o] = (float)sc->obst_radius[o] * (1.0f + 1e-6f) + 1e-6f;
        float mx = 0.f;
        for (int i = 0; i < SM_MAX_MOV_ROBOT; ++i) { d.contact_thresh[o][i] = (float)sc->contact_thresh[o][i]; mx = fmaxf(mx, d.contact_thresh[o][i]); }
        d.contact_thresh_max[o] = mx;
        for (int k = 0; k < 3; ++k) { d.obst_bmin[o][k] = FLT_MAX; d.obst_bmax[o][k] = -FLT_MAX; }
        for (int sI = d.obst_shape_off[o]; sI < d.obst_shape_off[o] + d.obst_shape_cnt[o] && o < sc->n_obstacles; ++sI)
            for (int k = 0; k < 3; ++k) {
                d.obst_bmin[o][k] = fminf(d.obst_bmin[o][k], d.shapes[sI].bmin[k] - d.shapes[sI].margin - 1e-6f);
                d.obst_bmax[o][k] = fmaxf(d.obst_bmax[o][k], d.shapes[sI].bmax[k] + d.shapes[sI].margin + 1e-6f);
            }
        d.obst_center_norm[o] = sqrtf(d.obst_center[o][0] * d.obst_center[o][0] + d.obst_center[o][1] * d.obst_center[o][1] +
                                      d.obst_center[o][2] * d.obst_center[o][2]) * (1.0f + 1e-6f);
    }
    d.use_target_points = sc->use_target_points; d.tp_normalize = sc->tp_normalize;
    d.obs_add_tp_pos = sc->obs_add_tp_pos; d.obs_add_tp_rel = sc->obs_add_tp_rel; d.start_at_rest = sc->start_at_rest;
    d.tp_radius = sc->tp_radius; d.tp_bonus = sc->tp_bonus; d.tp_reward_factor = sc->tp_reward_factor;
    d.tp_min_static = sc->tp_min_static; d.tp_min_self = sc->tp_min_self;
    for (int i = 0; i < 3; ++i) {
        d.tp_box_min[i] = sc->tp_box_min[i]; d.tp_box_max[i] = sc->tp_box_max[i];
        d.tp_rel_min[i] = sc->tp_rel_min[i]; d.tp_rel_max[i] = sc->tp_rel_max[i];
        d.tp_local[i] = (float)(sc->target_t[i] + sc->target_R[3 * i] * sc->target_offset[0] +
                                sc->target_R[3 * i + 1] * sc->target_offset[1] + sc->target_R[3 * i + 2] * sc->target_offset[2]);
    }
    {   // a change of joint j by dq moves the target link point by at most dq * tp_rho[j]
        const float ln = sqrtf(d.tp_local[0] * d.tp_local[0] + d.tp_local[1] * d.tp_local[1] + d.tp_local[2] * d.tp_local[2]);
        for (int j = 0; j < SM_MAX_JOINTS; ++j) {
            float rho = 0.f;
            if (j < sc->n_joints) {
                rho = ln;
                for (int i = j + 1; i < sc->n_joints; ++i)
                    rho += sqrtf(d.jt[i][0] * d.jt[i][0] + d.jt[i][1] * d.jt[i][1] + d.jt[i][2] * d.jt[i][2]);
                rho *= 1.0f + 1e-5f;
            }
            d.tp_rho[j] = rho;
        }
    }
    // coarse contact phase: a change of joint j by dq moves the sphere centre of a contact slot in frame f by at most
    // dq * (sum of the fixed joint offsets between frame j+1 and f, plus the centre's own offset)
    for (int slot = 0; slot < sc->n_mov_contact; ++slot) {
        const SmShape& h = sc->shapes[sc->mov_contact[slot]];
        const float cn = sqrtf((float)(h.center[0] * h.center[0] + h.center[1] * h.center[1] + h.center[2] * h.center[2]));
        for (int j = 0; j < SM_MAX_JOINTS; ++j) {
            float rho = 0.f;
            if (j < h.frame) {
                rho = cn;
                for (int i = j + 1; i < h.frame; ++i)
                    rho += sqrtf(d.jt[i][0] * d.jt[i][0] + d.jt[i][1] * d.jt[i][1] + d.jt[i][2] * d.jt[i][2]);
                rho *= 1.0f + 1e-5f;
            }
            d.contact_rho[slot][j] = rho;
        }
    }
    d.planet_steps = sc->planet_steps; d.planet_shift = sc->planet_shift; d.obs_planet_size = sc->obs_planet_size;
    d.planet_obs_half[0] = sc->planet_obs_half[0]; d.planet_obs_half[1] = sc->planet_obs_half[1];
    for (int i = 0; i < 3; ++i) {
        d.ball_obs_pos_min[i] = sc->ball_obs_pos_min[i]; d.ball_obs_pos_max[i] = sc->ball_obs_pos_max[i];
        d.ball_obs_vel_min[i] = sc->ball_obs_vel_min[i]; d.ball_obs_vel_max[i] = sc->ball_obs_vel_max[i];
        d.start_box_min[i] = sc->start_box_min[i]; d.start_box_max[i] = sc->start_box_max[i];
        d.target_offset[i] = (float)sc->target_offset[i]; d.target_t[i] = (float)sc->target_t[i];
        d.ball_sphere_center[i] = sc->ball_sphere_center[i];
        d.ball_target_box_min[i] = sc->ball_target_box_min[i]; d.ball_target_box_max[i] = sc->ball_target_box_max[i];
        d.ball_invalid_min[i] = sc->ball_invalid_min[i]; d.ball_invalid_max[i] = sc->ball_invalid_max[i];
        d.ball_final_min[i] = sc->ball_final_min[i]; d.ball_final_max[i] = sc->ball_final_max[i];
    }
    for (int i = 0; i < 9; ++i) d.target_R[i] = (float)sc->target_R[i];
    d.ball_active_xy = sc->ball_active_xy;
    d.static_cap = sc->static_cap; d.moving_query = sc->moving_query; d.collision_dist = sc->collision_dist;
    d.w_self = sc->w_self; d.w_static = sc->w_static; d.w_moving = sc->w_moving;
    d.d_self = sc->d_self; d.d_static = sc->d_static; d.d_moving = sc->d_moving;
    d.w_low_acc = sc->w_low_acc; d.thr_low_acc = sc->thr_low_acc; d.w_low_vel = sc->w_low_vel; d.thr_low_vel = sc->thr_low_vel;
    d.punish_action = sc->punish_action; d.terminate_self = sc->terminate_self;
    d.terminate_static = sc->terminate_static; d.terminate_moving = sc->terminate_moving;
    d.action_thresh = sc->action_thresh; d.action_max_punishment = sc->action_max_punishment;
    d.termination_bonus = sc->termination_bonus; d.early_termination_punishment = sc->early_termination_punishment;
    d.reward_scale = sc->reward_scale != 0.0 ? sc->reward_scale : 1.0;
    d.episode_steps = sc->episode_steps; d.obs_size = sc->obs_size;
    d.kinematic_sampling_probability = sc->kinematic_sampling_probability;
    d.stay_in_state_probability = sc->stay_in_state_probability;
    d.min_start_distance = sc->min_start_distance; d.min_start_self = sc->min_start_self;
    d.ball_target_min_static = sc->ball_target_min_static; d.ball_target_min_self = sc->ball_target_min_self;
    d.ball_sphere_radius = sc->ball_sphere_radius; d.ball_height_min = sc->ball_height_min;
    d.ball_height_max = sc->ball_height_max; d.ball_angle_min = sc->ball_angle_min; d.ball_angle_max = sc->ball_angle_max;
    d.ball_speed = sc->ball_speed; d.ball_radius = sc->ball_radius;
    d.ball_high_angle_probability = sc->ball_high_angle_probability; d.plane_z = sc->plane_z;
    d.ball_check_invalid = sc->ball_check_invalid; d.ball_random_initial = sc->ball_random_initial;
    d.has_table = sc->has_table;
    // ---------------- the human obstacle (SmHuman -> DevHuman)
    std::vector<short> hpairs;
    std::vector<float> hthresh;
    if (sc->human.enabled) {
        const SmHuman& h = sc->human;
        DevHuman& u = d.hu;
        if (h.n_joints != SM_HUMAN_JOINTS) return fail(SM_ERR_SCENE, "the human must have 8 joints");
        if (sc->n_obstacles != 1 || sc->obst_kind[0] != SM_OBST_HUMAN) return fail(SM_ERR_SCENE, "a human scene has the human as its only moving obstacle");
        if (h.brake_checks < 1 || h.brake_checks > 7) return fail(SM_ERR_SCENE, "human brake_checks must be in 1..7");
        if (h.brake_checks * 22 > SM_HBRAKE_POSES) return fail(SM_ERR_SCENE, "too many collision checks per step for the pose buffer");
        for (int j = 0; j < 8; ++j)
            if (h.joint_parent[j] != ((j & 3) == 0 ? 0 : j)) return fail(SM_ERR_SCENE, "the human is expected as two serial arms of four joints");
        env->human = true;
        u.enabled = 1; u.n_joints = h.n_joints; u.check_braking = h.check_braking; u.brake_checks = h.brake_checks;
        u.initial_braking_trajectory = h.initial_braking_trajectory;
        u.n_brake_pairs = h.n_brake_pairs; u.shape_off = h.shape_off; u.n_arm_shapes = h.n_arm_shapes; u.n_shapes = h.n_shapes;
        for (int i = 0; i < 9; ++i) u.baseR[i] = (float)h.base_R[i];
        for (int i = 0; i < 3; ++i) u.baset[i] = (float)h.base_t[i];
        for (int j = 0; j < 8; ++j) {
            u.joint_parent[j] = h.joint_parent[j];
            for (int i = 0; i < 9; ++i) u.jR[j][i] = (float)h.joint_R[j][i];
            for (int i = 0; i < 3; ++i) { u.jt[j][i] = (float)h.joint_t[j][i]; u.jaxis[j][i] = (float)h.joint_axis[j][i]; }
            u.lim.pos_lo[j] = h.pos_lo[j]; u.lim.pos_hi[j] = h.pos_hi[j]; u.lim.vel_max[j] = h.vel_max[j];
            u.lim.acc_max[j] = h.acc_max[j]; u.lim.jerk_max[j] = h.jerk_max[j];
            u.lim.inv_jts[j] = (1.0 / (h.jerk_max[j] * sc->ts)) * (1.0 + 1e-12);
            u.lim.inv_2a[j] = (1.0 / (2.0 * h.acc_max[j])) * (1.0 + 1e-12);
        }
        u.brake_safety = h.brake_safety; u.brake_timeout = h.brake_timeout; u.tp_radius = h.tp_radius;
        u.log_std_lo = h.log_std_lo; u.log_std_hi = h.log_std_hi;
        for (int i = 0; i < 3; ++i) {
            u.tp_box_min[i] = h.tp_box_min[i]; u.tp_box_max[i] = h.tp_box_max[i];
            u.tp_rel_min[i] = h.tp_rel_min[i]; u.tp_rel_max[i] = h.tp_rel_max[i];
            u.start_box_min[i] = h.start_box_min[i]; u.start_box_max[i] = h.start_box_max[i];
            for (int r = 0; r < 2; ++r) u.tp_local[r][i] = (float)h.tp_local[r][i];
        }
        for (int r = 0; r < 2; ++r)   // a change of joint 4 r + i by dq moves the target link point of arm r by at most dq * tp_rho[r][i]
            for (int i = 0; i < 4; ++i) {
                float rho = sqrtf(u.tp_local[r][0] * u.tp_local[r][0] + u.tp_local[r][1] * u.tp_local[r][1] +
                                  u.tp_local[r][2] * u.tp_local[r][2]);
                for (int m = i + 1; m < 4; ++m) {
                    const float* t = u.jt[4 * r + m];
                    rho += sqrtf(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
                }
                u.tp_rho[r][i] = rho * (1.0f + 1e-5f);
            }
        u.kinematic_sampling_probability = h.kinematic_sampling_probability;
        u.stay_in_state_probability = h.stay_in_state_probability;
        u.min_start_static = h.min_start_static; u.min_start_self = h.min_start_self;
        u.tp_min_static = h.tp_min_static; u.tp_min_self = h.tp_min_self;
        {   // np.linspace(ts / C, ts, C) of the braking-trajectory check (ctlp.py:3166-3168), operation by operation
            const int C = h.brake_checks;
            volatile double start = sc->ts / (double)C;
            volatile double step = C > 1 ? (sc->ts - start) / (double)(C - 1) : 0.0;
            for (int m = 1; m <= C; ++m) {
                volatile double prod = (double)(m - 1) * step;
                u.brake_t[m] = (C <= 1 || m == C) ? sc->ts : start + prod;
            }
        }
        for (int s = 0; s < h.n_shapes && s < 64; ++s) u.shape_link[s] = (unsigned char)h.shape_link[s];
        float tmax = 0.f;
        hthresh.resize((size_t)SM_MAX_HLINKS * SM_MAX_MOV_ROBOT, 0.f);
        for (int l = 0; l < SM_MAX_HLINKS; ++l)
            for (int r = 0; r < SM_MAX_MOV_ROBOT; ++r) {
                hthresh[(size_t)l * SM_MAX_MOV_ROBOT + r] = (float)h.contact_thresh[l][r];
                tmax = fmaxf(tmax, (float)h.contact_thresh[l][r]);
            }
        u.contact_thresh_max = tmax;
        if (const int rc_b = human_brake_bounds(sc, u, hpairs)) return rc_b;
        // link groups: runs of consecutive human shapes in the same frame, with a bounding sphere in frame coordinates
        int ng = 0;
        for (int s = 0; s < h.n_shapes;) {
            const int fr = sc->shapes[h.shape_off + s].frame;
            int e = s;
            while (e < h.n_shapes && sc->shapes[h.shape_off + e].frame == fr) ++e;
            if (ng >= SM_HGROUPS) return fail(SM_ERR_SCENE, "the human has more link groups than expected");
            float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
            for (int q = s; q < e; ++q) {
                const SmShape& sh = sc->shapes[h.shape_off + q];
                for (int i = sh.vert_off; i < sh.vert_off + sh.vert_cnt; ++i)
                    for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], (float)sc->verts[3 * i + k]); hi[k] = fmaxf(hi[k], (float)sc->verts[3 * i + k]); }
            }
            float cc[3], rad = 0.f, mrg = 0.f;
            for (int k = 0; k < 3; ++k) cc[k] = 0.5f * (lo[k] + hi[k]);
            for (int q = s; q < e; ++q) {
                const SmShape& sh = sc->shapes[h.shape_off + q];
                mrg = fmaxf(mrg, (float)sh.margin);
                for (int i = sh.vert_off; i < sh.vert_off + sh.vert_cnt; ++i) {
                    const float dx = (float)sc->verts[3 * i] - cc[0], dy = (float)sc->verts[3 * i + 1] - cc[1], dz = (float)sc->verts[3 * i + 2] - cc[2];
                    rad = fmaxf(rad, sqrtf(dx * dx + dy * dy + dz * dz));
                }
            }
            u.grp_frame[ng] = fr - 100; u.grp_off[ng] = s; u.grp_cnt[ng] = e - s;
            for (int k = 0; k < 3; ++k) u.grp_c[ng][k] = cc[k];
            u.grp_r[ng] = rad * (1.0f + 1e-6f) + mrg + 1e-6f;
            const float cn = sqrtf(cc[0] * cc[0] + cc[1] * cc[1] + cc[2] * cc[2]);
            for (int j = 0; j < 8; ++j) {
                float rho = 0.f;
                const int jf = fr - 101;   // the joint that moves the group's frame (-1: the base)
                if (jf >= 0 && (j >> 2) == (jf >> 2) && j <= jf) {
                    rho = cn;
                    for (int i = j + 1; i <= jf; ++i) rho += sqrtf(u.jt[i][0] * u.jt[i][0] + u.jt[i][1] * u.jt[i][1] + u.jt[i][2] * u.jt[i][2]);
                    rho *= 1.0f + 1e-5f;
                }
                u.grp_rho[ng][j] = rho;
            }
            ++ng;
            s = e;
        }
        for (int g = ng; g < SM_HGROUPS; ++g) { u.grp_frame[g] = 0; u.grp_off[g] = 0; u.grp_cnt[g] = 0; u.grp_r[g] = 0.f; }
        for (int k = 0; k < 3; ++k) { u.trunk_wmin[k] = FLT_MAX; u.trunk_wmax[k] = -FLT_MAX; }
        for (int s = 0; s < h.n_shapes; ++s) {
            const SmShape& sh = sc->shapes[h.shape_off + s];
            if (sh.frame != 100) continue;
            for (int i = sh.vert_off; i < sh.vert_off + sh.vert_cnt; ++i)
                for (int k = 0; k < 3; ++k) {
                    const float w = (float)(h.base_R[3 * k] * sc->verts[3 * i] + h.base_R[3 * k + 1] * sc->verts[3 * i + 1] +
                                            h.base_R[3 * k + 2] * sc->verts[3 * i + 2] + h.base_t[k]);
                    u.trunk_wmin[k] = fminf(u.trunk_wmin[k], w - (float)sh.margin - 1e-5f);
                    u.trunk_wmax[k] = fmaxf(u.trunk_wmax[k], w + (float)sh.margin + 1e-5f);
                }
        }
    }

    int rc = upload(&env->d_verts, verts);
    if (rc) return rc;
    d.verts = env->d_verts;
    while (lut.empty() || lut.size() % 4) lut.push_back(0u);   // staged in 16-byte vectors
    if ((rc = upload(&env->d_lut, lut))) { return rc; }
    d.lut = env->d_lut;
    if ((rc = upload(&env->d_hwidth, hwidth))) { return rc; }
    d.hwidth = env->d_hwidth;
    d.n_lut_words = (int)lut.size();
    if (env->human) {
        if ((rc = upload(&env->d_hpairs, hpairs))) return rc;
        if ((rc = upload(&env->d_hthresh, hthresh))) return rc;
        d.hu.brake_pairs = env->d_hpairs;
        d.hu.contact_thresh = env->d_hthresh;
        const size_t N = (size_t)num_envs;
        CU(cudaMalloc((void**)&env->d_hrange, N * 8 * 4 * sizeof(double)));
        CU(cudaMalloc((void**)&env->d_hbacc, N * SM_HBRAKE_STEPS * 8 * sizeof(double)));
        CU(cudaMalloc((void**)&env->d_hposes, N * SM_HBRAKE_POSES * 8 * sizeof(float)));
        CU(cudaMalloc((void**)&env->d_hbinfo, N * 4 * sizeof(int)));
        CU(cudaMemset(env->d_hbinfo, 0, N * 4 * sizeof(int)));
        CU(cudaMalloc((void**)&env->d_hunits, (N * SM_HBRAKE_POSES + 16) * sizeof(int)));
        CU(cudaMemset(env->d_hunits, 0, (N * SM_HBRAKE_POSES + 16) * sizeof(int)));
        CU(cudaMalloc((void**)&env->d_hscratch, N * SM_SCRATCH_FLOATS * sizeof(float)));
        CU(cudaMemset(env->d_hscratch, 0, N * SM_SCRATCH_FLOATS * sizeof(float)));
        CU(cudaMalloc((void**)&env->d_hpolicy, N * 16 * sizeof(float)));
        CU(cudaMemset(env->d_hpolicy, 0, N * 16 * sizeof(float)));
        env->smem_bytes_hplan = human_plan_smem_bytes(sc->human.n_arm_shapes);
    }
    for (int o = 0; o < sc->n_obstacles; ++o) {
        if (sc->obst_kind[o] != SM_OBST_PLANET) continue;
        std::vector<float4> pp(sc->planet_steps), pq(sc->planet_steps);
        for (int i = 0; i < sc->planet_steps; ++i) {
            pp[i] = make_float4((float)sc->planet_pos[o][3 * i], (float)sc->planet_pos[o][3 * i + 1],
                                (float)sc->planet_pos[o][3 * i + 2], 0.f);
            pq[i] = make_float4((float)sc->planet_quat[o][4 * i], (float)sc->planet_quat[o][4 * i + 1],
                                (float)sc->planet_quat[o][4 * i + 2], (float)sc->planet_quat[o][4 * i + 3]);
        }
        if ((rc = upload(&env->d_ppos[o], pp)) || (rc = upload(&env->d_pquat[o], pq))) { return rc; }
        d.planet_pos[o] = env->d_ppos[o];
        d.planet_quat[o] = env->d_pquat[o];
    }
    if (sc->n_obstacles > 0 && sc->obst_kind[0] == SM_OBST_PLANET) {
        std::vector<double> pl(sc->planet_local_xy, sc->planet_local_xy + 2 * sc->planet_steps);
        if ((rc = upload(&env->d_plocal, pl))) { return rc; }
        d.planet_local_xy = env->d_plocal;
    }
    {   // image of the shared-memory tables of the geometry kernels
        std::vector<SceneImage> img(1);
        memset(img.data(), 0, sizeof(SceneImage));
        SceneSmem& si = img[0].scene;
        memcpy(si.shapes, d.shapes, sizeof(si.shapes));
        memcpy(si.jR, d.jR, sizeof(si.jR)); memcpy(si.jt, d.jt, sizeof(si.jt)); memcpy(si.jaxis, d.jaxis, sizeof(si.jaxis));
        memcpy(si.static_pairs, d.static_pairs, sizeof(si.static_pairs));
        memcpy(si.self_pairs, d.self_pairs, sizeof(si.self_pairs));
        memcpy(si.mov_reward, d.mov_reward, sizeof(si.mov_reward));
        memcpy(si.mov_contact, d.mov_contact, sizeof(si.mov_contact));
        memcpy(si.contact_thresh, d.contact_thresh, sizeof(si.contact_thresh));
        memcpy(img[0].pair_tab, d.pair_tab, sizeof(img[0].pair_tab));
        memcpy(img[0].pair_rm, d.pair_rm, sizeof(img[0].pair_rm));
        if ((rc = upload(&env->d_scene_img, img))) { return rc; }
        d.scene_img = reinterpret_cast<const uint4*>(env->d_scene_img);
    }
    // pools: one start state per env is plenty of variety up to 65536; balls are consumed faster
    env->start_pool_n = num_envs < 65536 ? (num_envs < 1024 ? 1024 : num_envs) : 65536;
    env->ball_pool_n = (sc->n_obstacles > 0 && sc->obst_kind[0] == SM_OBST_BALL) ? 4 * env->start_pool_n : 0;
    CU(cudaMalloc((void**)&env->d_start_pool, (size_t)env->start_pool_n * SM_POOL_STRIDE * sizeof(double)));
    CU(cudaMemset(env->d_start_pool, 0, (size_t)env->start_pool_n * SM_POOL_STRIDE * sizeof(double)));
    if (env->ball_pool_n) CU(cudaMalloc((void**)&env->d_ball_pool, (size_t)env->ball_pool_n * SM_BALL_STRIDE * sizeof(double)));
    if (env->human) {
        env->htarget_pool_n = 2 * env->start_pool_n;
        CU(cudaMalloc((void**)&env->d_hstart_pool, (size_t)env->start_pool_n * SM_HPOOL_STRIDE * sizeof(double)));
        CU(cudaMemset(env->d_hstart_pool, 0, (size_t)env->start_pool_n * SM_HPOOL_STRIDE * sizeof(double)));
        CU(cudaMalloc((void**)&env->d_hpool_brake, (size_t)env->start_pool_n * SM_HBRAKE_STEPS * 8 * sizeof(double)));
        CU(cudaMemset(env->d_hpool_brake, 0, (size_t)env->start_pool_n * SM_HBRAKE_STEPS * 8 * sizeof(double)));
        CU(cudaMalloc((void**)&env->d_hpool_bcount, (size_t)env->start_pool_n * sizeof(int)));
        CU(cudaMemset(env->d_hpool_bcount, 0, (size_t)env->start_pool_n * sizeof(int)));
        CU(cudaMalloc((void**)&env->d_htarget_pool, (size_t)2 * env->htarget_pool_n * 4 * sizeof(double)));
        CU(cudaMemset(env->d_htarget_pool, 0, (size_t)2 * env->htarget_pool_n * 4 * sizeof(double)));
    }
    if (sc->use_target_points) {
        env->target_pool_n = 4 * env->start_pool_n;
        CU(cudaMalloc((void**)&env->d_target_pool, (size_t)env->target_pool_n * 4 * sizeof(double)));
        CU(cudaMemset(env->d_target_pool, 0, (size_t)env->target_pool_n * 4 * sizeof(double)));
    }
    CU(cudaMalloc((void**)&env->d_scratch, (size_t)num_envs * SM_SCRATCH_FLOATS * sizeof(float)));
    CU(cudaMemset(env->d_scratch, 0, (size_t)num_envs * SM_SCRATCH_FLOATS * sizeof(float)));
    CU(cudaMalloc((void**)&env->d_worklist, 2 * 8 * sizeof(int)));  // per env range: item counter, overflow count
    CU(cudaMemset(env->d_worklist, 0, 2 * 8 * sizeof(int)));
    {   // item buffer: the mean is a few dozen items per env-step; sized generously, overflow is reported loudly
        long long cap = (long long)num_envs * 192;
        if (cap < 65536) cap = 65536;
        if (const char* ov = getenv("SMENV_ITEM_CAPACITY")) {  // tests shrink the buffer to exercise the overflow report
            const long long v = atoll(ov);
            if (v > 0) cap = v;
        }
        env->item_capacity = (int)(cap > 0x7fffffffLL / 2 ? 0x7fffffffLL / 2 : cap);
        CU(cudaMalloc((void**)&env->d_items, (size_t)env->item_capacity * sizeof(GjkItem)));
        CU(cudaMalloc((void**)&env->d_res, (size_t)num_envs * SM_RES_STRIDE * sizeof(unsigned)));
        CU(cudaMemset(env->d_res, 0xff, (size_t)num_envs * SM_RES_STRIDE * sizeof(unsigned)));
        CU(cudaHostAlloc((void**)&env->h_flag, sizeof(int), cudaHostAllocMapped));
        *env->h_flag = 0;
        CU(cudaHostGetDevicePointer((void**)&env->d_flag, env->h_flag, 0));
        CU(cudaHostAlloc((void**)&env->h_step, sizeof(uint32_t), cudaHostAllocDefault));
        *env->h_step = 0;
        CU(cudaMalloc((void**)&env->d_step, sizeof(uint32_t)));
        CU(cudaMemset(env->d_step, 0, sizeof(uint32_t)));
    }
    CU(cudaMalloc((void**)&env->d_tasks, ((size_t)num_envs * 16 + 8) * sizeof(int)));
    CU(cudaMemset(env->d_tasks, 0, ((size_t)num_envs * 16 + 8) * sizeof(int)));
    CU(cudaMalloc((void**)&env->d_hpar, (size_t)num_envs * 8 * SM_HPAR * sizeof(double)));
    CU(cudaMalloc((void**)&env->d_cwork, ((size_t)num_envs * SM_COARSE_LANES + 8) * sizeof(int)));
    CU(cudaMemset(env->d_cwork, 0, ((size_t)num_envs * SM_COARSE_LANES + 8) * sizeof(int)));
    for (int c = 0; c < 8; ++c) {
        CU(cudaStreamCreateWithFlags(&env->side_streams[c], cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&env->side_fork[c], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&env->side_join[c], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&env->joint_fork[c], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&env->joint_join[c], cudaEventDisableTiming));
    }
    CU(cudaMalloc((void**)&env->d_heavy, ((size_t)num_envs * 8 + 8) * sizeof(int)));
    CU(cudaMemset(env->d_heavy, 0, ((size_t)num_envs * 8 + 8) * sizeof(int)));
    if (sc->human.enabled) {
        CU(cudaMalloc((void**)&env->d_hheavy, ((size_t)num_envs * 8 + 8) * sizeof(int)));
        CU(cudaMemset(env->d_hheavy, 0, ((size_t)num_envs * 8 + 8) * sizeof(int)));
        CU(cudaMalloc((void**)&env->d_htasks, ((size_t)num_envs * 16 + 8) * sizeof(int)));
        CU(cudaMemset(env->d_htasks, 0, ((size_t)num_envs * 16 + 8) * sizeof(int)));
        CU(cudaMalloc((void**)&env->d_hhpar, (size_t)num_envs * 8 * SM_HPAR * sizeof(double)));
    }
    CU(cudaMalloc((void**)&env->d_counters, 24 * sizeof(unsigned long long)));
    CU(cudaMemset(env->d_counters, 0, 24 * sizeof(unsigned long long)));

    env->smem_bytes = smem_bytes_for(sc->n_verts, SM_WARPS_PER_BLOCK);
    env->smem_bytes_broad = smem_bytes_for(0, SM_WARPS_PER_BLOCK);
    {   // the planning kernels' shared memory (scene image + per-warp scratch, a compile-time size) is above the 48 KB default
        static bool raised[SM_MAX_DEVICES] = {};
        if (!raised[device % SM_MAX_DEVICES]) {
            const int b = (int)env->smem_bytes_broad;
            CU(cudaFuncSetAttribute(contact_coarse_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
            CU(cudaFuncSetAttribute(contact_coarse_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
            CU(cudaFuncSetAttribute(contact_plan_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
            CU(cudaFuncSetAttribute(contact_plan_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
            CU(cudaFuncSetAttribute(distance_plan_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
            CU(cudaFuncSetAttribute(distance_plan_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
            raised[device % SM_MAX_DEVICES] = true;
        }
    }
    env->smem_bytes_gjk = gjk_smem_bytes(sc->n_verts, d.n_lut_words, sc->n_shapes);
    {   // opt-in shared-memory limits are per function and process wide: only ever raised, so that an env created
        // earlier with bigger tables keeps launching
        size_t& lim_gjk = g_smem_gjk[device % SM_MAX_DEVICES];
        size_t& lim_geom = g_smem_geom[device % SM_MAX_DEVICES];
        if (env->smem_bytes_gjk > lim_gjk) {
            CU(cudaFuncSetAttribute(gjk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<false, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<true, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<false, 768>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<true, 768>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<false, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<true, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<false, 384>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            CU(cudaFuncSetAttribute(gjk_kernel<true, 384>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_gjk));
            lim_gjk = env->smem_bytes_gjk;
        }
        if (env->smem_bytes > lim_geom) {
            CU(cudaFuncSetAttribute(fill_ball_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes));
            CU(cudaFuncSetAttribute(fill_start_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes));
            CU(cudaFuncSetAttribute(fill_target_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes));
            CU(cudaFuncSetAttribute(distances_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes));
            CU(cudaFuncSetAttribute(debug_gjk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes));
            CU(cudaFuncSetAttribute(fill_human_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes));
            lim_geom = env->smem_bytes;
        }
    }
    // persistent grid: as many CTAs as fit on the device at once (a multiple of the SM count), each looping over envs
    int sms = 0, per_sm = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, distances_kernel, SM_WARPS_PER_BLOCK * 32, env->smem_bytes));
    if (per_sm < 1) { return fail(SM_ERR_CUDA, "pool kernels do not fit on an SM"); }
    env->grid = sms * per_sm;
    env->sms = sms;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, distance_plan_kernel<false>, SM_WARPS_PER_BLOCK * 32, env->smem_bytes_broad));
    if (per_sm < 1) { return fail(SM_ERR_CUDA, "planning kernels do not fit on an SM"); }
    env->grid_broad = sms * per_sm;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gjk_kernel<false>, GJK_THREADS, env->smem_bytes_gjk));
    if (per_sm < 1) { return fail(SM_ERR_CUDA, "gjk kernel does not fit on an SM"); }
    if (per_sm == 1 && !getenv("SMENV_GJK_256")) {   // one big CTA instead of a half-empty SM
        int per_sm_512 = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_512, gjk_kernel<false, 512>, 512, env->smem_bytes_gjk));
        if (per_sm_512 >= 1) { env->gjk_threads = 512; per_sm = per_sm_512; }
        // 24 warps under an 80-register cap (8 bytes of spill) hide more of the dependent-issue latency than 16 warps at
        // 107 registers: space_bm GJK 221 -> 211 us, Human 170 -> 166 us; 32 warps at 64 registers spill and lose
        int per_sm_768 = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_768, gjk_kernel<false, 768>, 768, env->smem_bytes_gjk));
        if (per_sm_768 >= 1 && !getenv("SMENV_GJK_512")) { env->gjk_threads = 768; per_sm = per_sm_768; }
    }
    if (const char* e = getenv("SMENV_GJK_THREADS")) {   // experiments: 24 / 32 warps under an 85 / 64-register cap
        const int t = atoi(e);
        int fit = 0;
        if (t == 768) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, gjk_kernel<false, 768>, 768, env->smem_bytes_gjk));
        if (t == 1024) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, gjk_kernel<false, 1024>, 1024, env->smem_bytes_gjk));
        if (t == 384) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, gjk_kernel<false, 384>, 384, env->smem_bytes_gjk));
        if (fit >= 1) { env->gjk_threads = t; per_sm = fit; }
    }
    env->grid_gjk = sms * per_sm;
    if (sc->human.enabled) {
        static size_t g_smem_hplan[SM_MAX_DEVICES] = {};   // under the create lock; only ever raised, like the limits above
        size_t& lim = g_smem_hplan[device % SM_MAX_DEVICES];
        if (env->smem_bytes_hplan > lim) {
            CU(cudaFuncSetAttribute(human_brake_plan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->smem_bytes_hplan));
            lim = env->smem_bytes_hplan;
        }
        int per = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, human_brake_plan_kernel, HBP_THREADS, env->smem_bytes_hplan));
        if (per < 1) { return fail(SM_ERR_CUDA, "the human's braking-check planning kernel does not fit on an SM"); }
        env->grid_hplan = sms * per;
    }
    // big batches step as two env ranges side by side: the latency-bound tails of one range's kernels (the longest
    // position-bound solve, the last GJK pairs) hide behind the other's (Space, 65 536 envs: 799 -> 748 us per step)
    if (const char* e = getenv("SMENV_STEP_RANGES")) env->step_ranges = atoi(e) < 1 ? 1 : (atoi(e) > 8 ? 8 : atoi(e));
    else env->step_ranges = num_envs >= 16384 ? 2 : 1;
    guard.env = nullptr;
    *out = env;
    return SM_OK;
}

extern "C" int smenv_destroy(SmEnv* env) {
    if (!env) return SM_OK;
    {
        DevLock dev_lock_(env);
        cudaSetDevice(env->device);
        SmEnv*& active = g_active[env->device % SM_MAX_DEVICES];
        if (active == env) { cudaDeviceSynchronize(); active = nullptr; }
    }
    cudaFree(env->d_verts); cudaFree(env->d_lut); cudaFree(env->d_hwidth); cudaFree(env->d_scene_img); cudaFree(env->d_plocal); cudaFree(env->d_start_pool); cudaFree(env->d_ball_pool); cudaFree(env->d_target_pool);
    cudaFree(env->d_counters); cudaFree(env->d_scratch); cudaFree(env->d_worklist); cudaFree(env->d_heavy); cudaFree(env->d_cwork); cudaFree(env->d_tasks); cudaFree(env->d_hpar); cudaFree(env->d_hheavy); cudaFree(env->d_htasks); cudaFree(env->d_hhpar); cudaFree(env->d_items); cudaFree(env->d_res);
    if (env->h_flag) cudaFreeHost(env->h_flag);
    if (env->h_step) cudaFreeHost(env->h_step);
    cudaFree(env->d_step);
    for (void* q : env->net_allocs) cudaFree(q);
    cudaFree(env->d_risk); cudaFree(env->d_backup); cudaFree(env->d_exec); cudaFree(env->d_risky); cudaFree(env->d_gate_list);
    cudaFree(env->d_hpairs); cudaFree(env->d_hthresh); cudaFree(env->d_hrange); cudaFree(env->d_hbacc); cudaFree(env->d_hposes);
    cudaFree(env->d_hbinfo); cudaFree(env->d_hunits); cudaFree(env->d_hscratch); cudaFree(env->d_hpolicy); cudaFree(env->d_hstart_pool); cudaFree(env->d_hpool_brake); cudaFree(env->d_hpool_bcount); cudaFree(env->d_htarget_pool);
    for (int i = 0; i <= SM_K_COUNT; ++i) if (env->ev[i]) cudaEventDestroy(env->ev[i]);
    for (int c = 0; c < 8; ++c) {
        if (env->chunk_streams[c]) cudaStreamDestroy(env->chunk_streams[c]);
        if (env->chunk_done[c]) cudaEventDestroy(env->chunk_done[c]);
    }
    if (env->chunk_fork) cudaEventDestroy(env->chunk_fork);
    for (int c = 0; c < 8; ++c) {
        if (env->side_streams[c]) cudaStreamDestroy(env->side_streams[c]);
        if (env->side_fork[c]) cudaEventDestroy(env->side_fork[c]);
        if (env->side_join[c]) cudaEventDestroy(env->side_join[c]);
        if (env->joint_fork[c]) cudaEventDestroy(env->joint_fork[c]);
        if (env->joint_join[c]) cudaEventDestroy(env->joint_join[c]);
    }
    if (env->host_graph) cudaGraphExecDestroy(env->host_graph);
    if (env->host_order) cudaEventDestroy(env->host_order);
    if (env->host_stream) cudaStreamDestroy(env->host_stream);
    for (int o = 0; o < SM_MAX_OBSTACLES; ++o) { cudaFree(env->d_ppos[o]); cudaFree(env->d_pquat[o]); }
    delete env;
    return SM_OK;
}

static int grid_for(const SmEnv* env, int items) {
    int blocks = (items + SM_WARPS_PER_BLOCK - 1) / SM_WARPS_PER_BLOCK;
    return blocks < env->grid ? blocks : env->grid;
}

extern "C" int smenv_pool_sizes(SmEnv* env, int* start_pool, int* ball_pool) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    if (start_pool) *start_pool = env->start_pool_n;
    if (ball_pool) *ball_pool = env->ball_pool_n;
    return SM_OK;
}
extern "C" int smenv_pool_ptrs(SmEnv* env, double** start_pool, double** ball_pool) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    if (start_pool) *start_pool = env->d_start_pool;
    if (ball_pool) *ball_pool = env->d_ball_pool;
    return SM_OK;
}

extern "C" int smenv_copy_pools(SmEnv* env, double* host_start, double* host_ball) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    CU(cudaSetDevice(env->device));
    CU(cudaDeviceSynchronize());
    if (host_start)
        CU(cudaMemcpy(host_start, env->d_start_pool, (size_t)env->start_pool_n * SM_POOL_STRIDE * sizeof(double),
                      cudaMemcpyDeviceToHost));
    if (host_ball && env->ball_pool_n)
        CU(cudaMemcpy(host_ball, env->d_ball_pool, (size_t)env->ball_pool_n * SM_BALL_STRIDE * sizeof(double),
                      cudaMemcpyDeviceToHost));
    return SM_OK;
}

extern "C" int smenv_fill_pools(SmEnv* env, uint64_t seed, SmStream s) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    PoolArgs A{env->d_start_pool, env->start_pool_n, env->d_ball_pool, env->ball_pool_n, (uint32_t)seed, (uint32_t)(seed >> 32),
               env->human ? env->d_hstart_pool : nullptr};
    if (env->human) {   // the nested env's pools first: the robot's start poses keep clear of the human's
        HumanPoolArgs H{env->d_hstart_pool, env->start_pool_n, env->d_htarget_pool, env->htarget_pool_n, (uint32_t)seed,
                        (uint32_t)(seed >> 32)};
        fill_human_pool_kernel<<<grid_for(env, env->start_pool_n + 2 * env->htarget_pool_n), SM_WARPS_PER_BLOCK * 32,
                                 env->smem_bytes, stream>>>(H);
        human_pool_braking_kernel<<<(env->start_pool_n * 8 + 255) / 256, 256, 0, stream>>>(env->d_hstart_pool, env->start_pool_n,
                                                                                         env->d_hpool_brake, env->d_hpool_bcount);
        env->launches += 2;
    }
    if (env->ball_pool_n) {
        fill_ball_pool_kernel<<<grid_for(env, env->ball_pool_n), SM_WARPS_PER_BLOCK * 32, env->smem_bytes, stream>>>(A);
        env->launches++;
    }
    fill_start_pool_kernel<<<grid_for(env, env->start_pool_n), SM_WARPS_PER_BLOCK * 32, env->smem_bytes, stream>>>(A);
    env->launches++;
    if (env->target_pool_n) {
        fill_target_pool_kernel<<<grid_for(env, env->target_pool_n), SM_WARPS_PER_BLOCK * 32, env->smem_bytes, stream>>>(
            env->d_target_pool, env->target_pool_n, (uint32_t)seed, (uint32_t)(seed >> 32));
        env->launches++;
    }
    CU(cudaGetLastError());
    env->pools_filled = true;
    return SM_OK;
}

// helper: is the pointer device memory?
static bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

__global__ void set_state_kernel(SmBuffers buf, int n, int nj, const double* q, const double* v, const double* a,
                                 const double* obst, const uint8_t* mask, double tvdt) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int env = i >> 5, lane = i & 31;
    if (env >= n || (mask && !mask[env])) return;
    int grp = lane >> 3, j = lane & 7;
    double val = 0.0;
    if (j < nj) {
        double qq = q[(size_t)env * nj + j], vv = v[(size_t)env * nj + j];
        // the reset poses the robot and runs one stepSimulation with the start state as motor target
        // (safe_motions_base.py:959-978): the tracked pose leaves the start position by track_vel * dt * v0
        val = grp == 0 ? qq : grp == 1 ? vv : grp == 2 ? a[(size_t)env * nj + j] : __dadd_rn(qq, __dmul_rn(tvdt, vv));
    }
    buf.kin[(size_t)env * SM_KIN_STRIDE + lane] = val;
    if (obst && lane < SM_OBST_STRIDE) buf.obst[(size_t)env * SM_OBST_STRIDE + lane] = obst[(size_t)env * SM_OBST_STRIDE + lane];
    if (lane == 0) {
        int* ep = buf.episode + 4 * (size_t)env;
        ep[0] = 0;
        ep[3] = 0;   // no risky action yet in this episode
        buf.ep_return[env] = 0.0;
    }
}

extern "C" int smenv_set_state(SmEnv* env, const SmBuffers* buf, const double* q, const double* v, const double* a,
                               const double* obst, const uint8_t* mask, SmStream s) {
    if (!env || !buf || !q || !v || !a) return fail(SM_ERR_ARG, "smenv_set_state: null argument");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    const int n = env->n, nj = env->host_scene.n_joints;
    // host pointers are staged through temporary device buffers
    std::vector<void*> tmp;
    auto stage = [&](const void* p, size_t bytes, const void** out) -> int {
        if (!p || is_device_ptr(p)) { *out = p; return SM_OK; }
        void* dptr = nullptr;
        CU(cudaMalloc(&dptr, bytes));
        tmp.push_back(dptr);
        CU(cudaMemcpyAsync(dptr, p, bytes, cudaMemcpyHostToDevice, stream));
        *out = dptr;
        return SM_OK;
    };
    const void *dq, *dv, *da, *dob, *dm;
    if ((rc = stage(q, (size_t)n * nj * 8, &dq)) || (rc = stage(v, (size_t)n * nj * 8, &dv)) ||
        (rc = stage(a, (size_t)n * nj * 8, &da)) || (rc = stage(obst, (size_t)n * SM_OBST_STRIDE * 8, &dob)) ||
        (rc = stage(mask, (size_t)n, &dm)))
        return rc;
    double dt = env->host_scene.ts / (double)env->host_scene.substeps;
    double tvdt = env->host_scene.track_vel * dt;
    set_state_kernel<<<(n * 32 + 255) / 256, 256, 0, stream>>>(*buf, n, nj, (const double*)dq, (const double*)dv,
                                                               (const double*)da, (const double*)dob,
                                                               (const uint8_t*)dm, tvdt);
    env->launches++;
    CU(cudaGetLastError());
    if (env->host_scene.use_target_points && buf->target) {  // first target point from the pool (if it is filled)
        target_init_kernel<<<(n + 255) / 256, 256, 0, stream>>>(*buf, n, nullptr, (const uint8_t*)dm,
                                                                env->pools_filled ? env->d_target_pool : nullptr,
                                                                env->pools_filled ? env->target_pool_n : 0,
                                                                (uint32_t)env->seed, (uint32_t)(env->seed >> 32));
        env->launches++;
    }
    if (buf->obs) {
        observation_kernel<<<(n * 32 + 255) / 256, 256, 0, stream>>>(*buf, n);
        env->launches++;
        CU(cudaGetLastError());
    }
    if (!tmp.empty()) {
        CU(cudaStreamSynchronize(stream));
        for (void* p : tmp) cudaFree(p);
    }
    return SM_OK;
}

extern "C" int smenv_set_targets(SmEnv* env, const SmBuffers* buf, const double* first_target, const uint8_t* mask,
                                 SmStream s) {
    if (!env || !buf || !buf->target || !first_target) return fail(SM_ERR_ARG, "smenv_set_targets: null argument");
    if (!env->host_scene.use_target_points) return fail(SM_ERR_STATE, "smenv_set_targets: the scene has no target points");
    if (mask && !is_device_ptr(mask)) return fail(SM_ERR_ARG, "smenv_set_targets: mask must be a device pointer");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    const int n = env->n;
    double* tmp = nullptr;
    const double* dft = first_target;
    if (!is_device_ptr(first_target)) {
        CU(cudaMalloc((void**)&tmp, (size_t)n * 3 * sizeof(double)));
        CU(cudaMemcpyAsync(tmp, first_target, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, stream));
        dft = tmp;
    }
    target_init_kernel<<<(n + 255) / 256, 256, 0, stream>>>(*buf, n, dft, mask, nullptr, 0, (uint32_t)env->seed,
                                                            (uint32_t)(env->seed >> 32));
    env->launches++;
    if (buf->obs) {
        observation_kernel<<<(n * 32 + 255) / 256, 256, 0, stream>>>(*buf, n);
        env->launches++;
    }
    CU(cudaGetLastError());
    if (tmp) { CU(cudaStreamSynchronize(stream)); cudaFree(tmp); }
    return SM_OK;
}

extern "C" int smenv_observation(SmEnv* env, const SmBuffers* buf, SmStream s) {
    if (!env || !buf || !buf->obs) return fail(SM_ERR_ARG, "smenv_observation: null argument");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    observation_kernel<<<(env->n * 32 + 255) / 256, 256, 0, stream>>>(*buf, env->n);
    env->launches++;
    CU(cudaGetLastError());
    return SM_OK;
}

extern "C" int smenv_reset(SmEnv* env, const SmBuffers* buf, const uint8_t* mask, SmStream s) {
    if (!env || !buf) return fail(SM_ERR_ARG, "smenv_reset: null argument");
    if (!env->pools_filled) return fail(SM_ERR_STATE, "smenv_reset: call smenv_fill_pools first");
    if (mask && !is_device_ptr(mask)) return fail(SM_ERR_ARG, "smenv_reset: mask must be a device pointer");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    ResetArgs A{*buf, env->n, mask, env->d_start_pool, env->start_pool_n, env->d_target_pool, env->target_pool_n,
                (uint32_t)env->seed, (uint32_t)(env->seed >> 32)};
    reset_kernel<<<(env->n * 32 + 255) / 256, 256, 0, stream>>>(A);
    env->launches++;
    if (env->human) {
        if (!buf->hkin || !buf->hstate || !buf->hbrake || !buf->hobs)
            return fail(SM_ERR_ARG, "smenv_reset: the Human scene needs the hkin / hstate / hbrake / hobs buffers");
        HumanArgs H;
        memset(&H, 0, sizeof(H));
        H.buf = *buf; H.n = env->n; H.env_base = 0; H.k0 = (uint32_t)env->seed; H.k1 = (uint32_t)(env->seed >> 32);
        H.mask = mask; H.start_pool = env->d_hstart_pool; H.start_pool_n = env->start_pool_n;
        H.pool_brake = env->d_hpool_brake; H.pool_bcount = env->d_hpool_bcount;
        H.target_pool = env->d_htarget_pool; H.target_pool_n = env->htarget_pool_n;
        human_reset_kernel<<<(env->n * 8 + 255) / 256, 256, 0, stream>>>(H, 0);
        env->launches++;
    }
    CU(cudaGetLastError());
    return SM_OK;
}

extern "C" int smenv_set_human_actions_external(SmEnv* env, int external) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    if (!env->human) return fail(SM_ERR_STATE, "smenv_set_human_actions_external: the scene has no human");
    env->human_external = external != 0;
    if (env->host_graph) { cudaGraphExecDestroy(env->host_graph); env->host_graph = nullptr; }
    return SM_OK;
}

extern "C" int smenv_human_pool_sizes(SmEnv* env, int* start_pool, int* target_pool) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    if (start_pool) *start_pool = env->human ? env->start_pool_n : 0;
    if (target_pool) *target_pool = env->human ? env->htarget_pool_n : 0;
    return SM_OK;
}

extern "C" int smenv_copy_human_pools(SmEnv* env, double* host_start, double* host_target) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    if (!env->human) return fail(SM_ERR_STATE, "smenv_copy_human_pools: the scene has no human");
    CU(cudaSetDevice(env->device));
    CU(cudaDeviceSynchronize());
    if (host_start)
        CU(cudaMemcpy(host_start, env->d_hstart_pool, (size_t)env->start_pool_n * SM_HPOOL_STRIDE * sizeof(double), cudaMemcpyDeviceToHost));
    if (host_target)
        CU(cudaMemcpy(host_target, env->d_htarget_pool, (size_t)2 * env->htarget_pool_n * 4 * sizeof(double), cudaMemcpyDeviceToHost));
    return SM_OK;
}

extern "C" int smenv_set_human_state(SmEnv* env, const SmBuffers* buf, const double* hq, const double* hv, const double* ha,
                                     const double* first_target, const int32_t* active_arm, const uint8_t* mask, SmStream s) {
    if (!env || !buf || !hq || !hv || !ha || !first_target) return fail(SM_ERR_ARG, "smenv_set_human_state: null argument");
    if (!env->human) return fail(SM_ERR_STATE, "smenv_set_human_state: the scene has no human");
    if (!buf->hkin || !buf->hstate || !buf->hbrake || !buf->hobs) return fail(SM_ERR_ARG, "smenv_set_human_state: human buffers missing");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    const int n = env->n;
    std::vector<void*> tmp;
    auto stage = [&](const void* p, size_t bytes, const void** out) -> int {
        if (!p || is_device_ptr(p)) { *out = p; return SM_OK; }
        void* dptr = nullptr;
        CU(cudaMalloc(&dptr, bytes));
        tmp.push_back(dptr);
        CU(cudaMemcpyAsync(dptr, p, bytes, cudaMemcpyHostToDevice, stream));
        *out = dptr;
        return SM_OK;
    };
    const void *dq, *dv, *da, *dt, *dar, *dm;
    if ((rc = stage(hq, (size_t)n * 64, &dq)) || (rc = stage(hv, (size_t)n * 64, &dv)) || (rc = stage(ha, (size_t)n * 64, &da)) ||
        (rc = stage(first_target, (size_t)n * 24, &dt)) || (rc = stage(active_arm, (size_t)n * 4, &dar)) ||
        (rc = stage(mask, (size_t)n, &dm)))
        return rc;
    HumanArgs H;
    memset(&H, 0, sizeof(H));
    H.buf = *buf; H.n = n; H.mask = (const uint8_t*)dm;
    human_set_state_kernel<<<(n * 8 + 255) / 256, 256, 0, stream>>>(H, (const double*)dq, (const double*)dv, (const double*)da,
                                                               (const double*)dt, (const int32_t*)dar);
    env->launches++;
    CU(cudaGetLastError());
    if (!tmp.empty()) {
        CU(cudaStreamSynchronize(stream));
        for (void* p : tmp) cudaFree(p);
    }
    return SM_OK;
}

#define SM_MAX_CHUNKS 8 /* env ranges that can be in flight at once (smenv_step_host) */

// SmBuffers as seen by a launch over the envs [e0, e0 + m)
static SmBuffers buffers_at(const SmBuffers& b, int e0, int nj, int obs_size) {
    SmBuffers o = b;
    o.kin = b.kin + (size_t)e0 * SM_KIN_STRIDE;
    o.obst = b.obst + (size_t)e0 * SM_OBST_STRIDE;
    o.episode = b.episode + (size_t)e0 * 4;
    o.ep_return = b.ep_return + e0;
    if (b.actions) o.actions = b.actions + (size_t)e0 * nj;
    if (b.obs) o.obs = b.obs + (size_t)e0 * obs_size;
    if (b.reward) o.reward = b.reward + e0;
    if (b.done) o.done = b.done + e0;
    if (b.term_reason) o.term_reason = b.term_reason + e0;
    if (b.info) o.info = b.info + (size_t)e0 * SM_INFO_STRIDE;
    if (b.target) o.target = b.target + (size_t)e0 * SM_TP_STRIDE;
    if (b.hkin) o.hkin = b.hkin + (size_t)e0 * SM_KIN_STRIDE;
    if (b.hstate) o.hstate = b.hstate + (size_t)e0 * SM_HSTATE_STRIDE;
    if (b.hbrake) o.hbrake = b.hbrake + (size_t)e0 * SM_HBRAKE_STEPS * SM_HUMAN_JOINTS;
    if (b.hobs) o.hobs = b.hobs + (size_t)e0 * SM_HOBS_STRIDE;
    if (b.hactions) o.hactions = b.hactions + (size_t)e0 * SM_HUMAN_JOINTS;
    if (b.epacc) o.epacc = b.epacc + (size_t)e0 * SM_EP_STRIDE;
    if (b.epinfo) o.epinfo = b.epinfo + (size_t)e0 * SM_EP_STRIDE;
    return o;
}

struct MlpSeg { const float* p; int stride, w; };
static int mlp_launch(SmEnv* env, int which, MlpSeg s0, MlpSeg s1, MlpSeg s2, float* out, int out_stride, int n,
                      cudaStream_t stream) {
    if (!env->net_loaded[which]) return fail(SM_ERR_STATE, "network not loaded (smenv_mlp_load)");
    const MlpNet& net = env->nets[which];
    if (s0.w + s1.w + s2.w != net.n_in) return fail(SM_ERR_ARG, "network input width does not match the loaded weights");
    MlpArgs M;
    M.net = net; M.n = n; M.out = out; M.out_stride = out_stride;
    const MlpSeg segs[3] = {s0, s1, s2};
    for (int i = 0; i < 3; ++i) { M.in[i] = segs[i].p; M.in_stride[i] = segs[i].stride; M.in_w[i] = segs[i].w; }
    const int tiles = (n + MLP_TILE_M - 1) / MLP_TILE_M;
    const int grid = tiles < env->sms ? tiles : env->sms;   // one CTA per SM (202 KB of shared memory, all of TMEM)
    mlp_kernel<<<grid, MLP_THREADS, MLP_SM_BYTES, stream>>>(M);
    env->launches++;
    CU(cudaGetLastError());
    return SM_OK;
}


// The risk gate over the envs of `bv` (a view of m envs): risk network on (risk observation, proposed action), backup
// policy on the risk observation, then the executed actions into `exec` (== bv.actions: in place).
static int mlp_exact_launch(SmEnv* env, int which, MlpSeg s0, MlpSeg s1, MlpSeg s2, const int* rows, const int* n_rows,
                            int max_rows, float* out, int out_stride, int n_write, cudaStream_t stream) {
    if (!env->net_loaded[which]) return fail(SM_ERR_STATE, "network not loaded (smenv_mlp_load)");
    MlpExactArgs X;
    memset(&X, 0, sizeof(X));
    X.net = env->nets[which]; X.rows = rows; X.n_rows = n_rows; X.n_rows_host = max_rows;
    const MlpSeg segs[3] = {s0, s1, s2};
    for (int i = 0; i < 3; ++i) { X.in[i] = segs[i].p; X.in_stride[i] = segs[i].stride; X.in_w[i] = segs[i].w; }
    X.out = out; X.out_stride = out_stride; X.n_write = n_write;
    int blocks = (max_rows + MLP_EXACT_ROWS - 1) / MLP_EXACT_ROWS;
    if (blocks > 4 * env->sms) blocks = 4 * env->sms;   // grid-stride over the list; blocks beyond its length exit at once
    if (blocks < 1) blocks = 1;
    mlp_exact_kernel<<<blocks, 256, MLP_EXACT_SMEM, stream>>>(X);
    env->launches++;
    CU(cudaGetLastError());
    return SM_OK;
}

// The risk gate over the envs of `bv` (a view of m envs starting at env e0 of the whole vector env): risk network on
// (risk observation, proposed action) on the tensor cores; in exact mode the rows within gate_band of the threshold are
// re-rated in float32 and the backup policy's action of the risky rows is computed in float32 on that subset; else the
// backup policy runs on the tensor cores for every row.  Executed actions go to `exec` (== bv.actions: in place).
static int gate_launch(SmEnv* env, const SmBuffers& bv, int e0, int m, int chunk, float threshold, float* risk, uint8_t* risky,
                       float* backup, float* exec, cudaStream_t stream) {
    const DevScene& hs = env->host_scene;
    const int nj = hs.n_joints, ow = hs.obs_size;
    // the risk observation is the observation without the target-point entries (observations.py:419-431): joint
    // position / velocity / acceleration, then the obstacle entries
    const int n_tp = hs.use_target_points ? 3 * hs.obs_add_tp_pos + 3 * hs.obs_add_tp_rel : 0;
    const MlpSeg kinem{bv.obs, ow, 3 * nj}, rest{bv.obs + 3 * nj + n_tp, ow, ow - 3 * nj - n_tp};
    const MlpSeg act{bv.actions, nj, nj}, none{nullptr, 0, 0};
    int rc;
    if ((rc = mlp_launch(env, SM_NET_RISK, kinem, rest, act, risk, 1, m, stream))) return rc;
    if (!env->gate_exact) {
        if ((rc = mlp_launch(env, SM_NET_BACKUP, kinem, rest, none, backup, MLP_MAX_OUT, m, stream))) return rc;
        risk_gate_kernel<<<(m + 255) / 256, 256, 0, stream>>>(bv.actions, exec, risk, backup, MLP_MAX_OUT, nj, m, threshold, risky);
        env->launches++;
        CU(cudaGetLastError());
        return SM_OK;
    }
    int* counts = env->d_gate_list + 2 * chunk;
    int* near_list = env->d_gate_list + 32 + e0;
    int* risky_list = env->d_gate_list + 32 + env->n + e0;
    CU(cudaMemsetAsync(counts, 0, 2 * sizeof(int), stream));
    gate_band_kernel<<<(m + 255) / 256, 256, 0, stream>>>(risk, m, threshold, env->gate_band, near_list, counts);
    env->launches++;
    if ((rc = mlp_exact_launch(env, SM_NET_RISK, kinem, rest, act, near_list, counts, m, risk, 1, 1, stream))) return rc;
    risk_decide_kernel<<<(m + 255) / 256, 256, 0, stream>>>(bv.actions, exec, risk, nj, m, threshold, risky, risky_list, counts + 1);
    env->launches++;
    if ((rc = mlp_exact_launch(env, SM_NET_BACKUP, kinem, rest, none, risky_list, counts + 1, m, exec, nj, nj, stream))) return rc;
    CU(cudaGetLastError());
    return SM_OK;
}

static void launch_gjk(SmEnv* env, const GjkArgs& G, cudaStream_t stream) {
    if (env->gjk_threads == 1024) {
        if (env->count) gjk_kernel<true, 1024><<<env->grid_gjk, 1024, env->smem_bytes_gjk, stream>>>(G);
        else gjk_kernel<false, 1024><<<env->grid_gjk, 1024, env->smem_bytes_gjk, stream>>>(G);
    } else if (env->gjk_threads == 768) {
        if (env->count) gjk_kernel<true, 768><<<env->grid_gjk, 768, env->smem_bytes_gjk, stream>>>(G);
        else gjk_kernel<false, 768><<<env->grid_gjk, 768, env->smem_bytes_gjk, stream>>>(G);
    } else if (env->gjk_threads == 512) {
        if (env->count) gjk_kernel<true, 512><<<env->grid_gjk, 512, env->smem_bytes_gjk, stream>>>(G);
        else gjk_kernel<false, 512><<<env->grid_gjk, 512, env->smem_bytes_gjk, stream>>>(G);
    } else if (env->gjk_threads == 384) {
        if (env->count) gjk_kernel<true, 384><<<env->grid_gjk, 384, env->smem_bytes_gjk, stream>>>(G);
        else gjk_kernel<false, 384><<<env->grid_gjk, 384, env->smem_bytes_gjk, stream>>>(G);
    } else {
        if (env->count) gjk_kernel<true><<<env->grid_gjk, GJK_THREADS, env->smem_bytes_gjk, stream>>>(G);
        else gjk_kernel<false><<<env->grid_gjk, GJK_THREADS, env->smem_bytes_gjk, stream>>>(G);
    }
}

// The kernels of one env step over the envs [e0, e0 + m) on `stream`, with the work lists of slot `chunk`: every list
// of the whole env ([0] = count, [1..k n] = entries) holds the sub-lists of the ranges back to back, the range's
// sub-list starting at entry k * e0 + chunk (its own count first).  Ranges in flight at once need distinct slots.
static int step_range(SmEnv* env, const SmBuffers* full, int e0, int m, int chunk, int auto_reset, int random_actions,
                      uint32_t step_counter, bool tk, cudaStream_t stream, const uint32_t* step_ptr = nullptr) {
    const SmBuffers buf_v = buffers_at(*full, e0, env->host_scene.n_joints, env->host_scene.obs_size);
    const SmBuffers* buf = &buf_v;
    const int per_env_items = env->item_capacity / env->n;
    int* worklist = env->d_worklist + 2 * chunk;
    float* scratch = env->d_scratch + (size_t)e0 * SM_SCRATCH_FLOATS;
    unsigned* res = env->d_res + (size_t)e0 * SM_RES_STRIDE;
    GjkItem* items = env->d_items + (size_t)e0 * per_env_items;
    const int capacity = e0 == 0 && m == env->n ? env->item_capacity : m * per_env_items;
    int* heavy = env->d_heavy + (size_t)e0 * 8 + chunk;
    int* cwork = env->d_cwork + (size_t)e0 * SM_COARSE_LANES + chunk;
    int* tasks = env->d_tasks + (size_t)e0 * 16 + chunk;
    JointArgs JA;
    JA.buf = *buf; JA.n = m; JA.random_actions = random_actions;
    JA.k0 = (uint32_t)env->seed; JA.k1 = (uint32_t)(env->seed >> 32);
    JA.step_counter = step_counter;
    JA.env_base = e0;
    JA.scratch = scratch;
    JA.worklist = worklist;  // clears the item counter and the overflow count
    JA.heavy = heavy;
    JA.cwork = cwork;
    JA.tasks = tasks;
    JA.hpar = env->d_hpar + (size_t)e0 * 8 * SM_HPAR;
    JA.counters = env->count ? env->d_counters : nullptr;
    JA.exec = nullptr;
    JA.set = 0; JA.nj = env->host_scene.n_joints; JA.defer = 0; JA.range_out = nullptr;
    JA.track_vel = env->host_scene.track_vel; JA.store_qset = env->host_scene.use_target_points;
    JA.keep_overflow = env->human ? 1 : 0;
    JA.clear_extra = nullptr;
    if (env->human) JA.worklist = nullptr;   // the nested env's kernels clear the counters (its braking check emits items first)
    const bool gate = env->gate_threshold >= 0.0f;
    if (gate) {   // actions.py:303-340: rate the proposed action, execute the backup policy's where it is risky
        if (!buf->obs) return fail(SM_ERR_ARG, "smenv_step: the risk gate needs the observation buffer");
        if (random_actions) {
            if (!buf->actions) return fail(SM_ERR_ARG, "smenv_step: the risk gate needs the action buffer");
            random_actions_kernel<<<(m * env->host_scene.n_joints + 255) / 256, 256, 0, stream>>>(
                const_cast<float*>(buf->actions), env->host_scene.n_joints, m, e0, step_counter, (uint32_t)env->seed,
                (uint32_t)(env->seed >> 32));
            env->launches++;
            JA.random_actions = 0;
        }
        float* exec = env->d_exec + (size_t)e0 * env->host_scene.n_joints;
        int rc = gate_launch(env, buf_v, e0, m, chunk, env->gate_threshold, env->d_risk + e0, env->d_risky + e0,
                             env->d_backup + (size_t)e0 * MLP_MAX_OUT, exec, stream);
        if (rc) return rc;
        JA.exec = exec;
    }
    static const bool dbg_sync = getenv("SMENV_DEBUG_SYNC") != nullptr;  // locate a faulting kernel: sync after each
#define SM_MARK(i)                                                                                           \
    do {                                                                                                     \
        if (tk) cudaEventRecord(env->ev[i], stream);                                                         \
        if (dbg_sync) {                                                                                      \
            cudaError_t e_ = cudaStreamSynchronize(stream);                                                  \
            if (e_ != cudaSuccess)                                                                           \
                return fail(SM_ERR_CUDA, std::string("kernel before mark ") + std::to_string(i) + ": " +     \
                                             cudaGetErrorString(e_));                                        \
        }                                                                                                    \
    } while (0)
    auto robot_joint_heavy = [&](cudaStream_t st) {   // the lists are at most 8 m / 16 m long; blocks beyond their length exit at once
        int hb = (m * 8 + SM_HEAVY_THREADS - 1) / SM_HEAVY_THREADS;
        if (hb > 8 * env->sms) hb = 8 * env->sms;
        joint_first_kernel<<<hb, SM_HEAVY_THREADS, 0, st>>>(JA);
        joint_solve_kernel<<<16 * env->sms, SM_HEAVY_THREADS, 0, st>>>(JA);  // warps take chunks of the task list
        joint_final_kernel<<<hb, SM_HEAVY_THREADS, 0, st>>>(JA);
    };
    // Human scene: the robot's joint kernels do not depend on the nested env; outside the measurement modes they run on
    // the range's side stream next to the human's policy / range / braking check (latency-bound kernels that leave most
    // of the SMs' issue slots free) and join before the planning kernels
    static const bool no_joint_fork = getenv("SMENV_NO_JOINT_FORK") != nullptr;
    const bool joints_aside = env->human && !tk && !dbg_sync && !no_joint_fork;
    cudaStream_t jstream = env->side_streams[chunk];
    if (joints_aside) {
        CU(cudaEventRecord(env->joint_fork[chunk], stream));
        CU(cudaStreamWaitEvent(jstream, env->joint_fork[chunk], 0));
        joint_kernel<<<(m * 8 + 255) / 256, 256, 0, jstream>>>(JA);
        robot_joint_heavy(jstream);
    }
    HumanArgs HA;
    memset(&HA, 0, sizeof(HA));
    if (!env->human && tk)
        for (int i = SM_K_HUMAN_POLICY; i < SM_K_JOINT; ++i) cudaEventRecord(env->ev[i], stream);
    if (env->human) {
        // ---------------- the nested env of the human up to its setpoints (Human.step, ctlp.py:4818-4840)
        if (!buf->hkin || !buf->hstate || !buf->hbrake || !buf->hobs || !buf->hactions)
            return fail(SM_ERR_ARG, "smenv_step: the Human scene needs the hkin / hstate / hbrake / hobs / hactions buffers");
        HA.buf = *buf; HA.n = m; HA.env_base = e0;
        HA.k0 = (uint32_t)env->seed; HA.k1 = (uint32_t)(env->seed >> 32); HA.step_counter = step_counter;
        HA.step_ptr = step_ptr;   // host-buffer step: the counter lives in device memory (graph replays)
        HA.policy_out = env->d_hpolicy + (size_t)e0 * 16;
        HA.range = env->d_hrange + (size_t)e0 * 32;
        HA.bacc = env->d_hbacc + (size_t)e0 * SM_HBRAKE_STEPS * 8;
        HA.poses = env->d_hposes + (size_t)e0 * SM_HBRAKE_POSES * 8;
        HA.binfo = env->d_hbinfo + (size_t)e0 * 4;
        HA.units = env->d_hunits + (size_t)e0 * SM_HBRAKE_POSES + chunk;
        HA.hscratch = env->d_hscratch + (size_t)e0 * SM_SCRATCH_FLOATS;
        HA.scratch = scratch;
        HA.items = items; HA.item_count = worklist; HA.capacity = capacity; HA.overflow = worklist + 1;
        HA.res = res;
        HA.target_pool = env->pools_filled ? env->d_htarget_pool : nullptr;
        HA.target_pool_n = env->pools_filled ? env->htarget_pool_n : 0;
        HA.start_pool = env->pools_filled ? env->d_hstart_pool : nullptr;
        HA.pool_brake = env->pools_filled ? env->d_hpool_brake : nullptr; HA.pool_bcount = env->d_hpool_bcount;
        HA.start_pool_n = env->pools_filled ? env->start_pool_n : 0;
        HA.cwork = cwork;
        HA.counters = env->count ? env->d_counters : nullptr;
        SM_MARK(SM_K_HUMAN_POLICY);
        if (!env->human_external) {
            if (!env->net_loaded[SM_NET_HUMAN])
                return fail(SM_ERR_STATE, "smenv_step: load the human's policy (smenv_mlp_load, SM_NET_HUMAN) or supply its "
                                          "actions (smenv_set_human_actions_external)");
            int rcm = mlp_launch(env, SM_NET_HUMAN, MlpSeg{buf->hobs, SM_HOBS_STRIDE, env->nets[SM_NET_HUMAN].n_in},
                                 MlpSeg{nullptr, 0, 0}, MlpSeg{nullptr, 0, 0}, env->d_hpolicy + (size_t)e0 * 16, 16, m, stream);
            if (rcm) return rcm;
            human_action_kernel<<<(m * 8 + 255) / 256, 256, 0, stream>>>(HA);
            env->launches++;
        }
        JointArgs JH = JA;
        JH.set = 1; JH.nj = SM_HUMAN_JOINTS; JH.defer = 1; JH.range_out = HA.range; JH.random_actions = 0; JH.exec = nullptr;
        JH.track_vel = 0.87; JH.store_qset = 1; JH.keep_overflow = 0;
        JH.scratch = HA.hscratch;
        JH.clear_extra = HA.units;
        JH.worklist = worklist;
        JH.heavy = env->d_hheavy + (size_t)e0 * 8 + chunk;
        JH.tasks = env->d_htasks + (size_t)e0 * 16 + chunk;
        JH.hpar = env->d_hhpar + (size_t)e0 * 8 * SM_HPAR;
        JH.cwork = nullptr;
        const int hb = std::min((m * 8 + SM_HEAVY_THREADS - 1) / SM_HEAVY_THREADS, 8 * env->sms);
        SM_MARK(SM_K_HUMAN_JOINT);
        joint_kernel<<<(m * 8 + 255) / 256, 256, 0, stream>>>(JH);
        joint_first_kernel<<<hb, SM_HEAVY_THREADS, 0, stream>>>(JH);
        joint_solve_kernel<<<16 * env->sms, SM_HEAVY_THREADS, 0, stream>>>(JH);
        joint_final_kernel<<<hb, SM_HEAVY_THREADS, 0, stream>>>(JH);
        CU(cudaMemsetAsync(JH.heavy, 0, sizeof(int), stream));   // the human's deferred-joint list is empty for the next step
        SM_MARK(SM_K_HUMAN_BRAKE_TRAJ);
        human_brake_traj_kernel<<<(m * 8 + 127) / 128, 128, 0, stream>>>(HA);
        env->launches += 5;
        SM_MARK(SM_K_HUMAN_BRAKE_PLAN);
        if (env->host_scene.hu.check_braking) {
            human_brake_plan_kernel<<<env->grid_hplan, HBP_THREADS, env->smem_bytes_hplan, stream>>>(HA);
            SM_MARK(SM_K_HUMAN_BRAKE_GJK);
            GjkArgs GB;
            GB.items = items; GB.n_items = worklist; GB.capacity = capacity; GB.res = res; GB.counters = env->d_counters;
            launch_gjk(env, GB, stream);
            env->launches += 2;
        }
        else SM_MARK(SM_K_HUMAN_BRAKE_GJK);
        CU(cudaMemsetAsync(worklist, 0, sizeof(int), stream));   // the items of the braking check are consumed
        SM_MARK(SM_K_HUMAN_ADVANCE);
        human_advance_kernel<<<(m * 8 + 255) / 256, 256, 0, stream>>>(HA);
        env->launches++;
        CU(cudaGetLastError());
    }
    if (joints_aside) {   // the robot's joints are done before the planning kernels read its sub-step poses
        CU(cudaEventRecord(env->joint_join[chunk], jstream));
        CU(cudaStreamWaitEvent(stream, env->joint_join[chunk], 0));
    } else {
        SM_MARK(SM_K_JOINT);
        joint_kernel<<<(m * 8 + 255) / 256, 256, 0, stream>>>(JA);
        SM_MARK(SM_K_JOINT_HEAVY);
        robot_joint_heavy(stream);
    }
    env->launches += 4;
    PlanArgs P;
    P.buf = *buf; P.n = m; P.scratch = scratch;
    P.items = items; P.item_count = worklist; P.capacity = capacity;
    P.overflow = worklist + 1; P.res = res;
    P.kin = buf->kin; P.obst = buf->obst; P.advance = 1; P.counters = env->d_counters;
    P.cwork = cwork;
    P.target = buf->target;
    P.hkin = buf->hkin;
    GjkArgs G;
    G.items = items; G.n_items = worklist; G.capacity = capacity; G.res = res;
    G.counters = env->d_counters;
    StepArgs A;
    A.buf = *buf; A.n = m; A.auto_reset = auto_reset;
    A.k0 = (uint32_t)env->seed; A.k1 = (uint32_t)(env->seed >> 32);
    A.env_base = e0;
    A.scratch = scratch;
    A.res = res;
    A.heavy = heavy;
    A.overflow = worklist + 1;
    A.host_flag = env->d_flag;
    A.start_pool = env->pools_filled ? env->d_start_pool : nullptr;
    A.start_pool_n = env->pools_filled ? env->start_pool_n : 0;
    A.ball_pool = env->pools_filled ? env->d_ball_pool : nullptr;
    A.ball_pool_n = env->pools_filled ? env->ball_pool_n : 0;
    A.target_pool = env->pools_filled ? env->d_target_pool : nullptr;
    A.target_pool_n = env->pools_filled ? env->target_pool_n : 0;
    A.counters = env->d_counters;
    A.risk = gate ? env->d_risk + e0 : nullptr;
    A.risky = gate ? env->d_risky + e0 : nullptr;
    const int T = SM_WARPS_PER_BLOCK * 32;
    const int blocks = (m + SM_WARPS_PER_BLOCK - 1) / SM_WARPS_PER_BLOCK;
    const int grid_p = blocks < env->grid_broad ? blocks : env->grid_broad;
    const int grid_f = (m + SM_FINISH_ENVS_PER_BLOCK - 1) / SM_FINISH_ENVS_PER_BLOCK;
    const bool contacts = env->host_scene.contact_stride > 0 && env->host_scene.n_obstacles > 0;
    SM_MARK(SM_K_CONTACT_PLAN);
    // The contact planning and the distance planning are independent (both only append to the item list): outside the
    // measurement modes they run side by side, the contact kernels on the slot's side stream.
    static const bool no_fork = getenv("SMENV_NO_FORK") != nullptr;
    const bool fork = contacts && !tk && !dbg_sync && !no_fork;
    cudaStream_t cstream = stream;
    if (fork) {
        cstream = env->side_streams[chunk];
        CU(cudaEventRecord(env->side_fork[chunk], stream));
        CU(cudaStreamWaitEvent(cstream, env->side_fork[chunk], 0));
    }
    if (contacts && env->human) {
        const int grid_c = (m * SM_COARSE_LANES + 255) / 256;
        hcontact_coarse_kernel<<<grid_c, 256, sizeof(SceneSmem), cstream>>>(HA);
        hcontact_plan_kernel<<<grid_p, T, sizeof(SceneSmem), cstream>>>(HA);
    } else if (contacts) {
        const int grid_c = (m * SM_COARSE_LANES + 255) / 256;
        if (env->count) {
            contact_coarse_kernel<true><<<grid_c, 256, env->smem_bytes_broad, cstream>>>(P);
            contact_plan_kernel<true><<<grid_p, T, env->smem_bytes_broad, cstream>>>(P);
        } else {
            contact_coarse_kernel<false><<<grid_c, 256, env->smem_bytes_broad, cstream>>>(P);
            contact_plan_kernel<false><<<grid_p, T, env->smem_bytes_broad, cstream>>>(P);
        }
    }
    SM_MARK(SM_K_DISTANCE_PLAN);
    if (env->count) distance_plan_kernel<true><<<grid_p, T, env->smem_bytes_broad, stream>>>(P);
    else distance_plan_kernel<false><<<grid_p, T, env->smem_bytes_broad, stream>>>(P);
    if (fork) {
        CU(cudaEventRecord(env->side_join[chunk], cstream));
        CU(cudaStreamWaitEvent(stream, env->side_join[chunk], 0));
    }
    SM_MARK(SM_K_GJK);
    launch_gjk(env, G, stream);
    SM_MARK(SM_K_FINISH);
    if (env->count) finish_kernel<true><<<grid_f, 256, 0, stream>>>(A);
    else finish_kernel<false><<<grid_f, 256, 0, stream>>>(A);
    if (env->human && auto_reset && env->pools_filled) {   // the nested env restarts with the main env
        human_reset_kernel<<<(m * 8 + 255) / 256, 256, 0, stream>>>(HA, 1);
        env->launches++;
    }
    SM_MARK(SM_K_COUNT);
#undef SM_MARK
    env->launches += contacts ? 5 : 3;
    CU(cudaGetLastError());
    return SM_OK;
}

// The count of the deferred-joint list is cleared by the finish kernel of the previous step; when the number of ranges
// changes, the new count slots lie inside the old lists and have to be cleared once.
static int set_list_layout(SmEnv* env, int chunks, cudaStream_t stream) {
    if (env->list_layout == chunks) return SM_OK;
    const int per = (env->n + chunks - 1) / chunks;
    for (int c = 0; c < chunks && c * per < env->n; ++c)
        CU(cudaMemsetAsync(env->d_heavy + (size_t)c * per * 8 + c, 0, sizeof(int), stream));
    if (env->d_hheavy)
        for (int c = 0; c < chunks && c * per < env->n; ++c)
            CU(cudaMemsetAsync(env->d_hheavy + (size_t)c * per * 8 + c, 0, sizeof(int), stream));
    env->list_layout = chunks;
    return SM_OK;
}

static int ensure_chunk_streams(SmEnv* env) {
    if (env->chunk_streams[0]) return SM_OK;
    int pr_least = 0, pr_greatest = 0;
    CU(cudaDeviceGetStreamPriorityRange(&pr_least, &pr_greatest));
    for (int c = 0; c < SM_MAX_CHUNKS; ++c) {
        const int prio = pr_greatest + c < pr_least ? pr_greatest + c : pr_least;   // earlier ranges first
        CU(cudaStreamCreateWithPriority(&env->chunk_streams[c], cudaStreamNonBlocking, prio));
        CU(cudaEventCreateWithFlags(&env->chunk_done[c], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&env->chunk_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&env->host_order, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&env->host_stream, cudaStreamNonBlocking));
    return SM_OK;
}

static int step_check(SmEnv* env, const SmBuffers* buf, int auto_reset, bool need_actions) {
    if (!env || !buf) return fail(SM_ERR_ARG, "smenv_step: null argument");
    if (need_actions && !buf->actions) return fail(SM_ERR_ARG, "smenv_step: actions missing");
    if (auto_reset && !env->pools_filled) return fail(SM_ERR_STATE, "smenv_step: auto_reset needs smenv_fill_pools");
    if (env->h_flag && *(volatile int*)env->h_flag != 0)
        return fail(SM_ERR_STATE, "smenv_step: the GJK item buffer of an earlier step overflowed by " +
                                      std::to_string(*(volatile int*)env->h_flag) + " items (capacity " +
                                      std::to_string(env->item_capacity) + "); results since then are invalid");
    return SM_OK;
}

static int step_impl(SmEnv* env, const SmBuffers* buf, int auto_reset, int random_actions, SmStream s) {
    int rc = step_check(env, buf, auto_reset, !random_actions);
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); rc = activate(env, stream);
    if (rc) return rc;
    const bool tk = env->time_kernels;
    int ranges = tk ? 1 : env->step_ranges;
    if (ranges > SM_MAX_CHUNKS) ranges = SM_MAX_CHUNKS;
    if (ranges > env->n) ranges = env->n;
    if (ranges < 1) ranges = 1;
    rc = set_list_layout(env, ranges, stream);
    if (rc) return rc;
    const uint32_t counter = env->step_counter++;
    if (ranges == 1) {
        rc = step_range(env, buf, 0, env->n, 0, auto_reset, random_actions, counter, tk, stream);
        if (rc) return rc;
    } else {   // env ranges side by side on internal streams: the latency-bound tails of one range hide behind the other
        rc = ensure_chunk_streams(env);
        if (rc) return rc;
        CU(cudaEventRecord(env->chunk_fork, stream));
        const int per = (env->n + ranges - 1) / ranges;
        for (int c = 0; c < ranges; ++c) {
            const int e0 = c * per, m = e0 + per <= env->n ? per : env->n - e0;
            if (m <= 0) break;
            CU(cudaStreamWaitEvent(env->chunk_streams[c], env->chunk_fork, 0));
            rc = step_range(env, buf, e0, m, c, auto_reset, random_actions, counter, false, env->chunk_streams[c]);
            if (rc) return rc;
            CU(cudaEventRecord(env->chunk_done[c], env->chunk_streams[c]));
            CU(cudaStreamWaitEvent(stream, env->chunk_done[c], 0));
        }
    }
    if (tk) {
        CU(cudaStreamSynchronize(stream));
        for (int i = 0; i < SM_K_COUNT; ++i) {
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, env->ev[i], env->ev[i + 1]));
            env->kernel_ms[i] += ms;
        }
        env->timed_steps++;
    }
    return SM_OK;
}

// Host-buffer step (the call an RL sampler makes): the envs are cut into `chunks` ranges, each on its own stream:
// actions host -> device, the step's kernels, observation / reward / done device -> host.  The copies of one range
// overlap the kernels of the others (the two copy engines and the SMs work at the same time), so the PCIe time hides
// behind the compute instead of adding to it.  The whole fork / join (chunks x (4 copies + 11 kernels)) is captured
// once into a CUDA graph and replayed with one launch per step: issued call by call it is bound by the host's launch
// rate.  Returns when the host buffers are complete.
struct HostStepKey {
    SmBuffers buf;
    const void* h[4];
    int auto_reset, chunks, count, pools, human_external, gate_exact;
    float gate, gate_band;
};

static int host_step_enqueue(SmEnv* env, const SmBuffers* buf, const float* h_actions, float* h_obs, float* h_reward,
                             uint8_t* h_done, int auto_reset, int chunks, uint32_t counter, cudaStream_t origin) {
    const int nj = env->host_scene.n_joints, od = env->host_scene.obs_size;
    // the step counter (Philox stream of the human's policy noise): copied from the pinned word the caller just set
    CU(cudaMemcpyAsync(env->d_step, env->h_step, sizeof(uint32_t), cudaMemcpyHostToDevice, origin));
    CU(cudaEventRecord(env->chunk_fork, origin));
    const int per = (env->n + chunks - 1) / chunks;
    for (int c = 0; c < chunks; ++c) {
        const int e0 = c * per, m = e0 + per <= env->n ? per : env->n - e0;
        if (m <= 0) break;
        cudaStream_t cs = env->chunk_streams[c];
        CU(cudaStreamWaitEvent(cs, env->chunk_fork, 0));
        // Human scene without the gate: only the robot's joint kernels read the actions, and they run on the range's side
        // stream (step_range): the copy goes there too, the nested env's chain starts without waiting for it
        static const bool no_joint_fork = getenv("SMENV_NO_JOINT_FORK") != nullptr || getenv("SMENV_DEBUG_SYNC") != nullptr;
        const bool copy_aside = env->human && env->gate_threshold < 0.0f && !no_joint_fork;
        cudaStream_t hs = cs;
        if (copy_aside) {
            hs = env->side_streams[c];
            CU(cudaStreamWaitEvent(hs, env->chunk_fork, 0));
        }
        CU(cudaMemcpyAsync((float*)buf->actions + (size_t)e0 * nj, h_actions + (size_t)e0 * nj,
                           (size_t)m * nj * sizeof(float), cudaMemcpyHostToDevice, hs));
        int rc = step_range(env, buf, e0, m, c, auto_reset, 0, counter, false, cs, env->d_step);
        if (rc) return rc;
        CU(cudaMemcpyAsync(h_obs + (size_t)e0 * od, buf->obs + (size_t)e0 * od, (size_t)m * od * sizeof(float),
                           cudaMemcpyDeviceToHost, cs));
        CU(cudaMemcpyAsync(h_reward + e0, buf->reward + e0, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost, cs));
        CU(cudaMemcpyAsync(h_done + e0, buf->done + e0, (size_t)m, cudaMemcpyDeviceToHost, cs));
        CU(cudaEventRecord(env->chunk_done[c], cs));
        CU(cudaStreamWaitEvent(origin, env->chunk_done[c], 0));
    }
    return SM_OK;
}

extern "C" int smenv_step_host(SmEnv* env, const SmBuffers* buf, const float* h_actions, float* h_obs, float* h_reward,
                               uint8_t* h_done, int auto_reset, int chunks, SmStream s) {
    int rc = step_check(env, buf, auto_reset, true);
    if (rc) return rc;
    if (!h_actions || !h_obs || !h_reward || !h_done || !buf->obs || !buf->reward || !buf->done)
        return fail(SM_ERR_ARG, "smenv_step_host: null host or device buffer");
    if (chunks < 1) chunks = 1;
    if (chunks > SM_MAX_CHUNKS) chunks = SM_MAX_CHUNKS;
    if (chunks > env->n) chunks = env->n;
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); rc = activate(env, stream);
    if (rc) return rc;
    rc = ensure_chunk_streams(env);
    if (rc) return rc;
    const uint32_t counter = env->step_counter++;
    CU(cudaStreamSynchronize(env->host_stream));   // the previous host step has read the pinned counter word (it returned
    *env->h_step = counter;                         // synchronised; a no-op in practice)
    rc = set_list_layout(env, chunks, stream);
    if (rc) return rc;
    // the internal origin stream comes after the work already queued on the caller's stream
    CU(cudaEventRecord(env->host_order, stream));
    CU(cudaStreamWaitEvent(env->host_stream, env->host_order, 0));
    static const bool no_graph = getenv("SMENV_DEBUG_SYNC") != nullptr || getenv("SMENV_NO_GRAPH") != nullptr;
    if (no_graph) {
        rc = host_step_enqueue(env, buf, h_actions, h_obs, h_reward, h_done, auto_reset, chunks, counter, env->host_stream);
        if (rc) return rc;
        CU(cudaStreamSynchronize(env->host_stream));
        return SM_OK;
    }
    static_assert(sizeof(HostStepKey) <= sizeof(env->host_graph_key), "host_graph_key too small");
    HostStepKey key;
    memset(&key, 0, sizeof(key));
    key.buf = *buf;
    key.h[0] = h_actions; key.h[1] = h_obs; key.h[2] = h_reward; key.h[3] = h_done;
    key.auto_reset = auto_reset; key.chunks = chunks; key.count = env->count ? 1 : 0; key.pools = env->pools_filled ? 1 : 0; key.gate = env->gate_threshold;
    key.human_external = env->human_external ? 1 : 0; key.gate_exact = env->gate_exact ? 1 : 0; key.gate_band = env->gate_band;
    if (!env->host_graph || memcmp(&key, env->host_graph_key, sizeof(key)) != 0) {
        if (env->host_graph) { cudaGraphExecDestroy(env->host_graph); env->host_graph = nullptr; }
        const unsigned long long launches0 = env->launches;
        CU(cudaStreamBeginCapture(env->host_stream, cudaStreamCaptureModeThreadLocal));
        rc = host_step_enqueue(env, buf, h_actions, h_obs, h_reward, h_done, auto_reset, chunks, counter, env->host_stream);
        cudaGraph_t graph = nullptr;
        cudaError_t ce = cudaStreamEndCapture(env->host_stream, &graph);
        env->host_graph_kernels = (int)(env->launches - launches0);
        env->launches = launches0;
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess) return fail(SM_ERR_CUDA, std::string("smenv_step_host: graph capture: ") + cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(&env->host_graph, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) {
            env->host_graph = nullptr;
            return fail(SM_ERR_CUDA, std::string("smenv_step_host: graph instantiate: ") + cudaGetErrorString(ce));
        }
        memcpy(env->host_graph_key, &key, sizeof(key));
    }
    CU(cudaGraphLaunch(env->host_graph, env->host_stream));
    env->launches += env->host_graph_kernels;
    CU(cudaStreamSynchronize(env->host_stream));
    return SM_OK;
}
extern "C" int smenv_set_step_ranges(SmEnv* env, int ranges) {
    if (!env) return fail(SM_ERR_ARG, "smenv_set_step_ranges: null env");
    if (ranges < 1 || ranges > SM_MAX_CHUNKS) return fail(SM_ERR_ARG, "smenv_set_step_ranges: 1..8 ranges");
    env->step_ranges = ranges;
    return SM_OK;
}
extern "C" int smenv_step(SmEnv* env, const SmBuffers* buf, int auto_reset, SmStream s) {
    return step_impl(env, buf, auto_reset, 0, s);
}
extern "C" int smenv_step_random(SmEnv* env, const SmBuffers* buf, int auto_reset, SmStream s) {
    return step_impl(env, buf, auto_reset, 1, s);
}

extern "C" int smenv_safe_range(SmEnv* env, const double* kin, double* lo, double* hi, int32_t* code, int n, SmStream s) {
    if (!env || !kin || !lo || !hi || !code) return fail(SM_ERR_ARG, "smenv_safe_range: null argument");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    safe_range_kernel<<<(n * 8 + 127) / 128, 128, 0, stream>>>(kin, lo, hi, code, n);
    env->launches++;
    CU(cudaGetLastError());
    return SM_OK;
}

extern "C" int smenv_distances(SmEnv* env, const double* kin, const double* obst, const double* hkin, float* d_static,
                               float* d_self, float* d_moving, int n, SmStream s) {
    if (!env || !kin || !obst || !d_static || !d_self || !d_moving) return fail(SM_ERR_ARG, "smenv_distances: null argument");
    if (n > env->n) return fail(SM_ERR_ARG, "smenv_distances: n exceeds the env count the buffers were sized for");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    // the same kernels as the step: plan the pair queries of the given poses, run them, decode the result records
    CU(cudaMemsetAsync(env->d_worklist, 0, 2 * sizeof(int), stream));
    PlanArgs P;
    memset(&P, 0, sizeof(P));
    P.n = n; P.scratch = env->d_scratch;
    P.items = env->d_items; P.item_count = env->d_worklist; P.capacity = env->item_capacity;
    P.overflow = env->d_worklist + 1; P.res = env->d_res;
    P.kin = kin; P.obst = obst; P.advance = 0; P.counters = env->d_counters;
    P.hkin = hkin;
    if (env->human && !hkin) return fail(SM_ERR_ARG, "smenv_distances: the Human scene needs the human's joint state");
    GjkArgs G;
    G.items = env->d_items; G.n_items = env->d_worklist; G.capacity = env->item_capacity; G.res = env->d_res;
    G.counters = env->d_counters;
    const int T = SM_WARPS_PER_BLOCK * 32;
    const int blocks = (n + SM_WARPS_PER_BLOCK - 1) / SM_WARPS_PER_BLOCK;
    const int grid_p = blocks < env->grid_broad ? blocks : env->grid_broad;
    distance_plan_kernel<false><<<grid_p, T, env->smem_bytes_broad, stream>>>(P);
    launch_gjk(env, G, stream);
    distances_out_kernel<<<(n + 255) / 256, 256, 0, stream>>>(env->d_res, obst, d_static, d_self, d_moving, n);
    env->launches += 3;
    CU(cudaGetLastError());
    return SM_OK;
}

extern "C" int smenv_enable_counters(SmEnv* env, int enable) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    env->count = enable != 0;
    return SM_OK;
}
extern "C" int smenv_counters(SmEnv* env, SmCounters* out, int reset) {
    if (!env || !out) return fail(SM_ERR_ARG, "null argument");
    CU(cudaSetDevice(env->device));
    unsigned long long h[24];
    CU(cudaMemcpy(h, env->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
    out->gjk_calls = h[0]; out->gjk_iters = h[1]; out->support_dots = h[2]; out->distance_items = h[3];
    out->env_steps = h[4]; out->contact_envs = h[5]; out->contact_items = h[6]; out->reserved = h[7];
    out->heavy_joints = h[8]; out->heavy_solves = h[9];
    for (int i = 0; i < 6; ++i) out->aux[i] = h[10 + i];
    out->brake_poses = h[16]; out->brake_pair_bounds = h[17];
    if (reset) CU(cudaMemset(env->d_counters, 0, sizeof(h)));
    return SM_OK;
}
// ------------------------------------------------------------------------------------------------------------------
// networks (smenv_mlp.cuh)
// ------------------------------------------------------------------------------------------------------------------
extern "C" int smenv_mlp_load(SmEnv* env, int which, int n_tc, const int32_t* dims, int hidden_act, int out_act,
                              const float* weights) {
    if (!env || !dims || !weights || which < 0 || which >= SM_NET_COUNT) return fail(SM_ERR_ARG, "smenv_mlp_load: bad argument");
    if (n_tc < 1 || n_tc > MLP_MAX_TC) return fail(SM_ERR_ARG, "smenv_mlp_load: 1..3 hidden layers are supported");
    const int n_in = dims[0], n_out = dims[n_tc + 1];
    const int k_in = n_in <= 16 ? 16 : n_in <= 32 ? 32 : 64;   // a power of two: divisible by every chunk width
    if (n_in < 1 || n_in > 64) return fail(SM_ERR_ARG, "smenv_mlp_load: input width must be in 1..64");
    if (n_out < 1 || n_out > MLP_MAX_OUT) return fail(SM_ERR_ARG, "smenv_mlp_load: output width must be in 1..16");
    const int out_pad = n_out <= 8 ? 8 : 16;
    if (dims[n_tc] * out_pad > MLP_WOUT_FLOATS)
        return fail(SM_ERR_ARG, "smenv_mlp_load: last hidden width x padded output width exceeds 2048");
    for (int l = 0; l < n_tc; ++l) {
        const int N = dims[1 + l];
        // a layer's width is the K of the next one, streamed in chunks of 64 columns: 16, 32, 48 or a multiple of 64
        if (N % 16 != 0 || N < 16 || (N > 64 && N % 64 != 0) || (N > 256 && N != 512))
            return fail(SM_ERR_ARG, "smenv_mlp_load: hidden widths must be 16, 32, 48, 64, 128, 192, 256 or 512");
    }
    if (dims[n_tc] > MLP_MAX_LAST) return fail(SM_ERR_ARG, "smenv_mlp_load: the last hidden layer may be at most 256 wide");
    CU(cudaSetDevice(env->device));
    MlpNet net;
    memset(&net, 0, sizeof(net));
    net.n_tc = n_tc; net.n_in = n_in; net.k_in = k_in; net.hidden_act = hidden_act; net.out_act = out_act; net.n_out = n_out; net.out_pad = out_pad;
    const float* wp = weights;
    int K_real = n_in, Kp = k_in;
    for (int l = 0; l < n_tc; ++l) {
        const int N = dims[1 + l];
        net.dims[l] = N;
        const int chunk_k = mlp_chunk_k(N, Kp);
        std::vector<__half> packed((size_t)N * Kp);
        for (int k = 0; k < Kp; ++k)
            for (int n = 0; n < N; ++n) {
                const int c = k / chunk_k, kl = k % chunk_k;
                const size_t off = (size_t)c * N * chunk_k * 2 + (size_t)(kl / 8) * (N / 8 * 128) + (size_t)(n / 8) * 128 +
                                   (size_t)(n % 8) * 16 + (size_t)(kl % 8) * 2;
                packed[off / 2] = __float2half_rn(k < K_real ? wp[(size_t)k * N + n] : 0.0f);
            }
        {   // float32 copy of the kernel for the exact evaluation of single rows
            float* dw32 = nullptr;
            CU(cudaMalloc((void**)&dw32, (size_t)K_real * N * sizeof(float)));
            env->net_allocs.push_back(dw32);
            CU(cudaMemcpy(dw32, wp, (size_t)K_real * N * sizeof(float), cudaMemcpyHostToDevice));
            net.w32[l] = dw32;
        }
        wp += (size_t)K_real * N;
        __half* dw = nullptr;
        float* db = nullptr;
        CU(cudaMalloc((void**)&dw, packed.size() * sizeof(__half)));
        env->net_allocs.push_back(dw);
        CU(cudaMemcpy(dw, packed.data(), packed.size() * sizeof(__half), cudaMemcpyHostToDevice));
        CU(cudaMalloc((void**)&db, N * sizeof(float)));
        env->net_allocs.push_back(db);
        CU(cudaMemcpy(db, wp, N * sizeof(float), cudaMemcpyHostToDevice));
        wp += N;
        net.w[l] = dw; net.b[l] = db;
        K_real = N; Kp = N;
    }
    {   // output layer, padded to out_pad columns
        std::vector<float> wo((size_t)K_real * out_pad, 0.0f), bo(out_pad, 0.0f);
        for (int k = 0; k < K_real; ++k)
            for (int o = 0; o < n_out; ++o) wo[(size_t)k * out_pad + o] = wp[(size_t)k * n_out + o];
        wp += (size_t)K_real * n_out;
        for (int o = 0; o < n_out; ++o) bo[o] = wp[o];
        float *dwo = nullptr, *dbo = nullptr;
        CU(cudaMalloc((void**)&dwo, wo.size() * sizeof(float)));
        env->net_allocs.push_back(dwo);
        CU(cudaMemcpy(dwo, wo.data(), wo.size() * sizeof(float), cudaMemcpyHostToDevice));
        CU(cudaMalloc((void**)&dbo, bo.size() * sizeof(float)));
        env->net_allocs.push_back(dbo);
        CU(cudaMemcpy(dbo, bo.data(), bo.size() * sizeof(float), cudaMemcpyHostToDevice));
        net.w_out = dwo; net.b_out = dbo;
    }
    env->nets[which] = net;
    env->net_loaded[which] = true;
    if (!env->d_risk) {
        CU(cudaMalloc((void**)&env->d_risk, (size_t)env->n * sizeof(float)));
        CU(cudaMalloc((void**)&env->d_backup, (size_t)env->n * MLP_MAX_OUT * sizeof(float)));
        CU(cudaMalloc((void**)&env->d_exec, (size_t)env->n * SM_MAX_JOINTS * sizeof(float)));
        CU(cudaMalloc((void**)&env->d_risky, (size_t)env->n));
        CU(cudaMemset(env->d_risky, 0, (size_t)env->n));
        CU(cudaMalloc((void**)&env->d_gate_list, ((size_t)env->n * 2 + 32) * sizeof(int)));
        CU(cudaMemset(env->d_gate_list, 0, ((size_t)env->n * 2 + 32) * sizeof(int)));
    }
    CU(cudaFuncSetAttribute(mlp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MLP_SM_BYTES));
    CU(cudaFuncSetAttribute(mlp_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MLP_EXACT_SMEM));
    return SM_OK;
}

extern "C" int smenv_mlp_forward(SmEnv* env, int which, const float* in0, int in0_w, const float* in1, int in1_w,
                                 float* out, int out_stride, int n, SmStream s) {
    if (!env || !in0 || !out || which < 0 || which >= SM_NET_COUNT || n <= 0) return fail(SM_ERR_ARG, "smenv_mlp_forward: bad argument");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    return mlp_launch(env, which, MlpSeg{in0, in0_w, in0_w}, MlpSeg{in1, in1 ? in1_w : 0, in1 ? in1_w : 0},
                      MlpSeg{nullptr, 0, 0}, out, out_stride, n, stream);
}

extern "C" int smenv_risk_gate(SmEnv* env, const SmBuffers* buf, float threshold, float* risk_out, uint8_t* risky_out,
                               SmStream s) {
    if (!env || !buf || !buf->actions || !buf->obs) return fail(SM_ERR_ARG, "smenv_risk_gate: null argument");
    if (!env->net_loaded[0] || !env->net_loaded[1]) return fail(SM_ERR_STATE, "smenv_risk_gate: load both networks first");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    return gate_launch(env, *buf, 0, env->n, 0, threshold, risk_out ? risk_out : env->d_risk, risky_out ? risky_out : env->d_risky,
                       env->d_backup, const_cast<float*>(buf->actions), stream);
}

extern "C" int smenv_set_risk_gate(SmEnv* env, float threshold) {
    if (!env) return fail(SM_ERR_ARG, "smenv_set_risk_gate: null env");
    if (threshold >= 0.0f && (!env->net_loaded[0] || !env->net_loaded[1]))
        return fail(SM_ERR_STATE, "smenv_set_risk_gate: load the risk network and the backup policy first (smenv_mlp_load)");
    env->gate_threshold = threshold >= 0.0f ? threshold : -1.0f;
    return SM_OK;
}

extern "C" int smenv_set_gate_exact(SmEnv* env, int exact, float band) {
    if (!env) return fail(SM_ERR_ARG, "smenv_set_gate_exact: null env");
    env->gate_exact = exact != 0;
    if (band > 0.0f) env->gate_band = band;
    if (env->host_graph) { cudaGraphExecDestroy(env->host_graph); env->host_graph = nullptr; }
    return SM_OK;
}

extern "C" int smenv_mlp_forward_exact(SmEnv* env, int which, const float* in0, int in0_w, const float* in1, int in1_w,
                                       float* out, int out_stride, int n_out, int n, SmStream s) {
    if (!env || !in0 || !out || which < 0 || which >= SM_NET_COUNT || n <= 0) return fail(SM_ERR_ARG, "smenv_mlp_forward_exact: bad argument");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    if (in0_w + (in1 ? in1_w : 0) != env->nets[which].n_in) return fail(SM_ERR_ARG, "network input width does not match the loaded weights");
    return mlp_exact_launch(env, which, MlpSeg{in0, in0_w, in0_w}, MlpSeg{in1, in1 ? in1_w : 0, in1 ? in1_w : 0},
                            MlpSeg{nullptr, 0, 0}, nullptr, nullptr, n, out, out_stride, n_out, stream);
}

extern "C" int smenv_set_seed(SmEnv* env, uint64_t seed) {
    if (!env) return fail(SM_ERR_ARG, "smenv_set_seed: null env");
    env->seed = seed;
    env->step_counter = 0;
    if (env->host_graph) { cudaGraphExecDestroy(env->host_graph); env->host_graph = nullptr; }   // the key is baked in
    return SM_OK;
}

extern "C" int smenv_random_actions(SmEnv* env, const SmBuffers* buf, SmStream s) {
    if (!env || !buf || !buf->actions) return fail(SM_ERR_ARG, "smenv_random_actions: null argument");
    cudaStream_t stream = (cudaStream_t)s;
    DevLock dev_lock_(env); int rc = activate(env, stream);
    if (rc) return rc;
    const int nj = env->host_scene.n_joints;
    random_actions_kernel<<<(env->n * nj + 255) / 256, 256, 0, stream>>>(const_cast<float*>(buf->actions), nj, env->n, 0,
                                                                         env->step_counter, (uint32_t)env->seed,
                                                                         (uint32_t)(env->seed >> 32));
    env->launches++;
    CU(cudaGetLastError());
    return SM_OK;
}

extern "C" int smenv_kernel_timing(SmEnv* env, int enable) {
    if (!env) return fail(SM_ERR_ARG, "null env");
    CU(cudaSetDevice(env->device));
    if (enable && !env->ev[0])
        for (int i = 0; i <= SM_K_COUNT; ++i) CU(cudaEventCreate(&env->ev[i]));
    env->time_kernels = enable != 0;
    return SM_OK;
}
extern "C" int smenv_kernel_times(SmEnv* env, double* ms_out, int* steps_out, int reset) {
    if (!env || !ms_out || !steps_out) return fail(SM_ERR_ARG, "null argument");
    for (int i = 0; i < SM_K_COUNT; ++i) ms_out[i] = env->kernel_ms[i];
    *steps_out = env->timed_steps;
    if (reset) {
        for (int i = 0; i < SM_K_COUNT; ++i) env->kernel_ms[i] = 0.0;
        env->timed_steps = 0;
    }
    return SM_OK;
}
extern "C" int smenv_launch_config(SmEnv* env, int32_t* out) {
    if (!env || !out) return fail(SM_ERR_ARG, "null argument");
    out[0] = env->grid_gjk; out[1] = env->gjk_threads; out[2] = (int32_t)env->smem_bytes_gjk; out[3] = env->host_scene.n_lut_words;
    out[4] = env->grid_broad; out[5] = (int32_t)env->smem_bytes_broad; out[6] = env->sms; out[7] = env->step_ranges;
    return SM_OK;
}
extern "C" int smenv_launch_count(SmEnv* env, unsigned long long* out) {
    if (!env || !out) return fail(SM_ERR_ARG, "null argument");
    *out = env->launches;
    return SM_OK;
}

// debug: trace one GJK call on the device (not part of the product path; used by tools/ and tests to explain parity)
extern "C" int smenv_debug_build_lut(const float* xyz, int n, int res, uint32_t* out, int capacity) {
    if (!xyz || n < 1 || n > 255) return fail(SM_ERR_ARG, "smenv_debug_build_lut: 1 .. 255 vertices");
    if (res != 4 && res != 8 && res != 12 && res != 16) return fail(SM_ERR_ARG, "smenv_debug_build_lut: res is 4, 8, 12 or 16");
    std::vector<float4> v(n);
    for (int i = 0; i < n; ++i) v[i] = make_float4(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], 0.f);
    std::vector<uint32_t> t;
    build_lut(v.data(), n, res, t);
    if (out) {
        if ((int)t.size() > capacity) return fail(SM_ERR_ARG, "smenv_debug_build_lut: buffer too small");
        memcpy(out, t.data(), t.size() * sizeof(uint32_t));
    }
    return (int)t.size();
}
extern "C" int smenv_debug_lut_cell(float dx, float dy, float dz, int res) { return lut_cell_res(dx, dy, dz, res); }

static_assert(SM_PLAN_HWIDTH_CELLS == 6 * SM_LUT_RES * SM_LUT_RES, "SmPlanBounds.hwidth holds one table per shape");
static_assert(SM_PLAN_MAX_PAIRS == SM_MAX_PLAN_PAIRS, "SmPlanBounds.pair_tab holds the whole pair table");
extern "C" int smenv_debug_plan_bounds(const SmScene* sc, SmPlanBounds* out) {
    if (!sc || !out) return fail(SM_ERR_ARG, "null argument");
    if (sc->n_shapes > SM_MAX_SHAPES || sc->n_verts <= 0) return fail(SM_ERR_SCENE, "bad shape table");
    std::vector<float4> verts(sc->n_verts);
    for (int i = 0; i < sc->n_verts; ++i)
        verts[i] = make_float4((float)sc->verts[3 * i], (float)sc->verts[3 * i + 1], (float)sc->verts[3 * i + 2], 0.f);
    std::vector<DevScene> dv(1);
    DevScene& d = dv[0];
    memset(&d, 0, sizeof(d));
    std::vector<float> hwidth;
    if (const int rc = plan_bounds(sc, verts, d, hwidth)) return rc;
    memset(out, 0, sizeof(*out));
    out->n_shapes = sc->n_shapes; out->n_pairs_fixed = d.n_pairs_fixed; out->n_pairs = d.n_pairs;
    out->self_query = d.self_query;
    for (int s = 0; s < sc->n_shapes; ++s) {
        const DevShape& g = d.shapes[s];
        out->center[s][0] = g.cx; out->center[s][1] = g.cy; out->center[s][2] = g.cz; out->radius[s] = g.radius;
        out->centroid[s][0] = g.gx; out->centroid[s][1] = g.gy; out->centroid[s][2] = g.gz;
        for (int k = 0; k < 3; ++k) { out->bmin[s][k] = g.bmin[k]; out->bmax[s][k] = g.bmax[k]; }
        memcpy(out->hwidth[s], hwidth.data() + g.hw, sizeof(out->hwidth[s]));
    }
    for (int p = 0; p < d.n_pairs; ++p) { out->pair_tab[p] = d.pair_tab[p]; out->pair_rm[p][0] = d.pair_rm[p].x; out->pair_rm[p][1] = d.pair_rm[p].y; }
    return SM_OK;
}

extern "C" int smenv_debug_human_bounds(const SmScene* sc, SmHumanBounds* out) {
    if (!sc || !out) return fail(SM_ERR_ARG, "null argument");
    if (!sc->human.enabled) return fail(SM_ERR_ARG, "smenv_debug_human_bounds: the scene has no human");
    DevHuman u;
    memset(&u, 0, sizeof(u));
    std::vector<short> hpairs;
    if (const int rc = human_brake_bounds(sc, u, hpairs)) return rc;
    memset(out, 0, sizeof(*out));
    out->n_gp = u.n_gp;
    for (int g = 0; g < 8; ++g) {
        out->gp_fa[g] = u.gp_fa[g]; out->gp_fb[g] = u.gp_fb[g];
        out->gp_a0[g] = u.gp_a0[g]; out->gp_na[g] = u.gp_na[g]; out->gp_b0[g] = u.gp_b0[g]; out->gp_nb[g] = u.gp_nb[g];
        out->gp_ra[g] = u.gp_ra[g]; out->gp_rb[g] = u.gp_rb[g]; out->gp_sra[g] = u.gp_sra[g]; out->gp_srb[g] = u.gp_srb[g];
        for (int k = 0; k < 3; ++k) {
            out->gp_ca[g][k] = u.gp_ca[g][k]; out->gp_cb[g][k] = u.gp_cb[g][k];
            out->gp_bmin[g][k] = u.gp_bmin[g][k]; out->gp_bmax[g][k] = u.gp_bmax[g][k];
        }
        for (int k = 0; k < 6; ++k) { out->gp_sa[g][k] = u.gp_sa[g][k]; out->gp_sb[g][k] = u.gp_sb[g][k]; }
    }
    for (int fi = 0; fi < 4; ++fi) {
        out->hf_s0[fi] = u.hf_s0[fi]; out->hf_sn[fi] = u.hf_sn[fi]; out->hf_rad[fi] = u.hf_rad[fi];
        for (int k = 0; k < 6; ++k) out->hf_seg[fi][k] = u.hf_seg[fi][k];
        const float* s = u.hf_seg[fi];
        const float dx = s[3] - s[0], dy = s[4] - s[1], dz = s[5] - s[2];
        out->hf_cover_rad[fi] = table_cover_radius(u.hf_rad[fi], sqrtf(dx * dx + dy * dy + dz * dz));
    }
    return SM_OK;
}

extern "C" int smenv_debug_gjk(SmEnv* env, const double* kin_host, const double* obst_host, int ia, int ib, float upper,
                               float* trace_host /* 32 x 8 */, float* result_host /* 4 + 12 * 9 */) {
    if (!env || !kin_host || !obst_host || !trace_host || !result_host) return fail(SM_ERR_ARG, "null argument");
    DevLock dev_lock_(env); int rc = activate(env, 0);
    if (rc) return rc;
    double *dk, *dob; float *dt, *dr;
    CU(cudaMalloc((void**)&dk, 32 * 8)); CU(cudaMalloc((void**)&dob, 16 * 8));
    CU(cudaMalloc((void**)&dt, 256 * 4)); CU(cudaMalloc((void**)&dr, 128 * 4));
    CU(cudaMemcpy(dk, kin_host, 32 * 8, cudaMemcpyHostToDevice)); CU(cudaMemcpy(dob, obst_host, 16 * 8, cudaMemcpyHostToDevice));
    CU(cudaMemset(dt, 0, 256 * 4)); CU(cudaMemset(dr, 0, 128 * 4));
    debug_gjk_kernel<<<1, 32, env->smem_bytes, 0>>>(dk, dob, ia, ib, upper, dt, dr);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(trace_host, dt, 256 * 4, cudaMemcpyDeviceToHost)); CU(cudaMemcpy(result_host, dr, 128 * 4, cudaMemcpyDeviceToHost));
    cudaFree(dk); cudaFree(dob); cudaFree(dt); cudaFree(dr);
    return SM_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// measured peaks of the vector pipes (bench.py's roofline denominators): dependent-free FMA chains, 8 accumulators per
// thread, all SMs filled; flops = 2 per FMA
// ------------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T a, T b) {
    T x0 = (T)threadIdx.x, x1 = x0 + (T)1, x2 = x0 + (T)2, x3 = x0 + (T)3, x4 = x0 + (T)4, x5 = x0 + (T)5, x6 = x0 + (T)6, x7 = x0 + (T)7;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
            x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

template <typename T>
static int measure_fma(int sms, int iters, double* tflops) {
    const int blocks = sms * 8, threads = 256;
    T* d = nullptr;
    CU(cudaMalloc((void**)&d, (size_t)blocks * threads * sizeof(T)));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    fma_peak_kernel<T><<<blocks, threads>>>(d, iters / 8, (T)0.999, (T)0.001);   // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0));
        fma_peak_kernel<T><<<blocks, threads>>>(d, iters, (T)0.999, (T)0.001);
        CU(cudaEventRecord(e1));
        CU(cudaEventSynchronize(e1));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 64.0 * (double)iters * (double)blocks * threads;
        if (ms > 0.f && fl / (ms * 1e-3) / 1e12 > best) best = fl / (ms * 1e-3) / 1e12;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d);
    *tflops = best;
    return SM_OK;
}

extern "C" int smenv_measure_fma_peaks(int device, double* tflops_fp32, double* tflops_fp64) {
    if (!tflops_fp32 || !tflops_fp64) return fail(SM_ERR_ARG, "smenv_measure_fma_peaks: null argument");
    CU(cudaSetDevice(device));
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    int rc = measure_fma<float>(sms, 4096, tflops_fp32);
    if (rc) return rc;
    return measure_fma<double>(sms, 1024, tflops_fp64);
}
