// C ABI of libmppi_b200.so (include/mppi_b200.h): handle management, launch orchestration,
// strict-mode multi-pass driver, NCCL sample sharding.  Host code only; kernels live in
// mppi_kernels.cu / mppi_mlp.cu.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mppi_device.cuh"
#include "mppi_launch.h"
#include "mppi_mlp.h"

namespace {

struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool load() {
        if (lib) return true;
        // Reuse the copy torch already mapped when there is one (same soname), else the system one.
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return false;
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && AllGather && CommDestroy && GetErrorString;
    }
};
NcclApi g_nccl;

}  // namespace

struct mppi_handle_s {
    mppi_config_t cfg{};
    TickArgs args{};
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int n_sm = 148, occ = 1, nx = 3;
    int grid_x = 1, grid_x_stash = 1;    // CTAs per robot: regenerate-noise kernels / stash kernels
    bool stash = false;                  // Philox ticks keep the chunk's noise in shared memory
    bool tpar = false;                   // ... and small sample counts run the horizon time-parallel (rollout_tpar), on grid_x_tpar CTAs
    int grid_x_tpar = 1;
    bool sum = false, strict = false;
    bool have_path = false;
    std::vector<double> path_h;          // host copy for the strict-mode step 1 (literal FP64)
    int n_path = 0, path_cols = 0;
    // device buffers
    float4 *d_path = nullptr;
    float *d_U = nullptr, *d_M = nullptr, *d_S = nullptr, *d_part = nullptr, *d_out = nullptr;
    float *d_x0 = nullptr, *d_opt = nullptr, *d_plant_log = nullptr;
    int plant_log_cap = 0;
    unsigned *d_loop = nullptr;                 // closed loop: running tick, first tick, ticket (see TickArgs::loop_state)
    cudaGraphExec_t loop_graph = nullptr;       // the n-tick closed loop, instantiated once per (n_ticks, arguments)
    cudaStream_t cap_stream = nullptr;          // private stream the loop is captured on
    int loop_graph_n = 0;
    TickArgs loop_graph_args{};
    int *d_idx = nullptr, *d_NC = nullptr;
    unsigned *d_ticket = nullptr;
    float *h_out = nullptr, *h_out_dev = nullptr;     // mapped pinned record of robot 0
    // strict mode
    unsigned *d_bp_n = nullptr;
    int *d_bp_s = nullptr;
    unsigned long long *d_first = nullptr, *h_first = nullptr;
    // strict mode, host side of a pass: [first-change word][breakpoint sample-steps][breakpoint indices] staged in pinned memory and
    // sent as ONE copy (d_first / d_bp_n point into d_bp_pack); and a host mirror of the carried index (strict handles change it only
    // through calls that know its value), so a tick does not start with a device round trip
    unsigned char *d_bp_pack = nullptr, *h_bp_pack = nullptr;
    int bp_cap = 0;
    int idx_mirror = 0;
    bool idx_mirror_ok = false;
    // multi-GPU
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    float *d_send = nullptr, *d_recv = nullptr;
    // fused peer-memory exchange
    bool p2p = false;
    unsigned long long *d_xchg = nullptr;
    unsigned long long *peer_buf[MPPI_MAX_PEERS] = {nullptr};
    unsigned p2p_seq = 0, p2p_timeout_ms = 2000;
    unsigned long long p2p_barrier_count = 0;
    // MLP dynamics
    MlpState *mlp = nullptr;
    // per-robot reference paths (batched fleets)
    float4 *d_paths = nullptr;
    int *d_path_len = nullptr;
    int path_cap = 0;
    // top-N viewer: per-sample costs of the last tick and their sorted order
    bool keep_costs = false;
    float *d_Sc = nullptr, *d_Ssorted = nullptr;
    int *d_sorted_idx = nullptr, *d_iota = nullptr;
    void *d_sort_temp = nullptr;
    size_t sort_temp_bytes = 0;
    // per-robot scenes (fleets): one SceneRec per robot, installed by mppi_set_robot_goals / mppi_set_robot_obstacles; the
    // components in use are args.scene_mask.  scene_stash: the rollout path of the scene instantiation (1 noise stash, 0
    // regenerate), chosen at the first install; -1 before.
    SceneRec *d_scene = nullptr;
    int scene_stash = -1;
    unsigned long long *d_trace = nullptr;     // per-CTA time stamps of the last tick (mppi_set_trace)
    int trace_n = 0;
    int trace_grid = 0;                        // CTAs per robot of the last traced launch
    // timing / bookkeeping
    bool timing = false;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    mppi_timings_t tm{};
    std::string err;
    std::vector<std::pair<void *, size_t>> guards;     // (buffer, payload bytes) of every guarded allocation
};

// Every device buffer of a handle is allocated with a 256-byte guard zone behind it (pattern 0xA5); mppi_debug_check_guards
// verifies that no kernel wrote past a buffer's end -- the bounds evidence the sanitize subset collects on pools where
// compute-sanitizer cannot run.
#define MPPI_GUARD_BYTES 256
template <typename T>
static cudaError_t gmalloc(mppi_handle_t h, T **p, size_t bytes) {
    void *raw = nullptr;
    cudaError_t e = cudaMalloc(&raw, bytes + MPPI_GUARD_BYTES);
    if (e != cudaSuccess) { *p = nullptr; return e; }
    e = cudaMemset((char *)raw + bytes, 0xA5, MPPI_GUARD_BYTES);
    if (e != cudaSuccess) { cudaFree(raw); *p = nullptr; return e; }
    *p = (T *)raw;
    h->guards.push_back({raw, bytes});
    return cudaSuccess;
}
template <typename T>
static void gfree(mppi_handle_t h, T *p) {
    if (!p) return;
    for (size_t i = 0; i < h->guards.size(); ++i)
        if (h->guards[i].first == (void *)p) { h->guards.erase(h->guards.begin() + i); break; }
    cudaFree((void *)p);
}

#define CK(h, call)                                                                         \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            if (h) (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);           \
            return MPPI_E_CUDA;                                                             \
        }                                                                                   \
    } while (0)

static int fail(mppi_handle_t h, int code, const char *msg) {
    if (h) h->err = msg;
    return code;
}

// finalize_tick raises out[MPPI_OUT_FAULT] of a robot whose costs were not finite, and the fused exchange raises out[7]
// (device + mapped host record) when a peer never published its triple; that tick was NOT applied (nominal and waypoint
// index untouched).  Report it once and clear it, so later ticks are judged on their own.  Call after a stream synchronize.
static int check_tick_faults(mppi_handle_t h) {
    const int R = h->cfg.n_robots;
    if (R > 1) {                                         // a fleet has no mapped record: read every robot's word back
        std::vector<float> fault((size_t)R);
        const size_t pitch = sizeof(float) * MPPI_OUT_STRIDE;
        CK(h, cudaMemcpy2DAsync(fault.data(), sizeof(float), h->d_out + MPPI_OUT_FAULT, pitch, sizeof(float), R,
                                cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        const int r = (int)(std::find_if(fault.begin(), fault.end(), [](float v) { return v != 0.f; }) - fault.begin());
        if (r == R) return MPPI_OK;
        CK(h, cudaMemset2DAsync(h->d_out + MPPI_OUT_FAULT, pitch, 0, sizeof(float), R, h->stream));
        h->err = "robot " + std::to_string(r) + ": non-finite sample costs (NaN/inf observed state); the tick was not applied "
                 "to that robot (its u0 row reads NaN, its nominal and waypoint index are unchanged)";
        return MPPI_E_NUMERIC;
    }
    if (h->h_out[MPPI_OUT_FAULT] != 0.f) {               // finalize_tick refused non-finite costs
        h->h_out[MPPI_OUT_FAULT] = 0.f;
        cudaMemsetAsync(h->d_out + MPPI_OUT_FAULT, 0, sizeof(float), h->stream);
        const bool handoff = h->mlp && mlp_take_fault(h->mlp, h->stream);
        return fail(h, MPPI_E_NUMERIC, handoff ? "learned-dynamics kernel: a cluster hand-off was missed (producer cluster not co-resident); "
                                                 "the tick was not applied"
                                               : "non-finite sample costs (NaN/inf observed state or learned residual); the tick was not applied");
    }
    if (!h->p2p || h->h_out[MPPI_OUT_PEER_TIMEOUT] == 0.f) return MPPI_OK;
    h->h_out[MPPI_OUT_PEER_TIMEOUT] = 0.f;
    cudaMemsetAsync(h->d_out + MPPI_OUT_PEER_TIMEOUT, 0, sizeof(float), h->stream);
    return fail(h, MPPI_E_NCCL, "peer-memory exchange timed out: a rank did not publish its (min, sum w, sum w*eps) triple; "
                               "this tick was not applied");
}

extern "C" {

int mppi_abi_version(void) { return MPPI_ABI_VERSION; }

const char *mppi_strerror(int s) {
    switch (s) {
        case MPPI_OK: return "ok";
        case MPPI_E_BADARG: return "invalid argument or configuration";
        case MPPI_E_CUDA: return "CUDA error (see mppi_last_error)";
        case MPPI_E_NCCL: return "NCCL error (see mppi_last_error)";
        case MPPI_E_STATE: return "call order: reference path / nominal / weights not set";
        case MPPI_E_UNSUPPORTED: return "mode combination not supported";
        case MPPI_E_NOMEM: return "out of memory";
        case MPPI_E_NUMERIC: return "non-finite sample costs: the tick was not applied (see mppi_last_error)";
        default: return "unknown status";
    }
}

const char *mppi_last_error(mppi_handle_t h) { return h ? h->err.c_str() : "null handle"; }

void mppi_default_config(mppi_config_t *c) {
    // defaults of controllers/mppi_differential_drive.py:400-410 with the perf modes off
    std::memset(c, 0, sizeof(*c));
    c->abi_version = MPPI_ABI_VERSION;
    c->model = MPPI_MODEL_DIFFDRIVE;
    c->K = 1000; c->T = 30; c->n_robots = 1; c->window = 20;
    c->cost_mode = MPPI_COST_LAST; c->waypoint_mode = MPPI_WP_STRICT;
    c->filter_kind = MPPI_FILTER_DIFFDRIVE; c->yaw_wrap = 0; c->collision = MPPI_COLLISION_NONE;
    c->K_global = 0; c->k_offset = 0;
    c->dt = 0.1; c->wheel_base = 2.5; c->u_max[0] = 5.0; c->u_max[1] = 3.14;
    c->param_exploration = 1e-4; c->param_lambda = 1.0; c->param_alpha = 0.2; c->temperature = 1e-4;
    c->sigma[0] = 0.1; c->sigma[3] = 0.01;
    c->stage_w[0] = 5; c->stage_w[1] = 5; c->stage_w[2] = 10;
    c->term_w[0] = 5; c->term_w[1] = 5; c->term_w[2] = 10;
    c->margin = 1.0; c->robot_radius = 0.5; c->vehicle_l = 4.0; c->vehicle_w = 3.0;
    c->cost_kind = MPPI_COSTKIND_PATH;
    c->ctrl_w[0] = c->ctrl_w[1] = 0.1; c->soft_obs_weight = 100.0; c->soft_obs_safety = 2.0;   // test/test_mppi_diff_obs.py:48,56-57
}

// The fixed filter operators (A14 / Q7) as T x T matrices, float64 then rounded once.
static void build_filter(int T, int kind, std::vector<float> &M) {
    std::vector<double> m((size_t)T * T, 0.0);
    if (kind == MPPI_FILTER_DIFFDRIVE) {
        // 'same' box convolution of width 10: y[n] = 0.1 * sum_{m=n-5}^{n+4} x[m]; head rows i<5
        // rescaled by 10/(i+5); the tail rescale lands on the last row for i=1..4 (the bug is kept)
        for (int n = 0; n < T; ++n)
            for (int j = n - 5; j <= n + 4; ++j)
                if (j >= 0 && j < T) m[(size_t)n * T + j] = 0.1;
        for (int i = 0; i < 5 && i < T; ++i)
            for (int j = 0; j < T; ++j) m[(size_t)i * T + j] *= 10.0 / (i + 5);
        for (int i = 1; i < 5; ++i)
            for (int j = 0; j < T; ++j) m[(size_t)(T - 1) * T + j] *= 10.0 / (i + 5);
    } else {
        // pad with the first 5 and the last 5 rows, 'same' box convolution, crop
        for (int n = 0; n < T; ++n)
            for (int j = n; j <= n + 9; ++j) {
                const int src = j < 5 ? j : (j < T + 5 ? j - 5 : j - 10);
                m[(size_t)n * T + src] += 0.1;
            }
    }
    M.resize((size_t)T * T);
    for (size_t i = 0; i < M.size(); ++i) M[i] = (float)m[i];
}

static void refresh_obstacle_args(mppi_handle_t h, const double *xyr, int m) {
    TickArgs &a = h->args;
    const mppi_config_t &c = h->cfg;
    a.n_obs = m;
    const double hl = 0.5 * c.vehicle_l * c.margin, hw = 0.5 * c.vehicle_w * c.margin;
    a.fp_hl = (float)hl; a.fp_hw = (float)hw;
    const double diag = std::sqrt(hl * hl + hw * hw);
    for (int i = 0; i < m; ++i) {
        a.obs_x[i] = (float)xyr[3 * i]; a.obs_y[i] = (float)xyr[3 * i + 1];
        const double r = xyr[3 * i + 2];
        if (c.collision == MPPI_COLLISION_CIRCLE) {
            const double rr = c.robot_radius * c.margin + r;
            a.obs_r2[i] = (float)(rr * rr);
        } else {
            a.obs_r2[i] = (float)(r * r);
        }
        const double far = (diag + r) * 1.001 + 1e-3;
        a.obs_far2[i] = (float)(far * far);
    }
}

int mppi_create(const mppi_config_t *cfg, mppi_handle_t *out) {
    if (!cfg || !out) return MPPI_E_BADARG;
    *out = nullptr;
    if (cfg->abi_version != MPPI_ABI_VERSION) return MPPI_E_BADARG;
    if (cfg->K < 1 || cfg->T < 1 || cfg->T > MPPI_MAX_T || cfg->n_robots < 1) return MPPI_E_BADARG;
    if (cfg->window < 1 || cfg->window > MPPI_MAX_WINDOW) return MPPI_E_BADARG;
    if (cfg->model < 0 || cfg->model > MPPI_MODEL_DIFFDRIVE_MLP) return MPPI_E_BADARG;
    if (cfg->filter_kind == MPPI_FILTER_DIFFDRIVE && cfg->T < 10) return MPPI_E_BADARG;   // the reference raises (:263)
    if (cfg->filter_kind == MPPI_FILTER_RACECAR && cfg->T < 5) return MPPI_E_BADARG;
    if (cfg->temperature <= 0.0 || cfg->dt <= 0.0) return MPPI_E_BADARG;
    const double det = cfg->sigma[0] * cfg->sigma[3] - cfg->sigma[1] * cfg->sigma[2];
    if (!(cfg->sigma[0] > 0.0) || !(det > 0.0)) return MPPI_E_BADARG;
    if (cfg->collision == MPPI_COLLISION_FOOTPRINT && cfg->model != MPPI_MODEL_BICYCLE) return MPPI_E_UNSUPPORTED;
    if (cfg->model == MPPI_MODEL_DIFFDRIVE_MLP &&
        (cfg->waypoint_mode != MPPI_WP_FROZEN || cfg->n_robots != 1 || cfg->collision != MPPI_COLLISION_NONE))
        return MPPI_E_UNSUPPORTED;
    if (cfg->cost_kind < MPPI_COSTKIND_PATH || cfg->cost_kind > MPPI_COSTKIND_TARGET_SOFT) return MPPI_E_BADARG;
    const bool pathless = cfg->cost_kind != MPPI_COSTKIND_PATH;
    if (pathless && cfg->model != MPPI_MODEL_DIFFDRIVE) return MPPI_E_UNSUPPORTED;       // both scripts drive a unicycle
    if (cfg->cost_kind == MPPI_COSTKIND_GOAL && cfg->collision == MPPI_COLLISION_FOOTPRINT) return MPPI_E_UNSUPPORTED;
    if (cfg->cost_kind == MPPI_COSTKIND_TARGET_SOFT && cfg->collision != MPPI_COLLISION_NONE) return MPPI_E_UNSUPPORTED;
    if (cfg->waypoint_mode == MPPI_WP_STRICT && cfg->n_robots != 1 && !pathless) return MPPI_E_UNSUPPORTED;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cfg->device >= ndev) return MPPI_E_CUDA;

    mppi_handle_t h = new (std::nothrow) mppi_handle_s();
    if (!h) return MPPI_E_NOMEM;
    h->cfg = *cfg;
    mppi_config_t &c = h->cfg;
    if (c.K_global <= 0) c.K_global = c.K;
    h->nx = (c.model == MPPI_MODEL_BICYCLE) ? 4 : 3;
    h->sum = c.cost_mode == MPPI_COST_SUM;
    h->strict = c.waypoint_mode == MPPI_WP_STRICT && c.cost_kind == MPPI_COSTKIND_PATH;   // no waypoint index without a path
    h->have_path = c.cost_kind != MPPI_COSTKIND_PATH;
#define CKC(call)                                                                           \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            std::fprintf(stderr, "mppi_create: %s: %s\n", #call, cudaGetErrorString(e_));  \
            mppi_destroy(h);                                                                \
            return MPPI_E_CUDA;                                                             \
        }                                                                                   \
    } while (0)
    CKC(cudaSetDevice(c.device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, c.device));
    h->n_sm = prop.multiProcessorCount;
    CKC(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;

    const int R = c.n_robots, T = c.T, K = c.K;
    // Small sample counts are latency-bound (one thread walks one sample through the whole horizon): spread them over
    // all SMs in CTAs that own as few as MPPI_MIN_CTA_SAMPLES samples (idle warps of a CTA cost nothing) instead of
    // filling 256-thread CTAs on a fraction of the SMs.
    int min_cta = 128;
    if (const char *env = std::getenv("MPPI_MIN_CTA_SAMPLES")) min_cta = std::max(32, std::min(MPPI_BLOCK, std::atoi(env)));
    const int chunks = (K + min_cta - 1) / min_cta;
    const int tick_model = (c.model == MPPI_MODEL_DIFFDRIVE_MLP) ? MPPI_MODEL_DIFFDRIVE : c.model;
    h->occ = std::max(1, mppi_tick_occupancy(tick_model, c.collision, c.cost_kind, h->sum, false, c.window, T, false));
    const int occ_stash = mppi_tick_occupancy(tick_model, c.collision, c.cost_kind, h->sum, false, c.window, T, true);
    h->stash = occ_stash >= MPPI_STASH_BLOCKS && c.model != MPPI_MODEL_DIFFDRIVE_MLP;
    int gx = (h->n_sm * h->occ + R - 1) / R;
    gx = std::max(1, std::min(gx, chunks));
    h->grid_x = gx;
    int gxs = (h->n_sm * std::max(1, occ_stash) + R - 1) / R;
    h->grid_x_stash = std::max(1, std::min(gxs, chunks));
    gx = std::max(h->grid_x, h->grid_x_stash);
    // Time-parallel rollout (mppi_device.cuh, rollout_tpar): when one robot's samples cannot fill the GPU anyway -- every CTA would own
    // <= MPPI_TPAR_SLOTS of them at two CTAs per SM -- the tick is bound by the latency of one thread's walk through the horizon, and
    // splitting the horizon into noise / recurrence / cost phases over all threads of the CTA cuts that latency (race-car K = 16 384,
    // H = 50: 73 -> 47 us per tick).  Dynamic-window kernels only: with the static 20-entry window the stage cost is too cheap next to
    // the recurrence for the split to pay (diff-drive K = 16 384, H = 30: 22.3 -> 24.6 us, measured).  MPPI_TPAR=0 / 1 overrides.
    {
        const int occ_tpar = (h->sum && c.cost_kind == MPPI_COSTKIND_PATH && c.window != 20 && c.model != MPPI_MODEL_DIFFDRIVE_MLP)
                                 ? mppi_tick_occupancy(tick_model, c.collision, c.cost_kind, true, false, c.window, T, 2) : 0;
        const int gt = std::max(1, std::min(h->n_sm * std::max(1, occ_tpar), (K + 7) / 8));
        const bool fits = occ_tpar >= 1 && (K + gt - 1) / gt <= MPPI_TPAR_SLOTS;
        bool want = R == 1;
        if (const char *env = std::getenv("MPPI_TPAR")) want = std::atoi(env) != 0;
        if (std::getenv("MPPI_VERBOSE"))
            std::fprintf(stderr, "mppi_create: time-parallel rollout: occ %d grid %d fits %d want %d (stash %d sum %d window %d K %d T %d)\n",
                         occ_tpar, gt, (int)fits, (int)want, (int)h->stash, (int)h->sum, c.window, K, T);
        if (want && fits) {
            h->tpar = true;
            h->grid_x_tpar = gt;
            gx = std::max(gx, gt);
        }
        if (std::getenv("MPPI_VERBOSE"))          // the path Philox ticks take, and its grid
            std::fprintf(stderr, "mppi_create: rollout path %s, %d CTAs per robot\n", h->tpar ? "tpar" : h->stash ? "stash" : "regenerate",
                         h->tpar ? h->grid_x_tpar : h->stash ? h->grid_x_stash : h->grid_x);
    }

    CKC(gmalloc(h, &h->d_U, sizeof(float) * R * T * 2));
    CKC(cudaMemset(h->d_U, 0, sizeof(float) * R * T * 2));
    CKC(gmalloc(h, &h->d_M, sizeof(float) * T * T));
    CKC(gmalloc(h, &h->d_S, sizeof(float) * (size_t)R * K));
    CKC(gmalloc(h, &h->d_NC, sizeof(int) * (size_t)K));
    const int gmax = (gx + MPPI_MERGE_GROUP_CTAS - 1) / MPPI_MERGE_GROUP_CTAS;      // two-level merge: group partials behind the block partials
    CKC(gmalloc(h, &h->d_part, sizeof(float) * (size_t)R * (gx + gmax) * MPPI_NF(T)));
    CKC(gmalloc(h, &h->d_out, sizeof(float) * (size_t)R * MPPI_OUT_STRIDE));
    CKC(cudaMemset(h->d_out, 0, sizeof(float) * (size_t)R * MPPI_OUT_STRIDE));
    CKC(gmalloc(h, &h->d_idx, sizeof(int) * R));
    CKC(cudaMemset(h->d_idx, 0, sizeof(int) * R));
    CKC(gmalloc(h, &h->d_ticket, sizeof(unsigned) * (size_t)R * (1 + gmax)));
    CKC(cudaMemset(h->d_ticket, 0, sizeof(unsigned) * (size_t)R * (1 + gmax)));
    CKC(cudaHostAlloc(&h->h_out, sizeof(float) * MPPI_OUT_STRIDE, cudaHostAllocMapped));
    std::memset(h->h_out, 0, sizeof(float) * MPPI_OUT_STRIDE);
    CKC(cudaHostGetDevicePointer(&h->h_out_dev, h->h_out, 0));
    CKC(gmalloc(h, &h->d_first, sizeof(unsigned long long)));
    CKC(cudaHostAlloc(&h->h_first, sizeof(unsigned long long), cudaHostAllocDefault));
    h->idx_mirror = 0; h->idx_mirror_ok = true;
    for (auto &e : h->ev) CKC(cudaEventCreate(&e));
    std::vector<float> M;
    build_filter(T, c.filter_kind, M);
    CKC(cudaMemcpy(h->d_M, M.data(), sizeof(float) * T * T, cudaMemcpyHostToDevice));

    TickArgs &a = h->args;
    std::memset(&a, 0, sizeof(a));
    a.K = K; a.T = T; a.window = c.window; a.yaw_wrap = c.yaw_wrap; a.clamp_nominal = c.clamp_nominal;
    a.k_offset = c.k_offset;
    {   // Q6: number of global sample indices k with k < (1.0 - param_exploration) * K, in doubles
        const double thr = (1.0 - c.param_exploration) * (double)c.K_global;
        long long n = (long long)std::ceil(thr);
        n = std::max(0LL, std::min((long long)c.K_global, n));
        a.n_exploit = (int)n;
    }
    a.dt = (float)c.dt; a.dt_over_L = (float)(c.dt / c.wheel_base);
    a.umax0 = (float)c.u_max[0]; a.umax1 = (float)c.u_max[1];
    for (int i = 0; i < 4; ++i) { a.sw[i] = (float)c.stage_w[i]; a.tw[i] = (float)c.term_w[i]; }
    const double gamma = c.param_lambda * (1.0 - c.param_alpha);       // :74
    a.use_gamma = gamma != 0.0;
    a.gq[0] = (float)(gamma * c.sigma[3] / det); a.gq[1] = (float)(-gamma * c.sigma[1] / det);
    a.gq[2] = (float)(-gamma * c.sigma[2] / det); a.gq[3] = (float)(gamma * c.sigma[0] / det);
    const double l00 = std::sqrt(c.sigma[0]), l10 = c.sigma[2] / l00;
    a.chol[0] = (float)l00; a.chol[1] = (float)l10; a.chol[2] = (float)std::sqrt(c.sigma[3] - l10 * l10);
    a.inv_temp = (float)(1.0 / c.temperature);
    for (int i = 0; i < 4; ++i) a.goal[i] = (float)c.goal[i];
    a.ctrl_w[0] = (float)c.ctrl_w[0]; a.ctrl_w[1] = (float)c.ctrl_w[1];
    a.soft_w = (float)c.soft_obs_weight; a.soft_sd = (float)c.soft_obs_safety;
    refresh_obstacle_args(h, nullptr, 0);
    a.U = h->d_U; a.idx = h->d_idx; a.M = h->d_M; a.part = h->d_part; a.ticket = h->d_ticket;
    a.part2 = h->d_part + (size_t)R * gx * MPPI_NF(T); a.ticket2 = h->d_ticket + R; a.merge_gmax = gmax;
    a.out = h->d_out; a.out_host = h->h_out_dev;
    if (c.model == MPPI_MODEL_DIFFDRIVE_MLP) {
        h->mlp = mlp_create(K, T);
        if (!h->mlp) { mppi_destroy(h); return MPPI_E_CUDA; }
    }
#undef CKC
    *out = h;
    return MPPI_OK;
}

int mppi_destroy(mppi_handle_t h) {
    if (!h) return MPPI_E_BADARG;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    if (h->p2p)
        for (int p = 0; p < h->world; ++p)
            if (p != h->rank && h->peer_buf[p]) cudaIpcCloseMemHandle(h->peer_buf[p]);
    gfree(h, h->d_xchg); gfree(h, h->d_trace); gfree(h, h->d_loop);
    if (h->loop_graph) cudaGraphExecDestroy(h->loop_graph);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    gfree(h, h->d_paths); gfree(h, h->d_path_len); gfree(h, h->d_scene);
    gfree(h, h->d_Sc); gfree(h, h->d_Ssorted); gfree(h, h->d_sorted_idx); gfree(h, h->d_iota); gfree(h, h->d_sort_temp);
    if (h->mlp) mlp_destroy(h->mlp);
    gfree(h, h->d_path); gfree(h, h->d_U); gfree(h, h->d_M); gfree(h, h->d_S); gfree(h, h->d_part);
    gfree(h, h->d_out); gfree(h, h->d_idx); gfree(h, h->d_NC); gfree(h, h->d_ticket); gfree(h, h->d_first);
    gfree(h, h->d_bp_n); gfree(h, h->d_bp_s); gfree(h, h->d_send); gfree(h, h->d_recv); gfree(h, h->d_x0); gfree(h, h->d_opt); gfree(h, h->d_plant_log);
    if (h->h_out) cudaFreeHost(h->h_out);
    if (h->h_first) cudaFreeHost(h->h_first);
    if (h->h_bp_pack) cudaFreeHost(h->h_bp_pack);
    gfree(h, h->d_bp_pack);
    for (auto &e : h->ev) if (e) cudaEventDestroy(e);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return MPPI_OK;
}

int mppi_set_stream(mppi_handle_t h, void *st) {
    if (!h) return MPPI_E_BADARG;
    if (h->own_stream && h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
    h->stream = (cudaStream_t)st;
    h->own_stream = false;
    return MPPI_OK;
}

int mppi_synchronize(mppi_handle_t h) {
    if (!h) return MPPI_E_BADARG;
    CK(h, cudaStreamSynchronize(h->stream));
    return check_tick_faults(h);                       // the asynchronous path (mppi_step_async) reports here
}

int mppi_set_ref_path(mppi_handle_t h, const double *path, int32_t n, int32_t ncol) {
    if (!h || !path || n < 1 || (ncol != 3 && ncol != 4)) return MPPI_E_BADARG;
    if (h->cfg.model == MPPI_MODEL_BICYCLE && ncol != 4) return fail(h, MPPI_E_BADARG, "bicycle model needs (N,4) path");
    if (h->cfg.cost_kind != MPPI_COSTKIND_PATH) return fail(h, MPPI_E_STATE, "goal / target cost kinds take no reference path");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    std::vector<float4> p((size_t)n);
    for (int i = 0; i < n; ++i) {
        const double *r = path + (size_t)i * ncol;
        p[i] = make_float4((float)r[0], (float)r[1], (float)r[2], ncol == 4 ? (float)r[3] : 0.f);
    }
    gfree(h, h->d_path); h->d_path = nullptr;
    gfree(h, h->d_bp_n); gfree(h, h->d_bp_s); h->d_bp_n = nullptr; h->d_bp_s = nullptr;
    CK(h, gmalloc(h, &h->d_path, sizeof(float4) * n));
    CK(h, cudaMemcpy(h->d_path, p.data(), sizeof(float4) * n, cudaMemcpyHostToDevice));
    CK(h, gmalloc(h, &h->d_bp_n, sizeof(unsigned) * (n + 2)));
    CK(h, gmalloc(h, &h->d_bp_s, sizeof(int) * (n + 2)));
    if (h->strict) {
        gfree(h, h->d_bp_pack); h->d_bp_pack = nullptr;
        if (h->h_bp_pack) { cudaFreeHost(h->h_bp_pack); h->h_bp_pack = nullptr; }
        h->bp_cap = n + 2;
        const size_t bytes = sizeof(unsigned long long) + (sizeof(unsigned) + sizeof(int)) * (size_t)h->bp_cap;
        CK(h, gmalloc(h, &h->d_bp_pack, bytes));
        CK(h, cudaHostAlloc(&h->h_bp_pack, bytes, cudaHostAllocDefault));
    }
    h->path_h.assign(path, path + (size_t)n * ncol);
    h->n_path = n; h->path_cols = ncol;
    h->args.path = h->d_path; h->args.n_path = n;
    h->args.path_len = nullptr; h->args.path_stride = 0;          // back to one shared path
    h->have_path = true;
    {   // a carried index past the end of a SHORTER new path is clamped to its last waypoint (what step 1 does at the path
        // end, mppi_differential_drive.py:97-99) instead of indexing the new path out of bounds
        std::vector<int> idx((size_t)h->cfg.n_robots);
        CK(h, cudaMemcpy(idx.data(), h->d_idx, sizeof(int) * idx.size(), cudaMemcpyDeviceToHost));
        bool changed = false;
        for (int &v : idx) { const int c = std::max(0, std::min(v, n - 1)); changed |= c != v; v = c; }
        if (changed) CK(h, cudaMemcpy(h->d_idx, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice));
        h->idx_mirror = idx[0]; h->idx_mirror_ok = true;
    }
    return MPPI_OK;
}

int mppi_set_ref_paths_spline(mppi_handle_t h, const float *d_wx, const float *d_wy, int32_t n_wp, double ds, int32_t max_points) {
    if (!h || !d_wx || !d_wy || n_wp < 2 || n_wp > MPPI_SPLINE_MAX_WAYPOINTS || !(ds > 0.0) || max_points < 2) return MPPI_E_BADARG;
    if (h->cfg.cost_kind != MPPI_COSTKIND_PATH) return fail(h, MPPI_E_STATE, "goal / target cost kinds take no reference path");
    if (h->strict || h->mlp) return fail(h, MPPI_E_UNSUPPORTED, "per-robot paths: frozen waypoint mode, analytic dynamics");
    if (h->cfg.model == MPPI_MODEL_BICYCLE) return fail(h, MPPI_E_UNSUPPORTED, "calc_spline_course yields (x, y, yaw): diff-drive paths");
    CK(h, cudaSetDevice(h->cfg.device));
    const int R = h->cfg.n_robots;
    if (h->path_cap < max_points) {
        CK(h, cudaStreamSynchronize(h->stream));
        gfree(h, h->d_paths); h->d_paths = nullptr;
        CK(h, gmalloc(h, &h->d_paths, sizeof(float4) * (size_t)R * max_points));
        h->path_cap = max_points;
    }
    if (!h->d_path_len) CK(h, gmalloc(h, &h->d_path_len, sizeof(int) * R));
    CK(h, mppi_launch_spline(d_wx, d_wy, R, n_wp, ds, h->path_cap, h->d_paths, h->d_path_len, h->stream));
    h->tm.launches++;
    std::vector<int> len((size_t)R);
    CK(h, cudaMemcpyAsync(len.data(), h->d_path_len, sizeof(int) * R, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    for (int r = 0; r < R; ++r)
        if (len[r] < 1) return fail(h, MPPI_E_BADARG, "a robot's course needs more than max_points samples (or its waypoints coincide)");
    h->args.path = h->d_paths; h->args.path_len = h->d_path_len; h->args.path_stride = h->path_cap;
    h->args.n_path = 0;
    h->have_path = true;
    return MPPI_OK;
}

int mppi_get_ref_path(mppi_handle_t h, int32_t robot, float *path_out, int32_t capacity, int32_t *n_out) {
    if (!h || !n_out || robot < 0 || robot >= h->cfg.n_robots || capacity < 0) return MPPI_E_BADARG;
    if (!h->have_path || h->cfg.cost_kind != MPPI_COSTKIND_PATH) return fail(h, MPPI_E_STATE, "no reference path set");
    CK(h, cudaSetDevice(h->cfg.device));
    int n = h->n_path;
    const float4 *src = h->d_path;
    if (h->args.path_len) {
        CK(h, cudaMemcpyAsync(&n, h->d_path_len + robot, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        src = h->d_paths + (size_t)robot * h->path_cap;
    }
    *n_out = n;
    if (path_out) {
        const int m = n < capacity ? n : capacity;
        CK(h, cudaMemcpyAsync(path_out, src, sizeof(float4) * m, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
    }
    return MPPI_OK;
}

int mppi_set_obstacles(mppi_handle_t h, const double *xyr, int32_t m) {
    if (!h || m < 0 || m > MPPI_MAX_OBSTACLES || (m > 0 && !xyr)) return MPPI_E_BADARG;
    if (h->cfg.cost_kind == MPPI_COSTKIND_TARGET_SOFT) return fail(h, MPPI_E_STATE, "TARGET_SOFT takes mppi_set_moving_obstacles");
    refresh_obstacle_args(h, xyr, m);
    h->args.scene_mask &= ~MPPI_SCENE_OBS;                 // back to one shared obstacle set
    return MPPI_OK;
}

int mppi_set_goal(mppi_handle_t h, const double *goal, int32_t n) {
    if (!h || !goal || n < 2 || n > 3) return MPPI_E_BADARG;
    if (h->cfg.cost_kind == MPPI_COSTKIND_PATH) return fail(h, MPPI_E_STATE, "handle was not created with a goal / target cost kind");
    for (int i = 0; i < n; ++i) { h->cfg.goal[i] = goal[i]; h->args.goal[i] = (float)goal[i]; }
    h->args.scene_mask &= ~MPPI_SCENE_GOAL;                // back to one shared goal
    return MPPI_OK;
}

int mppi_set_moving_obstacles(mppi_handle_t h, const double *pos, const double *vel, int32_t m) {
    if (!h || m < 0 || m > MPPI_MAX_OBSTACLES || (m > 0 && (!pos || !vel))) return MPPI_E_BADARG;
    if (h->cfg.cost_kind != MPPI_COSTKIND_TARGET_SOFT) return fail(h, MPPI_E_STATE, "handle was not created with MPPI_COSTKIND_TARGET_SOFT");
    TickArgs &a = h->args;
    a.n_obs = m;
    for (int i = 0; i < m; ++i) {
        a.obs_x[i] = (float)pos[2 * i]; a.obs_y[i] = (float)pos[2 * i + 1];
        a.obs_vx[i] = (float)vel[2 * i]; a.obs_vy[i] = (float)vel[2 * i + 1];
    }
    a.scene_mask &= ~MPPI_SCENE_OBS;                       // back to one shared obstacle set
    return MPPI_OK;
}

// ---- per-robot scenes (fleets) ---------------------------------------------------------------------------------------------
// Checks common to both installs; allocates the table and picks the scene instantiation's rollout path on first use: the
// handle's noise-stash path (time-parallel handles too: the scene instantiations have no time-parallel variant) when that
// kernel can be resident, else its regenerate-noise variant.  The grid widths stay the ones mppi_create computed.
static int scene_modes_supported(mppi_handle_t h) {
    if (h->strict || h->mlp) return fail(h, MPPI_E_UNSUPPORTED, "per-robot goals / obstacles: frozen waypoint mode, analytic dynamics");
    if (h->world > 1) return fail(h, MPPI_E_UNSUPPORTED, "per-robot goals / obstacles: one GPU (no sample sharding)");
    return MPPI_OK;
}

static int prepare_scene(mppi_handle_t h) {
    CK(h, cudaSetDevice(h->cfg.device));
    if (h->scene_stash < 0) {
        const mppi_config_t &c = h->cfg;
        const bool want_stash = h->stash || h->tpar;
        const int occ_st = want_stash ? mppi_tick_occupancy(c.model, c.collision, c.cost_kind, h->sum, false, c.window, c.T, 1, true) : 0;
        const int occ_rg = occ_st >= 1 ? 0 : mppi_tick_occupancy(c.model, c.collision, c.cost_kind, h->sum, false, c.window, c.T, 0, true);
        if (occ_st < 1 && occ_rg < 1)
            return fail(h, MPPI_E_UNSUPPORTED, "per-robot goals / obstacles are built for diff-drive + circles and bicycle + footprint "
                                               "on a path, and for the GOAL (no obstacles or circles) and TARGET_SOFT cost kinds");
        h->scene_stash = occ_st >= 1 ? 1 : 0;
        if (std::getenv("MPPI_VERBOSE"))
            std::fprintf(stderr, "mppi_set_robot_*: scene ticks take the %s path, %d CTAs per robot (occ %d)%s\n",
                         h->scene_stash ? "stash" : "regenerate", h->scene_stash ? h->grid_x_stash : h->grid_x,
                         h->scene_stash ? occ_st : occ_rg,
                         h->tpar ? "; this handle's shared-scene ticks are time-parallel, its scene ticks are not" : "");
    }
    if (!h->d_scene) {
        CK(h, gmalloc(h, &h->d_scene, sizeof(SceneRec) * h->cfg.n_robots));
        CK(h, cudaMemsetAsync(h->d_scene, 0, sizeof(SceneRec) * h->cfg.n_robots, h->stream));
    }
    return MPPI_OK;
}

int mppi_set_robot_obstacles(mppi_handle_t h, const float *d_obs, const int32_t *d_count, int32_t m, int32_t ncol) {
    if (!h || m < 0 || m > MPPI_MAX_OBSTACLES || (ncol != 3 && ncol != 4) || (m > 0 && !d_obs)) return MPPI_E_BADARG;
    if (int rc = scene_modes_supported(h)) return rc;
    const mppi_config_t &c = h->cfg;
    if (ncol == 4 && c.cost_kind != MPPI_COSTKIND_TARGET_SOFT)
        return fail(h, MPPI_E_STATE, "moving obstacles [x, y, vx, vy] belong to MPPI_COSTKIND_TARGET_SOFT handles");
    if (ncol == 3 && (c.cost_kind == MPPI_COSTKIND_TARGET_SOFT || c.collision == MPPI_COLLISION_NONE))
        return fail(h, MPPI_E_STATE, "static circles [x, y, r] need a handle created with circle or footprint collision");
    if (int rc = prepare_scene(h)) return rc;
    const double hl = 0.5 * c.vehicle_l * c.margin, hw = 0.5 * c.vehicle_w * c.margin;       // as refresh_obstacle_args
    CK(h, mppi_launch_scene_obstacles(d_obs, d_count, c.n_robots, m, ncol, c.collision == MPPI_COLLISION_CIRCLE,
                                      c.robot_radius * c.margin, std::sqrt(hl * hl + hw * hw), h->d_scene, h->stream));
    h->tm.launches++;
    h->args.scene = h->d_scene;
    h->args.scene_mask |= MPPI_SCENE_OBS;
    return MPPI_OK;
}

int mppi_set_robot_goals(mppi_handle_t h, const float *d_goal, int32_t n) {
    if (!h || !d_goal || n < 2 || n > 3) return MPPI_E_BADARG;
    if (int rc = scene_modes_supported(h)) return rc;
    const int kind = h->cfg.cost_kind;
    if (kind == MPPI_COSTKIND_PATH) return fail(h, MPPI_E_STATE, "handle was not created with a goal / target cost kind");
    if (n != (kind == MPPI_COSTKIND_GOAL ? 2 : 3))
        return fail(h, MPPI_E_BADARG, "per-robot goals: n = 2 (GOAL: goal point) or 3 (TARGET_SOFT: target pose)");
    if (int rc = prepare_scene(h)) return rc;
    CK(h, mppi_launch_scene_goals(d_goal, h->cfg.n_robots, n, h->d_scene, h->stream));
    h->tm.launches++;
    h->args.scene = h->d_scene;
    h->args.scene_mask |= MPPI_SCENE_GOAL;
    return MPPI_OK;
}

// The per-robot scene is threaded through the fleet tick (mppi_step_batched, mppi_run_closed_loop) only.
static int scene_refused(mppi_handle_t h, const char *what) {
    if (!h->args.scene_mask) return MPPI_OK;
    h->err = std::string(what) + ": per-robot goals / obstacles are installed; they are run by mppi_step_batched and "
                                 "mppi_run_closed_loop (mppi_set_goal / mppi_set_obstacles / mppi_set_moving_obstacles "
                                 "return the handle to the shared scene)";
    return MPPI_E_STATE;
}

int mppi_set_nominal(mppi_handle_t h, const float *u) {
    if (!h || !u) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(h->d_U, u, sizeof(float) * h->cfg.n_robots * h->cfg.T * 2, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_get_nominal(mppi_handle_t h, float *u) {
    if (!h || !u) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(u, h->d_U, sizeof(float) * h->cfg.n_robots * h->cfg.T * 2, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_set_waypoint_idx(mppi_handle_t h, const int32_t *idx) {
    if (!h || !idx) return MPPI_E_BADARG;
    // the reference fails on an index outside the path (min() of the empty window slice, mppi_differential_drive.py:214);
    // here it would send the window search out of bounds, so it is refused
    const int limit = h->args.path_len ? h->path_cap : (h->have_path && h->cfg.cost_kind == MPPI_COSTKIND_PATH ? h->n_path : INT32_MAX);
    for (int r = 0; r < h->cfg.n_robots; ++r)
        if (idx[r] < 0 || idx[r] >= limit) return fail(h, MPPI_E_BADARG, "waypoint index outside the reference path");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(h->d_idx, idx, sizeof(int) * h->cfg.n_robots, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    h->idx_mirror = idx[0]; h->idx_mirror_ok = true;
    return MPPI_OK;
}

int mppi_get_waypoint_idx(mppi_handle_t h, int32_t *idx) {
    if (!h || !idx) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(idx, h->d_idx, sizeof(int) * h->cfg.n_robots, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_set_mlp(mppi_handle_t h, const float *const W[4], const float *const b[4]) {
    if (!h || !W || !b) return MPPI_E_BADARG;
    if (!h->mlp) return fail(h, MPPI_E_STATE, "handle was not created with MPPI_MODEL_DIFFDRIVE_MLP");
    CK(h, cudaSetDevice(h->cfg.device));
    if (mlp_set_weights(h->mlp, 3, 2, W, b, nullptr, nullptr, nullptr, nullptr, h->stream) != cudaSuccess)
        return fail(h, MPPI_E_CUDA, "mlp_set_weights failed");
    return MPPI_OK;
}

int mppi_set_mlp_ex(mppi_handle_t h, int32_t n_in, int32_t n_hidden, const float *const *W, const float *const *b,
                    const double *in_mean, const double *in_scale, const double *out_mean, const double *out_scale) {
    if (!h || !W || !b || (n_in != 3 && n_in != 5) || n_hidden < 1) return MPPI_E_BADARG;
    if (!h->mlp) return fail(h, MPPI_E_STATE, "handle was not created with MPPI_MODEL_DIFFDRIVE_MLP");
    if (n_hidden != 2 && n_hidden != 3)
        return fail(h, MPPI_E_UNSUPPORTED, "the tensor-core rollout runs residuals with two or three 512-wide tanh layers "
                                           "(saved_models/mlp_diff*.pth, mlp_diff_300x100_3l*.pth)");
    for (int i = 0; i < n_hidden + 2; ++i) if (!W[i] || !b[i]) return MPPI_E_BADARG;
    if (in_scale) for (int c = 0; c < n_in; ++c) if (!(in_scale[c] != 0.0)) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    if (mlp_set_weights(h->mlp, n_in, n_hidden, W, b, in_mean, in_scale, out_mean, out_scale, h->stream) != cudaSuccess)
        return fail(h, MPPI_E_CUDA, "mlp_set_weights failed");
    return MPPI_OK;
}

int mppi_mlp_schedule_cut(int32_t c, int32_t n_clusters, int32_t n_units, int32_t T) {
    if (c < 0 || n_clusters <= 0 || n_units < 0 || T <= 0) return -1;
    return mlp_bal_cut(c, n_clusters, n_units, T);
}

int mppi_set_timing(mppi_handle_t h, int32_t on) {
    if (!h) return MPPI_E_BADARG;
    h->timing = on != 0;
    return MPPI_OK;
}

int mppi_get_timings(mppi_handle_t h, mppi_timings_t *out) {
    if (!h || !out) return MPPI_E_BADARG;
    *out = h->tm;
    return MPPI_OK;
}

int mppi_get_stats(mppi_handle_t h, mppi_stats_t *out) {
    if (!h || !out) return MPPI_E_BADARG;
    float hdr[MPPI_OUT_HDR];
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(hdr, h->d_out, sizeof(hdr), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    out->rho = hdr[3]; std::memcpy(&out->min_collisions, &hdr[4], 4);
    out->eta = hdr[5]; out->ess = hdr[6]; std::memcpy(&out->idx, &hdr[2], 4);
    out->u_first[0] = hdr[8]; out->u_first[1] = hdr[9];
    return MPPI_OK;
}

// ---------------------------------------------------------------------------------------------
static void set_x0(mppi_handle_t h, const double *x0) {
    for (int i = 0; i < 4; ++i) h->args.x0[i] = i < h->nx ? (float)x0[i] : 0.f;
}

static void set_seed(mppi_handle_t h, uint64_t seed, uint64_t tick) {
    h->args.seed_lo = (uint32_t)seed; h->args.seed_hi = (uint32_t)(seed >> 32);
    h->args.tick = (uint32_t)tick;
}

static int host_nearest(mppi_handle_t h, int s, double x, double y) {
    // literal FP64 step 1 (mppi_differential_drive.py:96 -> :201-220), first minimum
    const int end = std::min(s + h->cfg.window, h->n_path);
    int best = s;
    double bd = INFINITY;
    for (int j = s; j < end; ++j) {
        const double dx = x - h->path_h[(size_t)j * h->path_cols], dy = y - h->path_h[(size_t)j * h->path_cols + 1];
        const double d = dx * dx + dy * dy;
        if (d < bd) { bd = d; best = j; }
    }
    return best;
}

// Strict waypoint mode: host-driven multi-pass rollout (SURVEY.md section 7).  Leaves the costs
// in d_S (or dS_user) and returns the index after the tick.
static int strict_costs(mppi_handle_t h, const double *x0, const float *d_eps, float *dS_user, int *idx_after) {
    int idx0 = h->idx_mirror;
    if (!h->idx_mirror_ok) {
        CK(h, cudaMemcpyAsync(&idx0, h->d_idx, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
    }
    h->idx_mirror_ok = false;               // until the caller has persisted the index this tick ends with
    idx0 = std::max(0, std::min(idx0, h->n_path - 1));
    const int s0 = host_nearest(h, idx0, x0[0], x0[1]);
    std::vector<unsigned> bpn{0u};
    std::vector<int> bps{s0};
    TickArgs a = h->args;
    a.S = h->d_S; a.NC = h->d_NC; a.S_user = dS_user; a.eps = d_eps;
    const int T = h->cfg.T;
    int k_first = 0;
    unsigned check_from = 0;
    int passes = 0;
    const unsigned long long none = ~0ull;
    while (true) {
        // one pinned staging buffer, one copy: [first-change word = none][bp_n[0..nbp)][bp_s[0..nbp)]
        const size_t nbp = bpn.size();
        if ((int)nbp > h->bp_cap || !h->d_bp_pack) return fail(h, MPPI_E_STATE, "strict mode: breakpoint buffer");
        std::memcpy(h->h_bp_pack, &none, sizeof(none));
        std::memcpy(h->h_bp_pack + sizeof(none), bpn.data(), sizeof(unsigned) * nbp);
        std::memcpy(h->h_bp_pack + sizeof(none) + sizeof(unsigned) * nbp, bps.data(), sizeof(int) * nbp);
        CK(h, cudaMemcpyAsync(h->d_bp_pack, h->h_bp_pack, sizeof(none) + (sizeof(unsigned) + sizeof(int)) * nbp, cudaMemcpyHostToDevice, h->stream));
        unsigned long long *d_first = reinterpret_cast<unsigned long long *>(h->d_bp_pack);
        const unsigned *d_bpn = reinterpret_cast<const unsigned *>(h->d_bp_pack + sizeof(none));
        const int *d_bps = reinterpret_cast<const int *>(h->d_bp_pack + sizeof(none) + sizeof(unsigned) * nbp);
        CK(h, mppi_launch_strict(a, h->cfg.model, h->cfg.collision, h->sum, d_eps != nullptr, d_bpn, d_bps,
                                 (int)nbp, k_first, check_from, d_first, h->stream));
        h->tm.launches++;
        CK(h, cudaMemcpyAsync(h->h_first, d_first, sizeof(none), cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        ++passes;
        const unsigned long long fc = *h->h_first;
        if (fc == none) break;
        const unsigned n_star = (unsigned)(fc >> 32);
        const int s_new = (int)(fc & 0xffffffffu);
        bpn.push_back(n_star + 1); bps.push_back(s_new);
        check_from = n_star + 1;
        k_first = (int)(check_from / (unsigned)(T + 1));
        if ((int)bpn.size() > h->n_path + 1) return fail(h, MPPI_E_STATE, "strict mode: too many index changes");
        if (k_first >= h->cfg.K) break;
    }
    h->tm.last_passes = passes;
    *idx_after = bps.back();
    return MPPI_OK;
}

static int launch_update(mppi_handle_t h, const TickArgs &a, bool inj) {
    const bool scene = a.scene_mask != 0;                // only the fleet entry points get here with a scene installed
    const int stash = scene ? h->scene_stash : (!inj && !(a.flags & F_FROM_S)) ? (h->tpar ? 2 : h->stash ? 1 : 0) : 0;
    dim3 grid(stash == 2 ? h->grid_x_tpar : stash ? h->grid_x_stash : h->grid_x, h->cfg.n_robots);
    if (a.trace) h->trace_grid = (int)grid.x;
    const int model = (h->cfg.model == MPPI_MODEL_DIFFDRIVE_MLP) ? MPPI_MODEL_DIFFDRIVE : h->cfg.model;
    if (h->world > 1 && h->p2p && (a.flags & F_UPDATE)) {
        TickArgs b = a;                      // exchange fused into the tick kernel: ONE launch, no NCCL call
        b.flags |= F_P2P;
        for (int p = 0; p < h->world; ++p) b.peer_buf[p] = h->peer_buf[p];
        b.p2p_rank = h->rank; b.p2p_world = h->world; b.p2p_seq = ++h->p2p_seq; b.p2p_timeout_ms = h->p2p_timeout_ms;
        CK(h, mppi_launch_tick(b, model, h->cfg.collision, h->cfg.cost_kind, h->sum, inj, stash, grid, h->stream));
        h->tm.launches++;
        return MPPI_OK;
    }
    if (h->world > 1 && (a.flags & F_UPDATE)) {
        TickArgs b = a;
        b.flags |= F_TRIPLE_OUT;
        b.triple_out = h->d_send;
        CK(h, mppi_launch_tick(b, model, h->cfg.collision, h->cfg.cost_kind, h->sum, inj, stash, grid, h->stream));
        const size_t nf = MPPI_NF(h->cfg.T);
        ncclResult_t r = g_nccl.AllGather(h->d_send, h->d_recv, nf, ncclFloat, h->comm, h->stream);
        if (r != ncclSuccess) { h->err = g_nccl.GetErrorString(r); return MPPI_E_NCCL; }
        CK(h, mppi_launch_merge(a, h->d_recv, h->world, h->stream));
        h->tm.launches += 2;
        return MPPI_OK;
    }
    CK(h, mppi_launch_tick(a, model, h->cfg.collision, h->cfg.cost_kind, h->sum, inj, stash, grid, h->stream, scene));
    h->tm.launches++;
    return MPPI_OK;
}

static int step_common(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick, bool sync_out,
                       float *u0_out, float *useq_out) {
    if (!h || !x0) return MPPI_E_BADARG;
    if (!h->have_path) return fail(h, MPPI_E_STATE, "mppi_set_ref_path has not been called");
    if (h->cfg.n_robots != 1) return fail(h, MPPI_E_BADARG, "use mppi_step_batched for n_robots > 1");
    if (int rc = scene_refused(h, "mppi_step")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    set_x0(h, x0);
    set_seed(h, seed, tick);
    if (h->timing) CK(h, cudaEventRecord(h->ev[0], h->stream));
    int strict_idx_after = -1;
    if (h->mlp) {
        int rc = mlp_rollout_costs(h->mlp, h->args, h->sum, d_eps, h->d_S, h->stream);
        if (rc != 0) return fail(h, rc == -2 ? MPPI_E_STATE : MPPI_E_CUDA, rc == -2 ? "mppi_set_mlp has not been called" : "MLP rollout launch failed");
        h->tm.launches += mlp_launches_per_tick(h->mlp);
        if (h->timing) CK(h, cudaEventRecord(h->ev[1], h->stream));
        TickArgs a = h->args;
        a.S = h->d_S; a.eps = d_eps;
        a.flags = F_UPDATE | F_FROM_S;      // K2 repeats step 1 (same result as in the MLP kernel) and persists the index
        int rc2 = launch_update(h, a, d_eps != nullptr);
        if (rc2 != MPPI_OK) return rc2;
    } else if (h->strict) {
        int rc = strict_costs(h, x0, d_eps, h->keep_costs ? h->d_Sc : nullptr, &strict_idx_after);
        if (rc != MPPI_OK) return rc;
        const int idx_after = strict_idx_after;
        if (h->timing) CK(h, cudaEventRecord(h->ev[1], h->stream));
        TickArgs a = h->args;
        a.S = h->d_S; a.NC = h->d_NC; a.eps = d_eps;
        a.flags = F_UPDATE | F_FROM_S | F_HOST_IDX;
        a.idx_host = idx_after;
        rc = launch_update(h, a, d_eps != nullptr);
        if (rc != MPPI_OK) return rc;
    } else {
        TickArgs a = h->args;
        a.eps = d_eps; a.S = h->keep_costs ? h->d_Sc : nullptr;
        a.flags = F_UPDATE | (h->keep_costs ? F_WRITE_S : 0);
        if (h->timing) CK(h, cudaEventRecord(h->ev[1], h->stream));
        int rc = launch_update(h, a, d_eps != nullptr);
        if (rc != MPPI_OK) return rc;
    }
    if (h->timing) CK(h, cudaEventRecord(h->ev[2], h->stream));
    if (sync_out || h->timing) {
        CK(h, cudaStreamSynchronize(h->stream));
        if (h->timing) {
            cudaEventElapsedTime(&h->tm.last_step_ms, h->ev[0], h->ev[2]);
            cudaEventElapsedTime(&h->tm.last_rollout_ms, h->ev[0], h->ev[1]);
            cudaEventElapsedTime(&h->tm.last_update_ms, h->ev[1], h->ev[2]);
        }
        if (int rc = check_tick_faults(h)) return rc;
        if (strict_idx_after >= 0) { h->idx_mirror = strict_idx_after; h->idx_mirror_ok = true; }     // the applied tick persisted it
        if (u0_out) { u0_out[0] = h->h_out[0]; u0_out[1] = h->h_out[1]; }
        if (useq_out) std::memcpy(useq_out, h->h_out + MPPI_OUT_HDR, sizeof(float) * 2 * h->cfg.T);
    }
    return MPPI_OK;
}

int mppi_step(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick,
              float *u0_out, float *useq_out) {
    return step_common(h, x0, d_eps, seed, tick, true, u0_out, useq_out);
}

int mppi_step_async(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick) {
    return step_common(h, x0, d_eps, seed, tick, false, nullptr, nullptr);
}

int mppi_rollout_costs(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick, float *d_S) {
    if (!h || !x0 || !d_S) return MPPI_E_BADARG;
    if (!h->have_path) return fail(h, MPPI_E_STATE, "mppi_set_ref_path has not been called");
    if (h->cfg.n_robots != 1) return MPPI_E_BADARG;
    if (int rc = scene_refused(h, "mppi_rollout_costs")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    set_x0(h, x0);
    set_seed(h, seed, tick);
    if (h->mlp) {
        if (mlp_rollout_costs(h->mlp, h->args, h->sum, d_eps, d_S, h->stream) != 0) return fail(h, MPPI_E_CUDA, "MLP rollout failed");
        h->tm.launches += mlp_launches_per_tick(h->mlp);
        TickArgs a = h->args;
        a.flags = F_IDX_ONLY;
        dim3 grid(1, 1);
        if (a.trace) h->trace_grid = 1;
        CK(h, mppi_launch_tick(a, MPPI_MODEL_DIFFDRIVE, MPPI_COLLISION_NONE, MPPI_COSTKIND_PATH, h->sum, false, false, grid, h->stream));
        h->tm.launches++;
    } else if (h->strict) {
        int idx_after = 0;
        int rc = strict_costs(h, x0, d_eps, d_S, &idx_after);
        if (rc != MPPI_OK) return rc;
        CK(h, cudaMemcpyAsync(h->d_idx, &idx_after, sizeof(int), cudaMemcpyHostToDevice, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));            // idx_after is a stack variable
        h->idx_mirror = idx_after; h->idx_mirror_ok = true;
    } else {
        TickArgs a = h->args;
        a.eps = d_eps; a.S = d_S; a.flags = F_WRITE_S;
        dim3 grid(h->grid_x, 1);
        if (a.trace) h->trace_grid = (int)grid.x;
        CK(h, mppi_launch_tick(a, h->cfg.model, h->cfg.collision, h->cfg.cost_kind, h->sum, d_eps != nullptr, false, grid, h->stream));
        h->tm.launches++;
    }
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_reduce_update(mppi_handle_t h, const float *d_S, const float *d_eps, uint64_t seed, uint64_t tick,
                       float *u0_out, float *useq_out, float *w_eps_out) {
    if (!h || !d_S) return MPPI_E_BADARG;
    if (!h->have_path) return fail(h, MPPI_E_STATE, "mppi_set_ref_path has not been called");
    if (h->cfg.n_robots != 1) return MPPI_E_BADARG;
    if (int rc = scene_refused(h, "mppi_reduce_update")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    set_seed(h, seed, tick);
    TickArgs a = h->args;
    a.eps = d_eps; a.S = const_cast<float *>(d_S);
    a.flags = F_UPDATE | F_FROM_S | F_KEEP_IDX | F_HOST_IDX;
    a.idx_host = 0;
    int rc = launch_update(h, a, d_eps != nullptr);
    if (rc != MPPI_OK) return rc;
    CK(h, cudaStreamSynchronize(h->stream));
    if (int rc2 = check_tick_faults(h)) return rc2;
    if (u0_out) { u0_out[0] = h->h_out[0]; u0_out[1] = h->h_out[1]; }
    if (useq_out) std::memcpy(useq_out, h->h_out + MPPI_OUT_HDR, sizeof(float) * 2 * h->cfg.T);
    if (w_eps_out) std::memcpy(w_eps_out, h->h_out + MPPI_OUT_HDR + 2 * MPPI_MAX_T, sizeof(float) * 2 * h->cfg.T);
    return MPPI_OK;
}

int mppi_generate_noise(mppi_handle_t h, uint64_t seed, uint64_t tick, float *d_eps_out) {
    return mppi_generate_noise_robot(h, seed, tick, 0, d_eps_out);
}

int mppi_generate_noise_robot(mppi_handle_t h, uint64_t seed, uint64_t tick, int32_t robot, float *d_eps_out) {
    if (!h || !d_eps_out || robot < 0 || robot >= h->cfg.n_robots) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    set_seed(h, seed, tick);
    CK(h, mppi_launch_noise(h->args, d_eps_out, robot, h->stream));
    h->tm.launches++;
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_get_trajectories(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick,
                          float *optimal_out, float *d_sampled_out) {
    if (!h || !x0) return MPPI_E_BADARG;
    if (h->cfg.n_robots != 1 || h->mlp) return fail(h, MPPI_E_UNSUPPORTED, "trajectories: single-robot analytic models only");
    if (int rc = scene_refused(h, "mppi_get_trajectories")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    set_x0(h, x0);
    set_seed(h, seed, tick);
    TickArgs a = h->args;
    a.eps = d_eps;
    const int nx = h->nx, T = h->cfg.T;
    if (optimal_out && !h->d_opt) CK(h, gmalloc(h, &h->d_opt, sizeof(float) * MPPI_MAX_T * 4));
    CK(h, mppi_launch_traj(a, h->cfg.model, h->d_out, optimal_out ? h->d_opt : nullptr, d_sampled_out, nullptr, 0, 1, h->stream));
    h->tm.launches++;
    if (optimal_out) CK(h, cudaMemcpyAsync(optimal_out, h->d_opt, sizeof(float) * T * nx, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_set_keep_costs(mppi_handle_t h, int32_t on) {
    if (!h) return MPPI_E_BADARG;
    if (h->cfg.n_robots != 1) return fail(h, MPPI_E_UNSUPPORTED, "per-sample costs are kept for single-robot handles");
    CK(h, cudaSetDevice(h->cfg.device));
    if (on && !h->d_Sc) {
        const int K = h->cfg.K;
        CK(h, gmalloc(h, &h->d_Sc, sizeof(float) * K));
        CK(h, gmalloc(h, &h->d_Ssorted, sizeof(float) * K));
        CK(h, gmalloc(h, &h->d_sorted_idx, sizeof(int) * K));
        CK(h, gmalloc(h, &h->d_iota, sizeof(int) * K));
        h->sort_temp_bytes = mppi_sort_costs_temp_bytes(K);
        CK(h, gmalloc(h, &h->d_sort_temp, h->sort_temp_bytes ? h->sort_temp_bytes : 16));
    }
    h->keep_costs = on != 0;
    return MPPI_OK;
}

int mppi_get_top_trajectories(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick,
                              int32_t n_top, int32_t index_shift, float *optimal_out, float *d_traj_out,
                              int32_t *d_idx_out, float *d_cost_out) {
    if (!h || !x0 || n_top < 1 || n_top > h->cfg.K || !d_traj_out || index_shift < 0 || index_shift > 1) return MPPI_E_BADARG;
    if (h->cfg.n_robots != 1 || h->mlp) return fail(h, MPPI_E_UNSUPPORTED, "trajectories: single-robot analytic models only");
    if (!h->keep_costs || !h->d_Sc) return fail(h, MPPI_E_STATE, "call mppi_set_keep_costs(h, 1) before the tick");
    if (int rc = scene_refused(h, "mppi_get_top_trajectories")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    set_x0(h, x0);
    set_seed(h, seed, tick);
    TickArgs a = h->args;
    a.eps = d_eps;
    const int nx = h->nx, T = h->cfg.T;
    CK(h, mppi_sort_costs(h->d_Sc, h->cfg.K, h->d_Ssorted, h->d_sorted_idx, h->d_iota, h->d_sort_temp, h->sort_temp_bytes, h->stream));
    if (optimal_out && !h->d_opt) CK(h, gmalloc(h, &h->d_opt, sizeof(float) * MPPI_MAX_T * 4));
    CK(h, mppi_launch_traj(a, h->cfg.model, h->d_out, optimal_out ? h->d_opt : nullptr, d_traj_out, h->d_sorted_idx, n_top,
                           index_shift, h->stream));
    h->tm.launches += 3;
    if (d_idx_out) CK(h, cudaMemcpyAsync(d_idx_out, h->d_sorted_idx, sizeof(int) * n_top, cudaMemcpyDeviceToDevice, h->stream));
    if (d_cost_out) CK(h, cudaMemcpyAsync(d_cost_out, h->d_Ssorted, sizeof(float) * n_top, cudaMemcpyDeviceToDevice, h->stream));
    if (optimal_out) CK(h, cudaMemcpyAsync(optimal_out, h->d_opt, sizeof(float) * T * nx, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_run_closed_loop(mppi_handle_t h, const double *x0, int32_t n_ticks, uint64_t seed, uint64_t tick0,
                         int32_t plant, float *states_out, float *controls_out) {
    if (!h || !x0 || n_ticks < 1 || !states_out || plant < 0 || plant > 1) return MPPI_E_BADARG;
    if (!h->have_path) return fail(h, MPPI_E_STATE, "mppi_set_ref_path has not been called");
    if (h->strict || h->mlp || h->world > 1)
        return fail(h, MPPI_E_UNSUPPORTED, "closed loop: frozen waypoint mode, one GPU, analytic dynamics");
    if (plant == 1 && h->cfg.model != MPPI_MODEL_BICYCLE) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    const int nx = h->nx, R = h->cfg.n_robots;
    const size_t log_floats = ((size_t)4 * (n_ticks + 1) + (size_t)2 * n_ticks) * R;
    if (h->plant_log_cap < n_ticks) {
        CK(h, cudaStreamSynchronize(h->stream));
        gfree(h, h->d_plant_log); h->d_plant_log = nullptr;
        if (h->loop_graph) { cudaGraphExecDestroy(h->loop_graph); h->loop_graph = nullptr; }     // it holds the old pointer
        CK(h, gmalloc(h, &h->d_plant_log, sizeof(float) * log_floats));
        CK(h, cudaMemset(h->d_plant_log, 0, sizeof(float) * log_floats));
        h->plant_log_cap = n_ticks;
    }
    if (!h->d_x0) CK(h, gmalloc(h, &h->d_x0, sizeof(float) * 4 * R));
    if (!h->d_loop) {
        CK(h, gmalloc(h, &h->d_loop, sizeof(unsigned) * 4));
        CK(h, cudaMemset(h->d_loop, 0, sizeof(unsigned) * 4));
    }
    std::vector<float> xs((size_t)4 * R, 0.f);
    for (int r = 0; r < R; ++r)
        for (int i = 0; i < nx; ++i) xs[(size_t)4 * r + i] = (float)x0[(size_t)r * nx + i];
    const unsigned loop0[4] = {(unsigned)tick0, (unsigned)tick0, 0u, 0u};          // running tick, first tick, ticket
    CK(h, cudaMemcpyAsync(h->d_x0, xs.data(), sizeof(float) * 4 * R, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(h->d_plant_log, xs.data(), sizeof(float) * 4 * R, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(h->d_loop, loop0, sizeof(loop0), cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));                 // xs / loop0 are stack / heap temporaries

    // The n ticks as ONE CUDA graph of n identical kernel nodes: every launch carries the same arguments (the running tick
    // and the log row come from d_loop, advanced by each launch's last CTA), so the instantiated graph is reused by every
    // later call with the same (n_ticks, plant, seed, sample-cost flag, obstacle set); MPPI_CLOSED_LOOP_GRAPH=0 falls back
    // to n stream launches (A/B measurements).  Per-robot goals / obstacles are read from the handle's table, whose pointer
    // never changes: re-installing them between calls does not re-instantiate the graph.
    set_seed(h, seed, 0);
    TickArgs a = h->args;
    a.x0_dev = h->d_x0; a.eps = nullptr; a.S = nullptr; a.flags = F_UPDATE;
    if (R > 1) a.out_host = nullptr;
    a.plant_state = h->d_x0; a.plant_log = h->d_plant_log; a.plant_mode = plant; a.plant_tick = 0; a.plant_n = n_ticks;
    a.loop_state = h->d_loop; a.loop_ticket = h->d_loop + 2;
    static const bool use_graph = [] { const char *e = std::getenv("MPPI_CLOSED_LOOP_GRAPH"); return !(e && e[0] == '0'); }();
    const bool same = h->loop_graph && h->loop_graph_n == n_ticks && std::memcmp(&h->loop_graph_args, &a, sizeof(TickArgs)) == 0;
    if (use_graph && !same) {
        if (h->loop_graph) { cudaGraphExecDestroy(h->loop_graph); h->loop_graph = nullptr; }
        cudaGraph_t g = nullptr;
        const int launches_before = h->tm.launches;
        // captured on a private stream (the caller's may be the legacy default stream, which cannot capture); the graph
        // itself is launched on the handle's stream
        if (!h->cap_stream) CK(h, cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
        cudaStream_t user_stream = h->stream;
        if (cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            return fail(h, MPPI_E_CUDA, "closed loop: cannot begin stream capture");
        }
        h->stream = h->cap_stream;
        int rc = MPPI_OK;
        for (int i = 0; i < n_ticks && rc == MPPI_OK; ++i) rc = launch_update(h, a, false);
        h->stream = user_stream;
        cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &g);
        h->tm.launches = launches_before;                     // captured, not launched yet
        if (rc != MPPI_OK || ce != cudaSuccess) { if (g) cudaGraphDestroy(g); cudaGetLastError(); return fail(h, MPPI_E_CUDA, "closed loop: graph capture failed"); }
        ce = cudaGraphInstantiate(&h->loop_graph, g, 0);
        cudaGraphDestroy(g);
        if (ce != cudaSuccess) { h->loop_graph = nullptr; return fail(h, MPPI_E_CUDA, "closed loop: graph instantiation failed"); }
        h->loop_graph_n = n_ticks; h->loop_graph_args = a;
    }
    if (use_graph) {
        CK(h, cudaGraphLaunch(h->loop_graph, h->stream));
        h->tm.launches += n_ticks;
    } else {
        for (int i = 0; i < n_ticks; ++i) {
            int rc = launch_update(h, a, false);
            if (rc != MPPI_OK) return rc;
        }
    }
    std::vector<float> log(log_floats);
    CK(h, cudaMemcpyAsync(log.data(), h->d_plant_log, sizeof(float) * log_floats, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i < (size_t)(n_ticks + 1) * R; ++i)
        for (int j = 0; j < nx; ++j) states_out[i * nx + j] = log[4 * i + j];
    if (controls_out) std::memcpy(controls_out, log.data() + (size_t)4 * (n_ticks + 1) * R, sizeof(float) * 2 * n_ticks * R);
    return check_tick_faults(h);
}

int mppi_step_batched(mppi_handle_t h, const float *d_x0, uint64_t seed, uint64_t tick, float *d_u0_out) {
    if (!h || !d_x0) return MPPI_E_BADARG;
    if (!h->have_path) return fail(h, MPPI_E_STATE, "mppi_set_ref_path has not been called");
    if (h->strict || h->mlp) return MPPI_E_UNSUPPORTED;
    CK(h, cudaSetDevice(h->cfg.device));
    set_seed(h, seed, tick);
    TickArgs a = h->args;
    // (R, nx) -> padded (R, 4) staging so every robot's state is one aligned read
    if (!h->d_x0) CK(h, gmalloc(h, &h->d_x0, sizeof(float) * 4 * h->cfg.n_robots));
    CK(h, cudaMemcpy2DAsync(h->d_x0, 4 * sizeof(float), d_x0, h->nx * sizeof(float), h->nx * sizeof(float),
                            h->cfg.n_robots, cudaMemcpyDeviceToDevice, h->stream));
    a.x0_dev = h->d_x0; a.eps = nullptr; a.S = nullptr; a.flags = F_UPDATE; a.u0_out = d_u0_out;
    a.out_host = nullptr;
    const bool scene = a.scene_mask != 0;
    const int stash = scene ? h->scene_stash : h->stash ? 1 : 0;
    dim3 grid(stash ? h->grid_x_stash : h->grid_x, h->cfg.n_robots);
    if (a.trace) h->trace_grid = (int)grid.x;
    CK(h, mppi_launch_tick(a, h->cfg.model, h->cfg.collision, h->cfg.cost_kind, h->sum, false, stash, grid, h->stream, scene));
    h->tm.launches++;
    return MPPI_OK;
}

int mppi_comm_get_unique_id(void *out128) {
    if (!out128) return MPPI_E_BADARG;
    if (!g_nccl.load()) return MPPI_E_NCCL;
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) return MPPI_E_NCCL;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    std::memcpy(out128, &id, 128);
    return MPPI_OK;
}

int mppi_comm_init(mppi_handle_t h, const void *uid, int32_t rank, int32_t world) {
    if (!h || !uid || world < 1 || rank < 0 || rank >= world) return MPPI_E_BADARG;
    if (h->cfg.n_robots != 1 || h->strict) return fail(h, MPPI_E_UNSUPPORTED, "sample sharding needs frozen mode, one robot");
    if (int rc = scene_refused(h, "mppi_comm_init")) return rc;
    if (!g_nccl.load()) return fail(h, MPPI_E_NCCL, "cannot load libnccl.so.2");
    CK(h, cudaSetDevice(h->cfg.device));
    ncclUniqueId id;
    std::memcpy(&id, uid, 128);
    ncclResult_t r = g_nccl.CommInitRank(&h->comm, world, id, rank);
    if (r != ncclSuccess) { h->err = g_nccl.GetErrorString(r); return MPPI_E_NCCL; }
    h->rank = rank; h->world = world;
    const size_t nf = MPPI_NF(h->cfg.T);
    CK(h, gmalloc(h, &h->d_send, sizeof(float) * nf));
    CK(h, gmalloc(h, &h->d_recv, sizeof(float) * nf * world));
    return MPPI_OK;
}

int mppi_comm_p2p_export(mppi_handle_t h, int32_t world, void *out64) {
    if (!h || !out64 || world < 2 || world > MPPI_MAX_PEERS) return MPPI_E_BADARG;
    if (h->cfg.n_robots != 1 || h->strict) return fail(h, MPPI_E_UNSUPPORTED, "sample sharding needs frozen mode, one robot");
    if (int rc = scene_refused(h, "mppi_comm_p2p_export")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    if (!h->d_xchg) {
        CK(h, gmalloc(h, &h->d_xchg, sizeof(unsigned long long) * MPPI_XCHG_TOTAL));
        CK(h, cudaMemset(h->d_xchg, 0, sizeof(unsigned long long) * MPPI_XCHG_TOTAL));
        CK(h, cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t ih;
    CK(h, cudaIpcGetMemHandle(&ih, h->d_xchg));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    std::memcpy(out64, &ih, 64);
    return MPPI_OK;
}

int mppi_comm_p2p_open(mppi_handle_t h, const void *handles, int32_t rank, int32_t world) {
    if (!h || !handles || world < 2 || world > MPPI_MAX_PEERS || rank < 0 || rank >= world) return MPPI_E_BADARG;
    if (!h->d_xchg) return fail(h, MPPI_E_STATE, "call mppi_comm_p2p_export first");
    if (int rc = scene_refused(h, "mppi_comm_p2p_open")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    for (int p = 0; p < world; ++p) {
        if (p == rank) { h->peer_buf[p] = h->d_xchg; continue; }
        cudaIpcMemHandle_t ih;
        std::memcpy(&ih, (const char *)handles + 64 * p, 64);
        void *ptr = nullptr;
        CK(h, cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess));
        h->peer_buf[p] = (unsigned long long *)ptr;
    }
    h->rank = rank; h->world = world; h->p2p = true; h->p2p_seq = 0; h->p2p_barrier_count = 0;
    if (const char *env = std::getenv("MPPI_P2P_TIMEOUT_MS")) h->p2p_timeout_ms = (unsigned)std::max(1, std::atoi(env));
    h->h_out[MPPI_OUT_PEER_TIMEOUT] = 0.f;              // no stale peer-timeout report from an earlier communicator
    CK(h, cudaMemsetAsync(h->d_out + MPPI_OUT_PEER_TIMEOUT, 0, sizeof(float), h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

int mppi_set_trace(mppi_handle_t h, int32_t on) {
    if (!h) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    if (on && !h->d_trace) {
        h->trace_n = 2 * (std::max(std::max(h->grid_x, h->grid_x_stash), h->grid_x_tpar) + 1);
        CK(h, gmalloc(h, &h->d_trace, sizeof(unsigned long long) * h->trace_n));
        CK(h, cudaMemset(h->d_trace, 0, sizeof(unsigned long long) * h->trace_n));
    }
    h->args.trace = on ? h->d_trace : nullptr;
    return MPPI_OK;
}

int mppi_get_trace(mppi_handle_t h, uint64_t *out, int32_t capacity, int32_t *n_ctas_out) {
    if (!h || !out || !n_ctas_out || capacity < 4) return MPPI_E_BADARG;
    if (!h->d_trace) return fail(h, MPPI_E_STATE, "call mppi_set_trace(h, 1) before the tick");
    CK(h, cudaSetDevice(h->cfg.device));
    const int n = std::min(capacity, h->trace_n);
    CK(h, cudaMemcpyAsync(out, h->d_trace, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->trace_grid == 0) return fail(h, MPPI_E_STATE, "no tick has been traced since mppi_set_trace(h, 1)");
    *n_ctas_out = h->trace_grid;
    return MPPI_OK;
}

int mppi_debug_check_guards(mppi_handle_t h) {
    if (!h) return MPPI_E_BADARG;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    unsigned char g[MPPI_GUARD_BYTES];
    int bad = 0;
    for (const auto &b : h->guards) {
        CK(h, cudaMemcpy(g, (const char *)b.first + b.second, MPPI_GUARD_BYTES, cudaMemcpyDeviceToHost));
        for (int i = 0; i < MPPI_GUARD_BYTES; ++i)
            if (g[i] != 0xA5) { ++bad; break; }
    }
    if (h->mlp) bad += mlp_check_guards(h->mlp);
    return bad;                                           // number of buffers whose guard zone was overwritten (0 = clean)
}

int mppi_comm_p2p_barrier(mppi_handle_t h) {
    if (!h) return MPPI_E_BADARG;
    if (!h->p2p || h->world < 2) return fail(h, MPPI_E_STATE, "no fused exchange on this handle");
    if (int rc = scene_refused(h, "mppi_comm_p2p_barrier")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    TickArgs b = h->args;
    for (int p = 0; p < h->world; ++p) b.peer_buf[p] = h->peer_buf[p];
    b.p2p_rank = h->rank; b.p2p_world = h->world; b.p2p_timeout_ms = h->p2p_timeout_ms;
    CK(h, mppi_launch_p2p_barrier(b, ++h->p2p_barrier_count, h->stream));
    h->tm.launches++;
    return MPPI_OK;
}

int mppi_comm_p2p_trace(mppi_handle_t h, uint64_t stamps_out[4]) {
    if (!h || !stamps_out) return MPPI_E_BADARG;
    if (!h->p2p || !h->d_xchg) return fail(h, MPPI_E_STATE, "no fused exchange on this handle");
    if (int rc = scene_refused(h, "mppi_comm_p2p_trace")) return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(stamps_out, h->d_xchg + MPPI_XCHG_WORDS, sizeof(uint64_t) * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return MPPI_OK;
}

}  // extern "C"
