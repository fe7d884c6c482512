// sm_100a kernels of the MPPI tick.
//   mppi_tick_kernel   K1+K2 fused: step-1 index update, Philox noise, K x T rollout with state in
//                      registers, costs, block-local soft-min, weighted-noise reduction, last-block
//                      log-sum-exp merge, filter, nominal update and shift -- one launch per tick.
//   mppi_strict_kernel literal waypoint-index mutation (quirk Q3) by the multi-pass rule.
//   mppi_merge_kernel  merge of per-GPU triples after the all-gather + finalize.
//   mppi_noise_kernel  exports the exact Philox noise tensor.
#include "mppi_device.cuh"
#include "mppi_launch.h"

#include <algorithm>
#include <array>
#include <atomic>
#include <mutex>
#include <utility>

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// lexicographic (ncoll, smooth) minimum over a warp
__device__ __forceinline__ void warp_lexmin(int &n, float &s) {
    const int nmin = __reduce_min_sync(0xffffffffu, n);
    float c = (n == nmin) ? s : CUDART_INF_F;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c = fminf(c, __shfl_xor_sync(0xffffffffu, c, o));
    n = nmin; s = c;
}

// exp(-((n - n0) * 1e10 + (s - s0)) / temperature): the weight of a (ncoll, smooth) cost
// relative to the reference cost (n0, s0), with the collision penalty kept out of the float sum.
__device__ __forceinline__ float rel_weight(int n, float s, int n0, float s0, float inv_temp) {
    const float d = (float)(n - n0) * MPPI_PENALTY + (s - s0);
    return __expf(-d * inv_temp);
}

struct MergeSmem {
    float red_s[MPPI_WARPS];
    int red_n[MPPI_WARPS];
    float col[4 + 2 * MPPI_MAX_T];      // merged triple (same layout as a partial)
    float weps[2 * MPPI_MAX_T];
    float upre[2 * MPPI_MAX_T];
};

// Merges P partials (layout MPPI_NF) into ms.col by the log-sum-exp rule of SURVEY.md 8e.  Runs in ONE CTA on the
// critical path of every tick, so it is organised for memory-level parallelism: the P scale factors are computed
// once (P exps, spread over the threads) into shared memory; then the CTA splits into G groups of NF/2 threads, a
// thread owns one float2 COLUMN PAIR of the partial layout and streams every G-th partial with 8 independent
// coalesced 8-byte loads in flight; the G group sums meet in shared memory.  `sc` is scratch lent by the caller:
// MPPI_MERGE_SCRATCH floats (the first MPPI_MERGE_TILE hold scale factors, the rest the group sums).
#define MPPI_MERGE_TWO_LEVEL_MIN 64     // smaller grids keep the single merge (one L2 round trip either way)
#define MPPI_MERGE_TILE 1000
#define MPPI_MERGE_GROUPS 4
#define MPPI_MERGE_SCRATCH (MPPI_MERGE_TILE + MPPI_MERGE_GROUPS * MPPI_NF_MAX)      // 2040 floats <= the 8 KB warpN region
static_assert(4 * MPPI_BLOCK <= MPPI_MERGE_SCRATCH, "merge fast path: group sums must fit the scratch");
__device__ void merge_partials(const TickArgs &a, const float *parts, int P, MergeSmem &ms, float *sc, int stride = 0) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NF = MPPI_NF(a.T);
    if (stride == 0) stride = NF;
    int n = INT_MAX;
    float s = CUDART_INF_F;
    int my_n = INT_MAX;                                       // key of this thread's first partial, kept for its weight
    float my_s = CUDART_INF_F;
    for (int p = tid; p < P; p += MPPI_BLOCK) {
        const int pn = __float_as_int(__ldcg(parts + (size_t)p * stride));
        const float ps = __ldcg(parts + (size_t)p * stride + 1);
        if (p == tid) { my_n = pn; my_s = ps; }
        if (pn < n || (pn == n && ps < s)) { n = pn; s = ps; }
    }
    warp_lexmin(n, s);
    if (lane == 0) { ms.red_n[warp] = n; ms.red_s[warp] = s; }
    __syncthreads();
    n = ms.red_n[0]; s = ms.red_s[0];
#pragma unroll
    for (int w = 1; w < MPPI_WARPS; ++w) {
        const int wn = ms.red_n[w]; const float ws = ms.red_s[w];
        if (wn < n || (wn == n && ws < s)) { n = wn; s = ws; }
    }
    // ---- fast path (even horizon: NF % 4 == 0, partials 16-byte aligned): a thread owns one float4 COLUMN QUAD, the CTA
    // splits into G = MPPI_BLOCK / (NF/4) groups (9 at T = 50) and a group's thread streams every G-th partial with up
    // to 12 independent 16-byte loads in flight: ~P/(12 G) dependent L2 round trips (3 at P = 296) instead of P/32
    if ((NF & 3) == 0 && (stride & 3) == 0 && MPPI_BLOCK / (NF >> 2) >= 2 && P <= MPPI_MERGE_TILE) {
        const int NQ = NF >> 2, G4 = min(MPPI_BLOCK / NQ, 16);
        const int g4 = tid / NQ, cq = tid - g4 * NQ;
        __syncthreads();
        if (tid < P) sc[tid] = rel_weight(my_n, my_s, n, s, a.inv_temp);      // no second L2 round trip for the first MPPI_BLOCK keys
        for (int p = tid + MPPI_BLOCK; p < P; p += MPPI_BLOCK) {
            const float *pp = parts + (size_t)p * stride;
            sc[p] = rel_weight(__float_as_int(__ldcg(pp)), __ldcg(pp + 1), n, s, a.inv_temp);
        }
        __syncthreads();
        float4 acc4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g4 < G4) {
            const float4 *col = reinterpret_cast<const float4 *>(parts) + cq;
            const size_t st4 = (size_t)stride >> 2;
            int p = g4;
            for (; p + 11 * G4 < P; p += 12 * G4) {
                float4 v[12];
#pragma unroll
                for (int i = 0; i < 12; ++i) v[i] = __ldcg(col + (size_t)(p + i * G4) * st4);
#pragma unroll
                for (int i = 0; i < 12; ++i) {
                    const float w = sc[p + i * G4];
                    acc4.x = fmaf(w, v[i].x, acc4.x); acc4.y = fmaf(w, v[i].y, acc4.y);
                    acc4.z = fmaf(w, v[i].z, acc4.z); acc4.w = fmaf(cq == 0 ? w * w : w, v[i].w, acc4.w);
                }
            }
            for (; p < P; p += G4) {
                const float4 v = __ldcg(col + (size_t)p * st4);
                const float w = sc[p];
                acc4.x = fmaf(w, v.x, acc4.x); acc4.y = fmaf(w, v.y, acc4.y);
                acc4.z = fmaf(w, v.z, acc4.z); acc4.w = fmaf(cq == 0 ? w * w : w, v.w, acc4.w);
            }
        }
        __syncthreads();                                      // every thread is done with sc[]: reuse it for the group sums
        float *red4 = sc;                                     // [G4][NF]: G4 * NF <= (MPPI_BLOCK / NQ) * 4 NQ = 4 MPPI_BLOCK floats... of which <= 1024 at 256 threads
        MPPI_DCHECK(G4 * NF <= MPPI_MERGE_SCRATCH && P <= MPPI_MERGE_TILE);
        if (g4 < G4) *reinterpret_cast<float4 *>(red4 + (size_t)g4 * NF + 4 * cq) = acc4;
        __syncthreads();
        for (int c = 2 + tid; c < NF; c += MPPI_BLOCK) {
            float t = red4[c];
            for (int gg = 1; gg < G4; ++gg) t += red4[(size_t)gg * NF + c];
            ms.col[c] = t;
        }
        if (tid == 0) { ms.col[0] = __int_as_float(n); ms.col[1] = s; }
        __syncthreads();
        return;
    }
    // column pairs: pair 0 = (n, s) is the key handled above, pair 1 = (eta, sum w^2), pairs 2.. = N[t][0..1]
    const int NP = NF >> 1;                                   // NF = 4 + 2T is even; every partial is 8-byte aligned
    const int G = min(MPPI_MERGE_GROUPS, MPPI_BLOCK / NP);    // T <= 126 -> NP <= 128 -> G >= 2; T = 127, 128 -> G = 1
    const int PPT = (NP + MPPI_BLOCK - 1) / MPPI_BLOCK;       // pairs per thread when one group does not cover them (G = 1)
    const int g = tid / NP, cp = tid - g * NP;
    const bool live = (G > 1) ? (g < G && cp >= 1) : true;
    float2 acc[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
    float *red = sc + MPPI_MERGE_TILE;
    for (int base = 0; base < P; base += MPPI_MERGE_TILE) {
        const int np = min(MPPI_MERGE_TILE, P - base);
        __syncthreads();
        for (int p = tid; p < np; p += MPPI_BLOCK) {
            const float *pp = parts + (size_t)(base + p) * stride;
            sc[p] = rel_weight(__float_as_int(__ldcg(pp)), __ldcg(pp + 1), n, s, a.inv_temp);
        }
        __syncthreads();
        if (G > 1) {
            if (live) {
                const float2 *col = reinterpret_cast<const float2 *>(parts + (size_t)base * stride) + cp;
                const size_t st2 = (size_t)stride >> 1;               // stride is even (NF or MPPI_NF_MAX)
                int p = g;
                for (; p + 7 * G < np; p += 8 * G) {
                    float2 v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = __ldcg(col + (size_t)(p + i * G) * st2);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float w = sc[p + i * G];
                        acc[0].x = fmaf(w, v[i].x, acc[0].x);
                        acc[0].y = fmaf(cp == 1 ? w * w : w, v[i].y, acc[0].y);
                    }
                }
                for (; p < np; p += G) {
                    const float2 v = __ldcg(col + (size_t)p * st2);
                    const float w = sc[p];
                    acc[0].x = fmaf(w, v.x, acc[0].x);
                    acc[0].y = fmaf(cp == 1 ? w * w : w, v.y, acc[0].y);
                }
            }
        } else {
            for (int j = 0; j < PPT && j < 2; ++j) {
                const int c2 = tid + j * MPPI_BLOCK;
                if (c2 < 1 || c2 >= NP) continue;
                const float2 *col = reinterpret_cast<const float2 *>(parts + (size_t)base * stride) + c2;
                const size_t st2 = (size_t)stride >> 1;
                for (int p = 0; p < np; ++p) {
                    const float2 v = __ldcg(col + (size_t)p * st2);
                    const float w = sc[p];
                    acc[j].x = fmaf(w, v.x, acc[j].x);
                    acc[j].y = fmaf(c2 == 1 ? w * w : w, v.y, acc[j].y);
                }
            }
        }
    }
    if (G > 1) {
        if (live) { red[g * MPPI_NF_MAX + 2 * cp] = acc[0].x; red[g * MPPI_NF_MAX + 2 * cp + 1] = acc[0].y; }
        __syncthreads();
        for (int c = 2 + tid; c < NF; c += MPPI_BLOCK) {
            float t = red[c];
            for (int gg = 1; gg < G; ++gg) t += red[gg * MPPI_NF_MAX + c];
            ms.col[c] = t;
        }
    } else {
        for (int j = 0; j < 2; ++j) {
            const int c2 = tid + j * MPPI_BLOCK;
            if (c2 >= 1 && c2 < NP) { ms.col[2 * c2] = acc[j].x; ms.col[2 * c2 + 1] = acc[j].y; }
        }
    }
    if (tid == 0) { ms.col[0] = __int_as_float(n); ms.col[1] = s; }
    __syncthreads();
}

// This tick's rows of `robot` in the closed-loop log: the plant state after the step, and the control applied.
__device__ __forceinline__ void plant_log_rows(const TickArgs &a, int robot, float *&lg, float *&lu) {
    const int R = gridDim.y;
    const int pt = a.loop_state ? (int)(__ldcg(a.loop_state) - __ldcg(a.loop_state + 1)) : a.plant_tick;
    lg = a.plant_log + 4 * ((size_t)(pt + 1) * R + robot);
    lu = a.plant_log + 4 * (size_t)(a.plant_n + 1) * R + 2 * ((size_t)pt * R + robot);
}

// A13-A15 + Q8 from the merged triple in ms.col: normalise, filter, update, shift, publish.
__device__ void finalize_tick(const TickArgs &a, int robot, int idx_new, MergeSmem &ms) {
    const int tid = threadIdx.x, T = a.T;
    const float eta = ms.col[2];
    const float inv_eta = 1.f / eta;
    float *U = a.U + (size_t)robot * T * 2;
    float *out = a.out + (size_t)robot * MPPI_OUT_STRIDE;
    // eta = sum of exp(-(S - min S)/tau) >= 1 whenever the costs are finite.  NaN / inf costs (a NaN observed state, a
    // learned residual that diverged, a missed hand-off in the learned-dynamics kernel) must not poison the nominal for
    // good: the tick is NOT applied and the fault is reported to the host (MPPI_E_NUMERIC).  In a fleet only this robot's
    // tick is refused: its u0 row and this tick's plant-log rows read NaN (not the previous tick's control), its nominal,
    // waypoint index and plant state stay as they were; every other robot owns its CTAs and is unaffected.
    if (!(eta > 0.f && eta < CUDART_INF_F)) {
        if (tid == 0) {
            out[MPPI_OUT_FAULT] = 1.f;
            if (robot == 0 && a.out_host) a.out_host[MPPI_OUT_FAULT] = 1.f;
            if (a.u0_out) { a.u0_out[2 * robot] = CUDART_NAN_F; a.u0_out[2 * robot + 1] = CUDART_NAN_F; }
            if (a.plant_state) {
                float *lg, *lu;
                plant_log_rows(a, robot, lg, lu);
                lg[0] = lg[1] = lg[2] = lg[3] = CUDART_NAN_F;
                lu[0] = lu[1] = CUDART_NAN_F;
            }
        }
        return;
    }
    for (int c = tid; c < 2 * T; c += MPPI_BLOCK) ms.weps[c] = ms.col[4 + c] * inv_eta;
    __syncthreads();
    for (int c = tid; c < 2 * T; c += MPPI_BLOCK) {
        const int n = c >> 1, u = c & 1;
        const float *Mrow = a.M + (size_t)n * T;
        float f = 0.f;
        for (int m = 0; m < T; ++m) f += Mrow[m] * ms.weps[2 * m + u];
        float up = U[c] + f;                            // u += w_epsilon (:141)
        if (a.clamp_nominal) up = clampf(up, u ? a.umax1 : a.umax0);     // Q9: the visualisation replay clamps u in place
        ms.upre[c] = up;
        out[MPPI_OUT_UPRE + c] = up;                    // kept for mppi_get_trajectories
        out[MPPI_OUT_UOLD + c] = U[c];
    }
    __syncthreads();
    float *oh = (robot == 0) ? a.out_host : nullptr;
    for (int c = tid; c < 2 * T; c += MPPI_BLOCK) {
        const int n = c >> 1, u = c & 1;
        const float v = ms.upre[2 * (n + 1 < T ? n + 1 : T - 1) + u];      // shift, last row kept (:162-163)
        U[c] = v;
        out[MPPI_OUT_HDR + c] = v;
        out[MPPI_OUT_HDR + 2 * MPPI_MAX_T + c] = ms.weps[c];
        if (oh) { oh[MPPI_OUT_HDR + c] = v; oh[MPPI_OUT_HDR + 2 * MPPI_MAX_T + c] = ms.weps[c]; }
    }
    if (tid == 0) {
        const float u0x = ms.upre[2 * (1 < T ? 1 : 0)], u0y = ms.upre[2 * (1 < T ? 1 : 0) + 1];   // Q8
        float hdr[MPPI_OUT_HDR];
        hdr[0] = u0x; hdr[1] = u0y; hdr[2] = __int_as_float(idx_new);
        hdr[3] = ms.col[1]; hdr[4] = ms.col[0]; hdr[5] = eta;
        hdr[6] = eta * eta / ms.col[3]; hdr[7] = 0.f; hdr[10] = out[MPPI_OUT_FAULT]; hdr[11] = 0.f;       // [7] = peer-timeout flag, set by the exchange when a rank never arrived
        hdr[8] = ms.upre[0]; hdr[9] = ms.upre[1];       // the textbook MPPI output: row 0 of the updated nominal before the shift
#pragma unroll
        for (int i = 0; i < MPPI_OUT_HDR; ++i) { out[i] = hdr[i]; if (oh) oh[i] = hdr[i]; }
        if (a.u0_out) { a.u0_out[2 * robot] = u0x; a.u0_out[2 * robot + 1] = u0y; }
        if (a.plant_state) {
            // A17: plant step between ticks.  0: DifferentialDrive.update_state (mppi_differential_drive.py:33-40),
            // unclamped u0; 1: Vehicle.update (models/vehicle.py:95-110), clamp then Euler bicycle.  One plant per robot.
            float *ps = a.plant_state + 4 * robot;
            float px = ps[0], py = ps[1], pyaw = ps[2], pv = ps[3];
            float sn, cs;
            sincos_cw(pyaw, sn, cs);
            if (a.plant_mode == 0) {
                px += u0x * cs * a.dt; py += u0x * sn * a.dt; pyaw += u0y * a.dt;
            } else {
                const float steer = clampf(u0x, a.umax0), accel = clampf(u0y, a.umax1);
                px += pv * cs * a.dt; py += pv * sn * a.dt; pyaw += pv * a.dt_over_L * tanf(steer); pv += accel * a.dt;
            }
            ps[0] = px; ps[1] = py; ps[2] = pyaw; ps[3] = pv;
            float *lg, *lu;
            plant_log_rows(a, robot, lg, lu);
            lg[0] = px; lg[1] = py; lg[2] = pyaw; lg[3] = pv;
            lu[0] = u0x; lu[1] = u0y;
        }
        if (!(a.flags & F_KEEP_IDX)) a.idx[robot] = idx_new;
    }
}

struct RunSmem {
    int n;                     // running lexicographic minimum of this block
    float s;
    float eta, e2;
    float N[2 * MPPI_MAX_T];   // running sum of w * eps, relative to (n, s)
    float w[MPPI_BLOCK];       // stash mode: this chunk's weights
    float warp_eta[MPPI_WARPS], warp_e2[MPPI_WARPS];
    float red_s[MPPI_WARPS];
    int red_n[MPPI_WARPS];
    unsigned long long key[MPPI_WARPS];
    unsigned ticket;
};

// Dynamic shared memory of the tick kernel:
//   STASH = true : float2 eps[T][MPPI_BLOCK] -- the noise of the chunk being rolled out, written in
//                  pass 1 and consumed by the weighted column sums, so Philox + Box-Muller run once.
//   STASH = false: float warpN[MPPI_WARPS][2*MPPI_MAX_T] -- per-warp partial sums of the
//                  regenerate-the-noise path (injected noise, K2 alone, horizons too long to stash).
extern __shared__ __align__(16) unsigned char mppi_dyn_smem[];

// The scene a tick scores against: the shared one in TickArgs, or (SCENE) this CTA's copy of its robot's record.
template <bool SCENE>
__device__ __forceinline__ auto &scene_src(const TickArgs &a) {
    if constexpr (SCENE) {
        __shared__ SceneRec rec;
        return rec;
    } else {
        return a;
    }
}

// STASH: 0 regenerate, 1 noise stash, 2 stash + time-parallel rollout.  SCENE: per-robot goal / obstacles (fleets).
template <int MODEL, int COLL, bool SUM, bool INJ, int WIN, int STASH, bool SCENE>
__device__ __forceinline__ void tick_body(const TickArgs &a, const uint32_t tick_add) {
    static_assert(mppi_tick_built(TickKey{MODEL, COLL, WIN, SUM, INJ, STASH, SCENE}), "a variant mppi_tick_built does not list");
    __shared__ TickSmem sm;
    __shared__ RunSmem run;
    __shared__ MergeSmem ms;
    float2 *stash = reinterpret_cast<float2 *>(mppi_dyn_smem);
    float (*warpN)[2 * MPPI_MAX_T] = reinterpret_cast<float (*)[2 * MPPI_MAX_T]>(mppi_dyn_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int robot = blockIdx.y, b = blockIdx.x, B = gridDim.x;
    const int T = a.T, K = a.K;

    if (a.trace && tid == 0 && robot == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.trace[2 * b] = t; }
    // ---- prologue: observed state, step-1 index update (A8 with update=True), window, nominal
    if (tid < 4) sm.x0[tid] = a.x0_dev ? a.x0_dev[robot * 4 + tid] : a.x0[tid];
    auto &sc = scene_src<SCENE>(a);
    if constexpr (SCENE) {
        // this robot's scene, each component from its per-robot record or from the shared fields; the obstacle count is
        // per CTA, so the obstacle loops stay warp-uniform
        const SceneRec &row = a.scene[robot];
        const bool pg = a.scene_mask & MPPI_SCENE_GOAL, po = a.scene_mask & MPPI_SCENE_OBS;
        if (tid < 4) sc.goal[tid] = pg ? row.goal[tid] : a.goal[tid];
        if (tid == 0) sc.n_obs = po ? row.n_obs : a.n_obs;
        if (tid < MPPI_MAX_OBSTACLES) {
            sc.obs_x[tid] = po ? row.obs_x[tid] : a.obs_x[tid];
            sc.obs_y[tid] = po ? row.obs_y[tid] : a.obs_y[tid];
            if constexpr (WIN == MPPI_WIN_TARGET) {
                sc.obs_vx[tid] = po ? row.obs_vx[tid] : a.obs_vx[tid];
                sc.obs_vy[tid] = po ? row.obs_vy[tid] : a.obs_vy[tid];
            } else {
                sc.obs_r2[tid] = po ? row.obs_r2[tid] : a.obs_r2[tid];
                sc.obs_far2[tid] = po ? row.obs_far2[tid] : a.obs_far2[tid];
            }
        }
    }
    __syncthreads();
    // the robot's reference path: shared, or its own row of the per-robot table (mppi_set_ref_paths_spline)
    const float4 *rpath = a.path_len ? a.path + (size_t)robot * a.path_stride : a.path;
    const int n_path = a.path_len ? a.path_len[robot] : a.n_path;
    int s_new;
    if (WIN < 0) {
        s_new = 0;                                      // goal / target cost kinds: no reference path, no carried index
    } else if (a.flags & F_HOST_IDX) {
        s_new = a.idx_host;
    } else {
        // a carried index outside the robot's path (per-robot courses of different lengths) is clamped to the last
        // waypoint, so the window below is never empty
        const int s_old = max(0, min(a.idx[robot], n_path - 1));
        unsigned long long key = ~0ull;
        MPPI_DCHECK(n_path >= 1 && s_old >= 0 && s_old < n_path && a.window <= MPPI_MAX_WINDOW);
        for (int j = tid; j < a.window && s_old + j < n_path; j += MPPI_BLOCK) {
            const float4 p = rpath[s_old + j];
            const float dx = sm.x0[0] - p.x, dy = sm.x0[1] - p.y;
            const unsigned long long kj = ((unsigned long long)__float_as_uint(dx * dx + dy * dy) << 32) | (unsigned)j;
            key = kj < key ? kj : key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other < key ? other : key;
        }
        if (lane == 0) run.key[warp] = key;
        __syncthreads();
        key = run.key[0];
#pragma unroll
        for (int w = 1; w < MPPI_WARPS; ++w) key = run.key[w] < key ? run.key[w] : key;
        s_new = s_old + (int)(key & 0xffffffffu);
    }
    {
        int nw = n_path - s_new; nw = nw < a.window ? nw : a.window;
        MPPI_DCHECK(WIN < 0 || (s_new >= 0 && s_new < n_path && nw >= 1));
        // static-window kernels read exactly 20 entries, dynamic ones whole chunks of 16
        const int fill = (WIN < 0) ? 0 : (WIN == 20) ? 20 : ((nw + 15) & ~15);
        for (int j = tid; j < fill; j += MPPI_BLOCK) {
            if (j < nw) {
                const float4 p = rpath[s_new + j];
                sm.wx[j] = -p.x; sm.wy[j] = -p.y; sm.wyv[j] = make_float2(p.z, p.w);
            } else {
                sm.wx[j] = -MPPI_SENTINEL; sm.wy[j] = -MPPI_SENTINEL; sm.wyv[j] = make_float2(0.f, 0.f);
            }
        }
        if (tid == 0) { sm.win_start = s_new; sm.n_win16 = fill >> 4; }
        if (WIN == 20) { __syncthreads(); fill_window_expanded(sm, nw, tid, MPPI_BLOCK); }
        if (WIN == 0) {
            __syncthreads();                            // the window is staged: bound every 16-entry chunk from shared memory
            for (int c = tid; c < (fill >> 4); c += MPPI_BLOCK) sm.cb[c] = chunk_bound(sm.wx, sm.wy, 16 * c, min(16, nw - 16 * c));
        }
        const float *Ur = a.U + (size_t)robot * T * 2;
        for (int t = tid; t < T; t += MPPI_BLOCK) {
            const float u0 = Ur[2 * t], u1 = Ur[2 * t + 1];
            sm.U[t] = make_float2(u0, u1);
            sm.Q[t] = make_float2(u0 * a.gq[0] + u1 * a.gq[2], u0 * a.gq[1] + u1 * a.gq[3]);
        }
        if (tid == 0) { run.n = INT_MAX; run.s = CUDART_INF_F; run.eta = 0.f; run.e2 = 0.f; }
        for (int c = tid; c < 2 * T; c += MPPI_BLOCK) run.N[c] = 0.f;
    }
    __syncthreads();

    // ---- this block's contiguous sample range (balanced over the grid), walked in chunks of MPPI_BLOCK samples:
    // thread tid owns chunk slot tid.  Its sample's values are one-element arrays walked by unrolled loops (SPT = 1, the
    // shape of rollout_samples): the compiler keeps them in memory until the loops are unrolled, and plain scalars, promoted
    // to registers earlier, compile 104 of the 134 tick kernels to differently scheduled machine code
    constexpr int SPT = 1;
    const int k_begin = (int)((long long)K * b / B);
    const int k_end = (a.flags & F_IDX_ONLY) ? k_begin : (int)((long long)K * (b + 1) / B);
    MPPI_DCHECK(k_begin >= 0 && k_end <= K && (!STASH || (size_t)T * MPPI_BLOCK * sizeof(float2) <= 232448));
    float *Srow = a.S ? a.S + (size_t)robot * K : nullptr;
    // (time-parallel rollout: chunks of MPPI_TPAR_SLOTS samples on chunk slots 0 .. MPPI_TPAR_SLOTS - 1, the other slots idle)
    constexpr int CHUNK_STRIDE = STASH == 2 ? MPPI_TPAR_SLOTS : MPPI_BLOCK;
    for (int base = k_begin; base < k_end; base += CHUNK_STRIDE) {
        int k[SPT], ksafe[SPT], ncoll[SPT];
        bool active[SPT], exploit[SPT];
        uint32_t kg[SPT];
        float smooth[SPT];
#pragma unroll
        for (int s = 0; s < SPT; ++s) {
            k[s] = base + tid + s * MPPI_BLOCK;
            active[s] = k[s] < k_end && (STASH != 2 || tid < MPPI_TPAR_SLOTS);
            ksafe[s] = active[s] ? k[s] : k_begin;             // an idle slot of the tail chunk replays a valid sample (weight 0)
            kg[s] = (uint32_t)(a.k_offset + ksafe[s]);
            exploit[s] = (int)kg[s] < a.n_exploit;
            smooth[s] = CUDART_INF_F; ncoll[s] = INT_MAX;
        }
        if constexpr (STASH == 2) {
            MPPI_DCHECK(!(a.flags & F_FROM_S) && (size_t)T * MPPI_TPAR_SLOTS * (sizeof(float2) + sizeof(float4)) <= 232448);
            float4 *zbuf = reinterpret_cast<float4 *>(mppi_dyn_smem + sizeof(float2) * (size_t)T * MPPI_TPAR_SLOTS);
            __shared__ TparSmem tps;
            rollout_tpar<MODEL, COLL, WIN>(a, sm, tps, base, min(k_end - base, MPPI_TPAR_SLOTS), (uint32_t)robot, stash, zbuf,
                                           smooth[0], ncoll[0], tick_add);
            if (active[0] && (a.flags & F_WRITE_S)) Srow[k[0]] = smooth[0] + MPPI_PENALTY * (float)ncoll[0];
        } else if (active[0]) {                                 // slots ascend with s: no active sample without the first
            if (a.flags & F_FROM_S) {
#pragma unroll
                for (int s = 0; s < SPT; ++s)
                    if (active[s]) { smooth[s] = Srow[k[s]]; ncoll[s] = a.NC ? a.NC[k[s]] : 0; }
            } else {
                rollout_samples<MODEL, COLL, SUM, INJ, WIN, SPT>(a, sc, sm, kg, ksafe, (uint32_t)robot, exploit,
                                                                 STASH ? stash + tid : nullptr, smooth, ncoll, tick_add);
#pragma unroll
                for (int s = 0; s < SPT; ++s) {
                    if (active[s] && (a.flags & F_WRITE_S)) Srow[k[s]] = smooth[s] + MPPI_PENALTY * (float)ncoll[s];
                    if (!active[s]) { smooth[s] = CUDART_INF_F; ncoll[s] = INT_MAX; }
                }
            }
        }
        if (!(a.flags & F_UPDATE)) continue;
        if (STASH == 1 && !active[0]) {             // tail chunk: a thread that rolled nothing out must not leave garbage (0 * NaN)
            for (int t = 0; t < T; ++t)
#pragma unroll
                for (int s = 0; s < SPT; ++s) stash[t * MPPI_BLOCK + s * MPPI_BLOCK + tid] = make_float2(0.f, 0.f);
        }

        // chunk minimum -> new running minimum
        int cn = ncoll[0]; float cs_ = smooth[0];
#pragma unroll
        for (int s = 1; s < SPT; ++s)
            if (ncoll[s] < cn || (ncoll[s] == cn && smooth[s] < cs_)) { cn = ncoll[s]; cs_ = smooth[s]; }
        warp_lexmin(cn, cs_);
        if (lane == 0) { run.red_n[warp] = cn; run.red_s[warp] = cs_; }
        __syncthreads();
        int mn = run.n; float mss = run.s;
#pragma unroll
        for (int w = 0; w < MPPI_WARPS; ++w) {
            const int wn = run.red_n[w]; const float ws = run.red_s[w];
            if (wn < mn || (wn == mn && ws < mss)) { mn = wn; mss = ws; }
        }
        const float rescale = (run.n == INT_MAX) ? 0.f : rel_weight(run.n, run.s, mn, mss, a.inv_temp);
        float w[SPT], wsum = 0.f, w2sum = 0.f;
#pragma unroll
        for (int s = 0; s < SPT; ++s) {
            w[s] = active[s] ? rel_weight(ncoll[s], smooth[s], mn, mss, a.inv_temp) : 0.f;
            wsum += w[s]; w2sum = fmaf(w[s], w[s], w2sum);
        }
        const float we = warp_sum(wsum), we2 = warp_sum(w2sum);
        if (lane == 0) { run.warp_eta[warp] = we; run.warp_e2[warp] = we2; }

        if (STASH) {
            // weighted column sums straight from the stash: warp `warp` owns rows t = warp, warp + MPPI_WARPS, ...
#pragma unroll
            for (int s = 0; s < SPT; ++s) run.w[tid + s * MPPI_BLOCK] = w[s];
            __syncthreads();
            constexpr int SCOLS = STASH == 2 ? MPPI_TPAR_SLOTS : MPPI_BLOCK;       // columns of a stash row
            float wr[SCOLS / 32];
#pragma unroll
            for (int i = 0; i < SCOLS / 32; ++i) wr[i] = run.w[lane + 32 * i];
            for (int t = warp; t < T; t += MPPI_WARPS) {
                const float2 *row = stash + t * SCOLS;
                float ax = 0.f, ay = 0.f;
#pragma unroll
                for (int i = 0; i < SCOLS / 32; ++i) {
                    const float2 e = row[lane + 32 * i];
                    ax = fmaf(wr[i], e.x, ax); ay = fmaf(wr[i], e.y, ay);
                }
                // two sums over 32 lanes: exchange halves, then one butterfly (6 shuffles)
                const bool hi = lane & 16;
                const float other = __shfl_xor_sync(0xffffffffu, hi ? ax : ay, 16);
                float p = (hi ? ay : ax) + other;
                p += __shfl_xor_sync(0xffffffffu, p, 8);
                p += __shfl_xor_sync(0xffffffffu, p, 4);
                p += __shfl_xor_sync(0xffffffffu, p, 2);
                p += __shfl_xor_sync(0xffffffffu, p, 1);
                if ((lane & 15) == 0) {
                    const int c = 2 * t + (lane >> 4);
                    run.N[c] = run.N[c] * rescale + p;
                }
            }
        } else {
            // regenerate (Philox) or re-read (injected) the eps rows of this thread's samples
            const bool any = __any_sync(0xffffffffu, wsum > 0.f);
            if (any) {
                const float2 *eps_k[SPT];
#pragma unroll
                for (int s = 0; s < SPT; ++s)
                    eps_k[s] = INJ ? reinterpret_cast<const float2 *>(a.eps) + (size_t)ksafe[s] * T : nullptr;
                for (int tp = 0; tp < T; tp += 2) {
                    float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
#pragma unroll
                    for (int s = 0; s < SPT; ++s) {
                        float e[4] = {0.f, 0.f, 0.f, 0.f};
                        if (INJ) {
                            const float2 ea = eps_k[s][tp];
                            e[0] = ea.x; e[1] = ea.y;
                            if (tp + 1 < T) { const float2 eb = eps_k[s][tp + 1]; e[2] = eb.x; e[3] = eb.y; }
                        } else {
                            philox_eps_pair(a, kg[s], (uint32_t)(tp >> 1), (uint32_t)robot, e, tick_add);
                        }
                        p0 = fmaf(w[s], e[0], p0); p1 = fmaf(w[s], e[1], p1); p2 = fmaf(w[s], e[2], p2); p3 = fmaf(w[s], e[3], p3);
                    }
                    // 4 values x 32 lanes -> 4 sums: halving butterfly (6 shuffles instead of 20)
                    {
                        const bool hi = lane & 16;
                        const float s0 = hi ? p0 : p2, s1 = hi ? p1 : p3;
                        const float r0 = __shfl_xor_sync(0xffffffffu, s0, 16), r1 = __shfl_xor_sync(0xffffffffu, s1, 16);
                        p0 = (hi ? p2 : p0) + r0; p1 = (hi ? p3 : p1) + r1;
                    }
                    {
                        const bool hi = lane & 8;
                        const float s0 = hi ? p0 : p1;
                        const float r0 = __shfl_xor_sync(0xffffffffu, s0, 8);
                        p0 = (hi ? p1 : p0) + r0;
                    }
                    p0 += __shfl_xor_sync(0xffffffffu, p0, 4);
                    p0 += __shfl_xor_sync(0xffffffffu, p0, 2);
                    p0 += __shfl_xor_sync(0xffffffffu, p0, 1);
                    if ((lane & 7) == 0) {
                        const int c = 2 * tp + (lane >> 3);
                        if (c < 2 * T) warpN[warp][c] = p0;
                    }
                }
            } else {
                for (int c = lane; c < 2 * T; c += 32) warpN[warp][c] = 0.f;
            }
            __syncthreads();
            for (int c = tid; c < 2 * T; c += MPPI_BLOCK) {
                float acc = run.N[c] * rescale;
#pragma unroll
                for (int wv = 0; wv < MPPI_WARPS; ++wv) acc += warpN[wv][c];
                run.N[c] = acc;
            }
        }
        __syncthreads();
        if (tid == 0) {
            float e1 = run.eta * rescale, e2 = run.e2 * rescale * rescale;
#pragma unroll
            for (int wv = 0; wv < MPPI_WARPS; ++wv) { e1 += run.warp_eta[wv]; e2 += run.warp_e2[wv]; }
            run.eta = e1; run.e2 = e2; run.n = mn; run.s = mss;
        }
        __syncthreads();
    }

    if (a.trace && tid == 0 && robot == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.trace[2 * b + 1] = t; }
    // ---- publish the block partial, elect the last block
    const int NF = MPPI_NF(T);
    float *parts = a.part + (size_t)robot * B * NF;
    if (a.flags & F_UPDATE) {
        if (B > 1) {
            float *mine = parts + (size_t)b * NF;
            for (int c = tid; c < 2 * T; c += MPPI_BLOCK) mine[4 + c] = run.N[c];
            if (tid == 0) { mine[0] = __int_as_float(run.n); mine[1] = run.s; mine[2] = run.eta; mine[3] = run.e2; }
        }
    }
    // TWO-LEVEL merge (grids of >= MPPI_MERGE_TWO_LEVEL_MIN CTAs): consecutive CTAs form groups of
    // MPPI_MERGE_GROUP_CTAS; the last CTA of a group to finish merges that group's partials into one group partial -- while the other
    // groups are still rolling out -- and the last GROUP merges the ~B/16 group partials and finalizes.  What stays on the tick's
    // critical path is one 16-way and one B/16-way merge (one L2 round trip each) instead of one B-way merge by a single CTA
    // (8.6 us of a 412 us tick at B = 296).  Same log-sum-exp rule at both levels; the grouping is fixed, so results stay deterministic.
    const bool two_level = (a.flags & F_UPDATE) && B >= MPPI_MERGE_TWO_LEVEL_MIN && a.part2 != nullptr;
    int n_merge = B;                                     // partials the finalizing CTA merges, and where they are
    const float *merge_src = parts;
    if (B > 1) {
        __threadfence();
        __syncthreads();
        if (two_level) {
            const int grp = b / MPPI_MERGE_GROUP_CTAS, g_first = grp * MPPI_MERGE_GROUP_CTAS;
            const int g_cnt = min(MPPI_MERGE_GROUP_CTAS, B - g_first), n_groups = (B + MPPI_MERGE_GROUP_CTAS - 1) / MPPI_MERGE_GROUP_CTAS;
            MPPI_DCHECK(n_groups <= a.merge_gmax);
            unsigned *gt = a.ticket2 + (size_t)robot * a.merge_gmax + grp;
            if (tid == 0) run.ticket = atomicAdd(gt, 1u);
            __syncthreads();
            if (run.ticket != (unsigned)(g_cnt - 1)) return;
            if (tid == 0) *gt = 0u;                         // re-arm for the next launch
            __threadfence();
            merge_partials(a, parts + (size_t)g_first * NF, g_cnt, ms, reinterpret_cast<float *>(mppi_dyn_smem));
            float *gp = a.part2 + ((size_t)robot * a.merge_gmax + grp) * NF;
            for (int c = tid; c < NF; c += MPPI_BLOCK) gp[c] = ms.col[c];
            __threadfence();
            __syncthreads();
            n_merge = n_groups;
            merge_src = a.part2 + (size_t)robot * a.merge_gmax * NF;
        }
        if (tid == 0) run.ticket = atomicAdd(&a.ticket[robot], 1u);
        __syncthreads();
        if (run.ticket != (unsigned)((two_level ? n_merge : B) - 1)) return;
        if (tid == 0) a.ticket[robot] = 0u;             // re-arm for the next launch
        __threadfence();
    }
    if (!(a.flags & F_UPDATE)) {
        if (tid == 0 && !(a.flags & F_KEEP_IDX)) a.idx[robot] = s_new;
        return;
    }
    if (B > 1) {
        merge_partials(a, merge_src, n_merge, ms, reinterpret_cast<float *>(mppi_dyn_smem));   // the noise stash is free by now
    } else {
        for (int c = tid; c < 2 * T; c += MPPI_BLOCK) ms.col[4 + c] = run.N[c];
        if (tid == 0) { ms.col[0] = __int_as_float(run.n); ms.col[1] = run.s; ms.col[2] = run.eta; ms.col[3] = run.e2; }
        __syncthreads();
    }
    if (a.trace && tid == 0 && robot == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.trace[2 * B] = t; }
    if (a.flags & F_P2P) {
        // ---- fused exchange over NVLink peer memory.  Every column of this GPU's triple goes to every rank (its own
        // buffer included) as ONE 8-byte store carrying (tick sequence number, float bits): the flag travels with the
        // datum (NCCL's "LL" idea), so there is no system-scope fence, no separate flag store and no second round trip --
        // the cost is one NVLink write latency after the slowest rank's last CTA.  G*NF words are written and polled by
        // the whole CTA in parallel.  Slots are double-buffered by tick parity: a rank can run at most one tick ahead of
        // a peer (it needs that peer's words of tick t to finish tick t), so parity t&1 is never overwritten while read.
        const int G = a.p2p_world, me = a.p2p_rank;
        const unsigned seq = a.p2p_seq, par = seq & 1u;
        unsigned long long t_stamp[4];
        if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_stamp[0]));
        for (int i = tid; i < G * NF; i += MPPI_BLOCK) {
            const int p = i / NF, c = i - p * NF;
            MPPI_DCHECK(MPPI_XCHG_SLOT(par, me) + c < MPPI_XCHG_WORDS && G <= MPPI_MAX_PEERS && me < G);
            unsigned long long *dst = a.peer_buf[p] + MPPI_XCHG_SLOT(par, me) + c;
            const unsigned long long v = ((unsigned long long)seq << 32) | (unsigned long long)__float_as_uint(ms.col[c]);
            asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(v) : "memory");
        }
        if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_stamp[1]));
        float *xs = reinterpret_cast<float *>(mppi_dyn_smem);       // [G][NF] gathered triples (the noise stash is free by now)
        bool ok = true;
        {
            unsigned long long t0;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            const unsigned long long limit = (unsigned long long)a.p2p_timeout_ms * 1000000ull;
            for (int i = tid; i < G * NF; i += MPPI_BLOCK) {
                const int r = i / NF, c = i - r * NF;
                const unsigned long long *src = a.peer_buf[me] + MPPI_XCHG_SLOT(par, r) + c;
                unsigned long long v, now;
                int spins = 0;
                do {
                    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
                    if ((unsigned)(v >> 32) == seq) break;
                    if ((++spins & 255) == 0) {                     // a dead peer must not hang the device
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                        if (now - t0 > limit) { ok = false; break; }
                    }
                } while (true);
                xs[r * NF + c] = __uint_as_float((unsigned)v);
            }
        }
        const int all_ok = __syncthreads_and(ok ? 1 : 0);
        if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_stamp[2]));
        if (!all_ok) {
            // a peer never arrived: leave the nominal and the waypoint index untouched and report it (the host returns
            // MPPI_E_NCCL from mppi_step / mppi_synchronize and clears the flag)
            if (tid == 0) { a.out[MPPI_OUT_PEER_TIMEOUT] = 1.f; if (a.out_host) a.out_host[MPPI_OUT_PEER_TIMEOUT] = 1.f; }
            return;
        }
        // merge in rank order: identical arithmetic, hence identical bits, on every rank
        {
            int n = __float_as_int(xs[0]); float s = xs[1];
            for (int r = 1; r < G; ++r) {
                const int rn = __float_as_int(xs[r * NF]); const float rs = xs[r * NF + 1];
                if (rn < n || (rn == n && rs < s)) { n = rn; s = rs; }
            }
            for (int c = 2 + tid; c < NF; c += MPPI_BLOCK) {
                float acc = 0.f;
                for (int r = 0; r < G; ++r) {
                    const float w = rel_weight(__float_as_int(xs[r * NF]), xs[r * NF + 1], n, s, a.inv_temp);
                    acc = fmaf(c == 3 ? w * w : w, xs[r * NF + c], acc);
                }
                ms.col[c] = acc;
            }
            __syncthreads();            // every thread has read ms.col[0..1]-independent inputs from xs; now publish the key
            if (tid == 0) { ms.col[0] = __int_as_float(n); ms.col[1] = s; }
            __syncthreads();
        }
        finalize_tick(a, robot, s_new, ms);
        if (tid == 0) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_stamp[3]));
            unsigned long long *tr = a.peer_buf[me] + MPPI_XCHG_WORDS;      // diagnostics: mppi_comm_p2p_trace
            tr[0] = t_stamp[0]; tr[1] = t_stamp[1]; tr[2] = t_stamp[2]; tr[3] = t_stamp[3];
        }
        return;
    }
    if (a.flags & F_TRIPLE_OUT) {
        for (int c = tid; c < NF; c += MPPI_BLOCK) a.triple_out[c] = ms.col[c];
        if (tid == 0) a.out[2] = __int_as_float(s_new);   // stash the new index for the merge kernel
        return;
    }
    finalize_tick(a, robot, s_new, ms);
    if (a.trace && tid == 0 && robot == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.trace[2 * B + 1] = t; }
}

// (scene instantiations are register-budgeted for MPPI_STASH_BLOCKS resident CTAs on both rollout paths: their obstacle and
// goal operands are shared-memory loads, not constant-bank operands)
template <int MODEL, int COLL, bool SUM, bool INJ, int WIN, int STASH, bool SCENE = false>
__global__ void __launch_bounds__(MPPI_BLOCK, (STASH || SCENE) ? MPPI_STASH_BLOCKS : MPPI_MIN_BLOCKS) mppi_tick_kernel(const __grid_constant__ TickArgs a) {
    // graph-captured closed loop: the tick this launch computes is read from device memory (every CTA reads it before any
    // CTA of the same launch can advance it: the advance happens after ALL CTAs have taken a ticket, below)
    const uint32_t tick_add = a.loop_state ? __ldcg(a.loop_state) : 0u;
    tick_body<MODEL, COLL, SUM, INJ, WIN, STASH, SCENE>(a, tick_add);
    if (a.loop_state) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            const unsigned total = gridDim.x * gridDim.y;
            if (atomicAdd(a.loop_ticket, 1u) == total - 1u) {
                *a.loop_ticket = 0u;
                __threadfence();
                atomicAdd(a.loop_state, 1u);
            }
        }
    }
}

// Merge of G per-GPU triples (after the all-gather) + finalize; identical on every rank.
__global__ void __launch_bounds__(MPPI_BLOCK) mppi_merge_kernel(const __grid_constant__ TickArgs a,
                                                                 const float *triples, int G) {
    __shared__ MergeSmem ms;
    __shared__ __align__(16) float sc[MPPI_MERGE_SCRATCH];
    merge_partials(a, triples, G, ms, sc);
    finalize_tick(a, 0, __float_as_int(a.out[2]), ms);
}

// Device-side barrier of the ranks of a fused exchange: every rank stores the barrier count into its word of every peer's
// buffer and waits until all of its own words have reached it (counts only grow, so a rank already in the next barrier
// cannot be missed).  Aligns the GPUs on the device, e.g. in front of a timed tick (no host round trip, no NCCL call).
__global__ void mppi_p2p_barrier_kernel(const __grid_constant__ TickArgs a, unsigned long long count) {
    const int G = a.p2p_world, me = a.p2p_rank, t = threadIdx.x;
    if (t >= G) return;
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(a.peer_buf[t] + MPPI_XCHG_BARRIER + me), "l"(count) : "memory");
    const unsigned long long *mine = a.peer_buf[me] + MPPI_XCHG_BARRIER + t;
    unsigned long long v, t0, now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    const unsigned long long limit = (unsigned long long)a.p2p_timeout_ms * 1000000ull;
    int spins = 0;
    do {
        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(mine) : "memory");
        if (v >= count) break;
        if ((++spins & 255) == 0) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (now - t0 > limit) { a.out[MPPI_OUT_PEER_TIMEOUT] = 1.f; if (a.out_host) a.out_host[MPPI_OUT_PEER_TIMEOUT] = 1.f; break; }
        }
    } while (true);
}

// A16: visualisation replays of the last tick.  Thread k < K replays sample k's clamped controls, thread K the
// updated nominal; both index the controls with t-1 (the last row first), as the reference does.
// With a selection list (`sel`, n_sel entries: the top-N viewer of test/test_mppi_diff_obs.py:102-110) row i of samp_out
// replays sample sel[i]; `shift` = 1 indexes the controls with t-1 (the reference classes), 0 with t (that script, :108).
template <int MODEL>
__global__ void mppi_traj_kernel(const __grid_constant__ TickArgs a, const float *__restrict__ rec,
                                 float *__restrict__ opt_out, float *__restrict__ samp_out,
                                 const int *__restrict__ sel, int n_sel, int shift) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_rows = sel ? n_sel : a.K;
    if (row > n_rows) return;
    const bool nominal = row == n_rows;
    if (nominal ? opt_out == nullptr : samp_out == nullptr) return;
    const int k = nominal ? a.K : (sel ? sel[row] : row);
    constexpr int NX = MODEL == MPPI_MODEL_BICYCLE ? 4 : 3;
    const int T = a.T;
    const float *upre = rec + MPPI_OUT_UPRE, *uold = rec + MPPI_OUT_UOLD;
    const uint32_t kg = (uint32_t)(a.k_offset + k);
    const bool exploit = (int)kg < a.n_exploit;
    float z[4] = {a.x0[0], a.x0[1], a.x0[2], a.x0[3]};
    float *dst = nominal ? opt_out : samp_out + (size_t)row * T * NX;
    for (int t = 0; t < T; ++t) {
        const int tc = shift ? (t + T - 1) % T : t;                       // u[t-1] with Python's negative index
        float v0, v1;
        if (nominal) {
            v0 = clampf(upre[2 * tc], a.umax0); v1 = clampf(upre[2 * tc + 1], a.umax1);
        } else {
            float e0, e1;
            if (a.eps) {
                const float2 ee = reinterpret_cast<const float2 *>(a.eps)[(size_t)k * T + tc];
                e0 = ee.x; e1 = ee.y;
            } else {
                float e[4];
                philox_eps_pair(a, kg, (uint32_t)(tc >> 1), 0u, e);
                e0 = e[2 * (tc & 1)]; e1 = e[2 * (tc & 1) + 1];
            }
            v0 = clampf(exploit ? __fadd_rn(uold[2 * tc], e0) : e0, a.umax0);
            v1 = clampf(exploit ? __fadd_rn(uold[2 * tc + 1], e1) : e1, a.umax1);
        }
        float sn, cs;
        sincos_cw(z[2], sn, cs);
        dyn_step<MODEL>(a, z, v0, v1, cs, sn);
#pragma unroll
        for (int i = 0; i < NX; ++i) dst[t * NX + i] = z[i];
    }
}

// The controls of those replays as a table, for the learned-dynamics viewers (mppi_mlp.cu replays it through the tick's own
// rollout): row i < n_rows = sample sel[i] (sample i without a selection), row n_rows = the updated nominal; same rule as above.
__global__ void mppi_traj_controls_kernel(const __grid_constant__ TickArgs a, const float *__restrict__ rec, float2 *__restrict__ ctl,
                                          const int *__restrict__ sel, int n_rows, int shift) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row > n_rows) return;
    const bool nominal = row == n_rows;
    const int k = nominal ? a.K : (sel ? sel[row] : row);
    const int T = a.T;
    const float *upre = rec + MPPI_OUT_UPRE, *uold = rec + MPPI_OUT_UOLD;
    const uint32_t kg = (uint32_t)(a.k_offset + k);
    const bool exploit = (int)kg < a.n_exploit;
    for (int t = 0; t < T; ++t) {
        const int tc = shift ? (t + T - 1) % T : t;
        float v0, v1;
        if (nominal) {
            v0 = clampf(upre[2 * tc], a.umax0); v1 = clampf(upre[2 * tc + 1], a.umax1);
        } else {
            float e0, e1;
            if (a.eps) {
                const float2 ee = reinterpret_cast<const float2 *>(a.eps)[(size_t)k * T + tc];
                e0 = ee.x; e1 = ee.y;
            } else {
                float e[4];
                philox_eps_pair(a, kg, (uint32_t)(tc >> 1), 0u, e);
                e0 = e[2 * (tc & 1)]; e1 = e[2 * (tc & 1) + 1];
            }
            v0 = clampf(exploit ? __fadd_rn(uold[2 * tc], e0) : e0, a.umax0);
            v1 = clampf(exploit ? __fadd_rn(uold[2 * tc + 1], e1) : e1, a.umax1);
        }
        ctl[(size_t)row * T + t] = make_float2(v0, v1);
    }
}

// (K,T,2) export of the Philox noise the tick kernel consumes
__global__ void mppi_noise_kernel(const __grid_constant__ TickArgs a, float *out, int robot) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.K) return;
    float2 *row = reinterpret_cast<float2 *>(out) + (size_t)k * a.T;
    for (int tp = 0; tp < a.T; tp += 2) {
        float e[4];
        philox_eps_pair(a, (uint32_t)(a.k_offset + k), (uint32_t)(tp >> 1), (uint32_t)robot, e);
        row[tp] = make_float2(e[0], e[1]);
        if (tp + 1 < a.T) row[tp + 1] = make_float2(e[2], e[3]);
    }
}

// ---- strict waypoint mode (Q3): literal evaluation order via the multi-pass rule ----------
// Evaluation n = k*(T+1) + t (t = 0..T-1 stage, t = T terminal) uses the window start given by
// the last breakpoint (bp_n <= n).  The first evaluation >= check_from whose argmin differs
// from its window start is reported through first_change = min((n << 32) | argmin).
template <int MODEL, int COLL, bool SUM, bool INJ>
__global__ void __launch_bounds__(MPPI_BLOCK) mppi_strict_kernel(const __grid_constant__ TickArgs a,
                                                                  const unsigned *bp_n, const int *bp_s, int nbp,
                                                                  int k_first, unsigned check_from,
                                                                  unsigned long long *first_change) {
    const int k = k_first + blockIdx.x * MPPI_BLOCK + threadIdx.x;
    if (k >= a.K) return;
    const int T = a.T;
    const uint32_t kg = (uint32_t)(a.k_offset + k);
    const bool exploit = (int)kg < a.n_exploit;
    float z[4] = {a.x0[0], a.x0[1], a.x0[2], a.x0[3]};
    float cs, sn;
    sincos_cw(z[2], sn, cs);
    float acc = 0.f;
    int nc = 0;
    int bp = 0;
    const float2 *eps_k = INJ ? reinterpret_cast<const float2 *>(a.eps) + (size_t)k * T : nullptr;
    float e[4];
    for (int t = 0; t <= T; ++t) {
        float v0 = 0.f, v1 = 0.f;
        if (t < T) {
            if (INJ) { const float2 ea = eps_k[t]; e[2 * (t & 1)] = ea.x; e[2 * (t & 1) + 1] = ea.y; }
            else if ((t & 1) == 0) philox_eps_pair(a, kg, (uint32_t)(t >> 1), 0u, e);
            const float u0 = a.U[2 * t], u1 = a.U[2 * t + 1];
            v0 = clampf(exploit ? __fadd_rn(u0, e[2 * (t & 1)]) : e[2 * (t & 1)], a.umax0);
            v1 = clampf(exploit ? __fadd_rn(u1, e[2 * (t & 1) + 1]) : e[2 * (t & 1) + 1], a.umax1);
            dyn_step<MODEL>(a, z, v0, v1, cs, sn);
            sincos_cw(z[2], sn, cs);
        }
        const unsigned n = (unsigned)k * (unsigned)(T + 1) + (unsigned)t;
        while (bp + 1 < nbp && bp_n[bp + 1] <= n) ++bp;
        const int s = bp_s[bp];
        int end = s + a.window; end = end < a.n_path ? end : a.n_path;
        float bd = CUDART_INF_F; int bj = s;
        for (int j = s; j < end; ++j) {
            const float4 p = a.path[j];
            const float dx = z[0] - p.x, dy = z[1] - p.y, d = dx * dx + dy * dy;
            if (d < bd) { bd = d; bj = j; }
        }
        if (bj != s && n >= check_from) atomicMin(first_change, ((unsigned long long)n << 32) | (unsigned)bj);
        const bool stage = t < T, last = (t == T - 1);
        if ((stage && (SUM || last)) || t == T) {
            MPPI_DCHECK(bj >= 0 && bj < a.n_path && bp < nbp);
            const float4 ref = a.path[bj];
            const float yaw_eff = a.yaw_wrap ? wrap_2pi(z[2]) : z[2];
            float c = tracking_cost<MODEL>(ref, z, yaw_eff, stage ? a.sw : a.tw);
            if (stage && a.use_gamma) {
                const float u0 = a.U[2 * t], u1 = a.U[2 * t + 1];
                c += (u0 * a.gq[0] + u1 * a.gq[2]) * v0 + (u0 * a.gq[1] + u1 * a.gq[3]) * v1;
            }
            const bool hit = collided<MODEL, COLL>(a, a, z[0], z[1], cs, sn);
            if (stage && !SUM) { acc = c; nc = hit ? 1 : 0; }      // Q1: assignment
            else { acc += c; nc += hit ? 1 : 0; }
        }
    }
    a.S[k] = acc;
    a.NC[k] = nc;
    if (a.S_user) a.S_user[k] = acc + MPPI_PENALTY * (float)nc;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// dispatch: a table of every built tick kernel, indexed by its packed key
// ------------------------------------------------------------------------------------------
namespace {
constexpr int kTickSlots = 2 * 3 * 4 * 2 * 2 * 3 * 2;      // model, collision, window, sum, inj, stash, scene
constexpr int kMaxDevices = 64;

// the table slot of a key whose fields are in range (built or not)
constexpr int tick_slot(const TickKey &k) {
    const int w = k.win == 20 ? 0 : k.win == 0 ? 1 : k.win == MPPI_WIN_GOAL ? 2 : 3;
    return (((((k.model * 3 + k.coll) * 4 + w) * 2 + k.sum) * 2 + k.inj) * 3 + k.stash) * 2 + k.scene;
}

// The i-th key in the order the table names the kernels, which is the order the device compiler meets them in.  Its inlining
// and scheduling of helpers several kernels share depend on that order, so it is the order the earlier if-chain dispatchers
// named them in: scene variants first, then goal, target and path kinds, model, collision; flags descending and window 20
// before the dynamic one, the window above sum and stash for scene variants and below them for the others.
constexpr int kTickOrder = 2 * 3 * 2 * 3 * 24;
constexpr TickKey ordered_key(int i) {
    TickKey k{};
    k.scene = i < kTickOrder / 2;
    const int kind = i / 144 % 3, w = k.scene ? i / 12 % 2 : i % 2;
    k.model = i / 72 % 2;
    k.coll = i / 24 % 3;
    k.win = kind == 0 ? MPPI_WIN_GOAL : kind == 1 ? MPPI_WIN_TARGET : w ? 0 : 20;
    k.sum = (k.scene ? i / 6 : i / 12) % 2 == 0;
    k.inj = (k.scene ? i / 3 : i / 6) % 2 == 0;
    k.stash = 2 - (k.scene ? i : i / 2) % 3;
    return k;
}

using TickKernel = void (*)(TickArgs);

template <int I>
constexpr TickKernel tick_kernel_at() {
    constexpr TickKey k = ordered_key(I);
    if constexpr (mppi_tick_built(k)) return mppi_tick_kernel<k.model, k.coll, k.sum, k.inj, k.win, k.stash, k.scene>;
    else return nullptr;
}
template <int... I>
constexpr std::array<TickKernel, kTickSlots> tick_table(std::integer_sequence<int, I...>) {
    std::array<TickKernel, kTickSlots> t{};
    ((t[tick_slot(ordered_key(I))] = tick_kernel_at<I>()), ...);
    return t;
}
constexpr std::array<TickKernel, kTickSlots> kTickKernels = tick_table(std::make_integer_sequence<int, kTickOrder>{});

// Opt-in of kTickKernels[s] to `dyn` bytes of dynamic shared memory on the current device.  The attribute belongs to the
// function, so every handle of a variant shares it: it is only ever RAISED, under one lock, and the slot's record keeps the
// largest size set per device.  Setting it to each new handle's own size would cut it below what a live handle with a longer
// horizon launches with, and that handle's next tick would fail with cudaErrorInvalidValue.  A size the record already
// covers is read without the lock: the record only grows.
cudaError_t opt_in_dyn_smem(int s, size_t dyn) {
    if (dyn <= 32 * 1024) return cudaSuccess;       // static shared memory (12 KB) counts against the 48 KB default limit too
    static std::atomic<unsigned> raised[kTickSlots][kMaxDevices];
    static std::mutex mu;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    std::atomic<unsigned> &rec = raised[s][dev];
    if (rec.load(std::memory_order_acquire) >= dyn) return cudaSuccess;
    std::lock_guard<std::mutex> lock(mu);
    if (rec.load(std::memory_order_relaxed) >= dyn) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute((const void *)kTickKernels[s], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e == cudaSuccess) rec.store((unsigned)dyn, std::memory_order_release);
    return e;
}
}  // namespace

size_t mppi_tick_dyn_smem(int T, int stash) {
    // regenerate path: per-warp column sums (8 KB), also large enough for the exchange's gathered triples
    const size_t small = std::max(sizeof(float) * MPPI_WARPS * 2 * MPPI_MAX_T, sizeof(float) * MPPI_MAX_PEERS * MPPI_NF_MAX);
    if (stash == 2) return std::max((sizeof(float2) + sizeof(float4)) * MPPI_TPAR_SLOTS * (size_t)T, small);   // noise + the states of every step
    return stash ? std::max(sizeof(float2) * (size_t)T * MPPI_BLOCK, small) : small;
}

cudaError_t mppi_launch_tick(const TickArgs &a, const TickKey &k, dim3 grid, cudaStream_t st) {
    if (!mppi_tick_built(k)) return cudaErrorInvalidValue;
    const int s = tick_slot(k);
    const size_t dyn = mppi_tick_dyn_smem(a.T, k.stash);
    if (const cudaError_t e = opt_in_dyn_smem(s, dyn)) return e;
    kTickKernels[s]<<<grid, MPPI_BLOCK, dyn, st>>>(a);
    return cudaGetLastError();
}

// Resident CTAs per SM of a variant (0 if it is not built or cannot launch).
int mppi_tick_occupancy(const TickKey &k, int T) {
    if (!mppi_tick_built(k)) return 0;
    const int s = tick_slot(k);
    const size_t dyn = mppi_tick_dyn_smem(T, k.stash);
    int nb = 0;
    if (opt_in_dyn_smem(s, dyn) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kTickKernels[s], MPPI_BLOCK, dyn) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return nb;
}

template <int MODEL, int COLL>
static cudaError_t launch_strict_mc(const TickArgs &a, bool sum, bool inj, const unsigned *bp_n, const int *bp_s,
                                    int nbp, int k_first, unsigned check_from, unsigned long long *fc, cudaStream_t st) {
    const int nblk = (a.K - k_first + MPPI_BLOCK - 1) / MPPI_BLOCK;
    if (nblk <= 0) return cudaSuccess;
    if (sum) {
        if (inj) mppi_strict_kernel<MODEL, COLL, true, true><<<nblk, MPPI_BLOCK, 0, st>>>(a, bp_n, bp_s, nbp, k_first, check_from, fc);
        else mppi_strict_kernel<MODEL, COLL, true, false><<<nblk, MPPI_BLOCK, 0, st>>>(a, bp_n, bp_s, nbp, k_first, check_from, fc);
    } else {
        if (inj) mppi_strict_kernel<MODEL, COLL, false, true><<<nblk, MPPI_BLOCK, 0, st>>>(a, bp_n, bp_s, nbp, k_first, check_from, fc);
        else mppi_strict_kernel<MODEL, COLL, false, false><<<nblk, MPPI_BLOCK, 0, st>>>(a, bp_n, bp_s, nbp, k_first, check_from, fc);
    }
    return cudaGetLastError();
}

cudaError_t mppi_launch_strict(const TickArgs &a, int model, int coll, bool sum, bool inj, const unsigned *bp_n,
                               const int *bp_s, int nbp, int k_first, unsigned check_from,
                               unsigned long long *first_change, cudaStream_t st) {
    if (model == MPPI_MODEL_DIFFDRIVE) {
        if (coll == MPPI_COLLISION_NONE) return launch_strict_mc<MPPI_MODEL_DIFFDRIVE, MPPI_COLLISION_NONE>(a, sum, inj, bp_n, bp_s, nbp, k_first, check_from, first_change, st);
        if (coll == MPPI_COLLISION_CIRCLE) return launch_strict_mc<MPPI_MODEL_DIFFDRIVE, MPPI_COLLISION_CIRCLE>(a, sum, inj, bp_n, bp_s, nbp, k_first, check_from, first_change, st);
    } else if (model == MPPI_MODEL_BICYCLE) {
        if (coll == MPPI_COLLISION_NONE) return launch_strict_mc<MPPI_MODEL_BICYCLE, MPPI_COLLISION_NONE>(a, sum, inj, bp_n, bp_s, nbp, k_first, check_from, first_change, st);
        if (coll == MPPI_COLLISION_FOOTPRINT) return launch_strict_mc<MPPI_MODEL_BICYCLE, MPPI_COLLISION_FOOTPRINT>(a, sum, inj, bp_n, bp_s, nbp, k_first, check_from, first_change, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t mppi_launch_p2p_barrier(const TickArgs &a, unsigned long long count, cudaStream_t st) {
    mppi_p2p_barrier_kernel<<<1, 32, 0, st>>>(a, count);
    return cudaGetLastError();
}

cudaError_t mppi_launch_merge(const TickArgs &a, const float *triples, int G, cudaStream_t st) {
    mppi_merge_kernel<<<1, MPPI_BLOCK, 0, st>>>(a, triples, G);
    return cudaGetLastError();
}

cudaError_t mppi_launch_traj(const TickArgs &a, int model, const float *rec, float *d_opt, float *d_samp,
                             const int *d_sel, int n_sel, int shift, cudaStream_t st) {
    const int n = (d_sel ? n_sel : a.K) + 1;
    if (model == MPPI_MODEL_BICYCLE) mppi_traj_kernel<MPPI_MODEL_BICYCLE><<<(n + 127) / 128, 128, 0, st>>>(a, rec, d_opt, d_samp, d_sel, n_sel, shift);
    else mppi_traj_kernel<MPPI_MODEL_DIFFDRIVE><<<(n + 127) / 128, 128, 0, st>>>(a, rec, d_opt, d_samp, d_sel, n_sel, shift);
    return cudaGetLastError();
}

cudaError_t mppi_launch_traj_controls(const TickArgs &a, const float *rec, float *d_ctl, const int *d_sel, int n_rows, int shift,
                                      cudaStream_t st) {
    mppi_traj_controls_kernel<<<(n_rows + 1 + 127) / 128, 128, 0, st>>>(a, rec, reinterpret_cast<float2 *>(d_ctl), d_sel, n_rows, shift);
    return cudaGetLastError();
}

cudaError_t mppi_launch_noise(const TickArgs &a, float *d_out, int robot, cudaStream_t st) {
    mppi_noise_kernel<<<(a.K + 255) / 256, 256, 0, st>>>(a, d_out, robot);
    return cudaGetLastError();
}

// ---- per-robot scenes (fleets): the caller's device rows converted into the handle's SceneRec table, in stream order ----
namespace {
// thread (r, j): obstacle slot j of robot r; the FP64 arithmetic is spelled out (no FMA contraction) so r2 / far2 carry the
// bits refresh_obstacle_args gives the same obstacle on the host
__global__ void mppi_scene_obstacles_kernel(const float *__restrict__ obs, const int *__restrict__ count, int R, int m, int ncol,
                                            bool circle, double rr_base, double diag, SceneRec *__restrict__ scene) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * MPPI_MAX_OBSTACLES) return;
    const int r = i / MPPI_MAX_OBSTACLES, j = i - r * MPPI_MAX_OBSTACLES;
    SceneRec &s = scene[r];
    if (j == 0) s.n_obs = count ? max(0, min(count[r], m)) : m;
    float x = 0.f, y = 0.f, r2 = 0.f, far2 = 0.f, vx = 0.f, vy = 0.f;
    if (j < m) {
        const float *row = obs + ((size_t)r * m + j) * ncol;
        x = row[0]; y = row[1];
        if (ncol == 4) {
            vx = row[2]; vy = row[3];
        } else {
            const double rad = (double)row[2];
            const double rr = circle ? __dadd_rn(rr_base, rad) : rad;
            r2 = (float)__dmul_rn(rr, rr);
            const double far = __dadd_rn(__dmul_rn(__dadd_rn(diag, rad), 1.001), 1e-3);
            far2 = (float)__dmul_rn(far, far);
        }
    }
    s.obs_x[j] = x; s.obs_y[j] = y; s.obs_r2[j] = r2; s.obs_far2[j] = far2; s.obs_vx[j] = vx; s.obs_vy[j] = vy;
}

__global__ void mppi_scene_goals_kernel(const float *__restrict__ goal, int R, int n, SceneRec *__restrict__ scene) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * 4) return;
    const int r = i >> 2, c = i & 3;
    scene[r].goal[c] = c < n ? goal[(size_t)r * n + c] : 0.f;
}
}  // namespace

cudaError_t mppi_launch_scene_obstacles(const float *d_obs, const int *d_count, int R, int m, int ncol, bool circle,
                                        double rr_base, double diag, SceneRec *d_scene, cudaStream_t st) {
    const int n = R * MPPI_MAX_OBSTACLES;
    mppi_scene_obstacles_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_obs, d_count, R, m, ncol, circle, rr_base, diag, d_scene);
    return cudaGetLastError();
}

cudaError_t mppi_launch_scene_goals(const float *d_goal, int R, int n, SceneRec *d_scene, cudaStream_t st) {
    mppi_scene_goals_kernel<<<(R * 4 + 255) / 256, 256, 0, st>>>(d_goal, R, n, d_scene);
    return cudaGetLastError();
}
