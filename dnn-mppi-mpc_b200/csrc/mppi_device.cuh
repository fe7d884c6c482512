// Device-side building blocks of the MPPI tick for sm_100a: Philox noise, dynamics steps,
// nearest-waypoint search, state costs, collision tests.  Reference semantics (file:line
// relative to the reference tree) are cited per function; SURVEY.md Appendix A is the spec.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math_constants.h>
#include <type_traits>
#include "../../include/mppi_b200.h"

// -DMPPI_DEBUG_CHECKS=1: device-side bounds / protocol assertions at every shared-memory and global hand-off (the build the
// sanitize subset runs when compute-sanitizer is not available on the pool; a failed check traps the kernel)
#ifndef MPPI_DEBUG_CHECKS
#define MPPI_DEBUG_CHECKS 0
#endif
#if MPPI_DEBUG_CHECKS
#include <assert.h>
#define MPPI_DCHECK(c) assert(c)
#else
#define MPPI_DCHECK(c) ((void)0)
#endif
#ifndef MPPI_BLOCK
#define MPPI_BLOCK 256
#endif
#define MPPI_WARPS (MPPI_BLOCK / 32)
#ifndef MPPI_SPT
#define MPPI_SPT 1                     // samples per thread of the tick kernel: independent rollouts interleaved in one
#endif                                 // instruction stream (ILP); a CTA walks its range in chunks of MPPI_CHUNK samples
#define MPPI_CHUNK (MPPI_BLOCK * MPPI_SPT)
#ifndef MPPI_MIN_BLOCKS
#define MPPI_MIN_BLOCKS (MPPI_BLOCK >= 512 ? 1 : 768 / MPPI_BLOCK)   // resident CTAs per SM the regenerate-noise tick kernels are register-budgeted for
#endif
#define MPPI_STASH_BLOCKS (MPPI_BLOCK >= 512 ? 1 : 512 / MPPI_BLOCK)  // ... and the stash kernels (512 samples' noise fill shared memory)
#define MPPI_PENALTY 1.0e10f           // mppi_race_car_obstacle.py:157
#define MPPI_SENTINEL 1.0e18f          // padded window entries: distance^2 = 1e36, never the minimum
#define MPPI_OUT_HDR 12                // u0 (post-shift, Q8), idx, rho, ncoll, eta, ess, p2p flag, first row of the PRE-shift nominal,
                                       // [10] non-finite-cost fault (the tick was not applied), [11] spare
#define MPPI_OUT_PEER_TIMEOUT 7
#define MPPI_OUT_FAULT 10
#define MPPI_OUT_STRIDE (MPPI_OUT_HDR + 8 * MPPI_MAX_T)   // header, U shifted, w_eps, U pre-shift, U before the tick
#define MPPI_OUT_UPRE (MPPI_OUT_HDR + 4 * MPPI_MAX_T)
#define MPPI_OUT_UOLD (MPPI_OUT_HDR + 6 * MPPI_MAX_T)
#define MPPI_NF(T) (4 + 2 * (T))
#define MPPI_MERGE_GROUP_CTAS 16         // two-level merge of the block partials: consecutive CTAs per group
#define MPPI_NF_MAX MPPI_NF(MPPI_MAX_T)
// exchange buffer of one rank (fused multi-GPU exchange): 2 parities x [MPPI_MAX_PEERS triples of NF_MAX 64-bit words];
// a word is (sequence number << 32 | float bits): the flag travels WITH the datum in one 8-byte store (the "LL" protocol),
// so a reader that sees the tick's sequence number in a word has that word's datum -- no fence, no separate flag
#define MPPI_XCHG_SLOT(par, r) (((par) * MPPI_MAX_PEERS + (r)) * MPPI_NF_MAX)
#define MPPI_XCHG_WORDS (2 * MPPI_MAX_PEERS * MPPI_NF_MAX)
#define MPPI_XCHG_TRACE 8              // globaltimer stamps of the last exchange (diagnostics), kept behind the words
#define MPPI_XCHG_BARRIER (MPPI_XCHG_WORDS + MPPI_XCHG_TRACE)   // then MPPI_MAX_PEERS words of the device-side rank barrier
#define MPPI_XCHG_TOTAL (MPPI_XCHG_BARRIER + MPPI_MAX_PEERS)

enum : int {
    F_WRITE_S = 1,       // store per-sample costs
    F_UPDATE = 2,        // weights + weighted noise + merge
    F_FROM_S = 4,        // skip the rollout, read costs from S_in (K2 alone)
    F_HOST_IDX = 8,      // skip step 1, window starts at idx_host
    F_TRIPLE_OUT = 16,   // multi-GPU: publish the merged per-GPU triple, do not finalize
    F_KEEP_IDX = 32,     // do not persist the waypoint index (K2 alone)
    F_IDX_ONLY = 64,     // only run step 1 and persist the index (MLP path, K1 alone)
    F_P2P = 128,         // multi-GPU: exchange the per-GPU triples over peer memory inside this kernel
    F_COST_SUM = 0x10000 // MLP kernel: cost_mode == sum (the tick kernel takes it as a template argument)
};

// One robot's scene in a fleet (mppi_set_robot_goals / mppi_set_robot_obstacles): the handle keeps one record per robot
// ([R], device), and a scene tick kernel loads its robot's record into shared memory in the prologue.  The fields carry the
// names TickArgs gives the shared scene, so collided / goal_cost / target_soft_cost read either one through a template.
struct SceneRec {
    float goal[4];                        // GOAL: (x, y); TARGET_SOFT: desired pose (x, y, yaw)
    int n_obs, pad_[3];                   // obstacles this robot uses (rows 0 .. n_obs - 1)
    float obs_x[MPPI_MAX_OBSTACLES], obs_y[MPPI_MAX_OBSTACLES];
    float obs_r2[MPPI_MAX_OBSTACLES], obs_far2[MPPI_MAX_OBSTACLES];     // as refresh_obstacle_args computes them (FP64)
    float obs_vx[MPPI_MAX_OBSTACLES], obs_vy[MPPI_MAX_OBSTACLES];       // TARGET_SOFT: moving obstacles
};
#define MPPI_SCENE_GOAL 1                 // TickArgs::scene_mask: the goal comes from the per-robot table
#define MPPI_SCENE_OBS 2                  // ... the obstacles come from the per-robot table

// Everything a tick needs, passed by value (kernel parameter = constant bank).
struct TickArgs {
    // static configuration
    int K, T, window, n_path, n_obs, yaw_wrap, use_gamma, clamp_nominal;
    int k_offset, n_exploit;          // global sample index of local sample 0; Q6 threshold on the global index
    float dt, dt_over_L, umax0, umax1;
    float sw[4], tw[4];
    float gq[4];                      // gamma * Sigma^-1, row-major
    float chol[3];                    // L00, L10, L11 of Sigma = L L^T
    float inv_temp;
    float obs_x[MPPI_MAX_OBSTACLES], obs_y[MPPI_MAX_OBSTACLES];
    float obs_r2[MPPI_MAX_OBSTACLES];     // collision radius^2: r^2 (footprint) or (r_robot*margin + r)^2 (circle)
    float obs_far2[MPPI_MAX_OBSTACLES];   // footprint quick reject: (half diagonal + r)^2, inflated
    float fp_hl, fp_hw;                   // footprint half length / half width incl. margin
    // cost kinds without a reference path (template WIN = MPPI_WIN_GOAL / MPPI_WIN_TARGET)
    float goal[4];                        // GOAL: (x, y); TARGET_SOFT: desired pose (x, y, yaw)
    float ctrl_w[2];                      // TARGET_SOFT: diagonal of R
    float soft_w, soft_sd;                // TARGET_SOFT: obstacle weight, safety distance
    float obs_vx[MPPI_MAX_OBSTACLES], obs_vy[MPPI_MAX_OBSTACLES];   // TARGET_SOFT: obstacle velocities (position = obs + vel * t*dt)
    // per tick
    float x0[4];
    uint32_t seed_lo, seed_hi, tick;
    int idx_host, flags;
    // pointers (device)
    const float4 *path;               // [n_path] (x, y, yaw, v); per-robot paths: [R][path_stride], robot r uses path_len[r] rows
    const int *path_len;              // null: every robot follows the one shared path
    int path_stride;
    const float *x0_dev;              // batched: [R][4], else null
    float *U;                         // [R][T][2] nominal, updated in place
    int *idx;                         // [R] carried waypoint index
    const float *M;                   // [T][T] filter operator
    const float *eps;                 // injected noise (K,T,2) or null
    float *S;                         // [R][K] costs out (F_WRITE_S) / in (F_FROM_S)
    int *NC;                          // [K] collided-evaluation counts kept apart from S (strict path), or null
    float *S_user;                    // [K] combined cost smooth + 1e10*n for the caller (strict path), or null
    float *part;                      // [R][B][NF]
    unsigned *ticket;                 // [R]
    float *part2;                     // [R][merge_gmax][NF]: partials of the merge groups (two-level merge)
    unsigned *ticket2;                // [R][merge_gmax]
    int merge_gmax;                   // groups of MPPI_MERGE_GROUP_CTAS consecutive CTAs a robot's grid row may have
    float *out;                       // [R][MPPI_OUT_STRIDE]
    float *out_host;                  // mapped pinned mirror of out (robot 0) or null
    float *u0_out;                    // batched: [R][2] or null
    float *triple_out;                // [NF] per-GPU triple (F_TRIPLE_OUT)
    float *plant_state;               // closed loop: [R][4] plant states, advanced by each robot's last block after the update, or null
    float *plant_log;                 // closed loop: [(n+1)][R][4] states and [n][R][2] controls behind them
    int plant_mode, plant_tick, plant_n;
    // graph-captured closed loop: every launch carries the SAME arguments; the running tick lives on the device.
    // loop_state[0] = absolute tick of this launch (added to `tick`), [1] = first tick of the loop (log row = [0] - [1]);
    // the grid's last CTA to finish (loop_ticket over all gridDim.x * gridDim.y CTAs) advances [0].  Null otherwise.
    unsigned *loop_state;
    unsigned *loop_ticket;
    // fused multi-GPU exchange (F_P2P): peer_buf[p] = rank p's exchange buffer (own buffer at index p2p_rank)
    unsigned long long *peer_buf[MPPI_MAX_PEERS];
    int p2p_rank, p2p_world;
    unsigned p2p_seq;
    unsigned p2p_timeout_ms;          // a peer that has not published within this time fails the tick (MPPI_E_NCCL)
    unsigned long long *trace;        // diagnostics (mppi_set_trace): %globaltimer of CTA b's start [2b] and end of its rollouts
                                      // [2b+1], then the last CTA's merge done [2B] and nominal updated [2B+1]; or null
    // per-robot scenes (read by the scene instantiations of the tick kernel only): [R] records; the components named in
    // scene_mask come from the robot's record, the others from the shared fields above
    const SceneRec *scene;
    int scene_mask;
};

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11) + Box-Muller.  Replaces np.random.multivariate_normal
// in _calc_epsilon (mppi_differential_drive.py:273-283).  Spec: oracle/mppi_oracle.py:philox_noise.
//   counter = (global sample k, timestep pair t/2, tick, robot), key = seed
//   u_i = ((r_i >> 9) + 0.5) * 2^-23  in (0,1);  z = sqrt(-2 ln u_a) * (cos, sin)(2 pi (u_b - 1/2))
//   (angle in (-pi, pi): the range where MUFU.SIN/COS are most accurate)
//   outputs (r0,r1) -> timestep 2p, (r2,r3) -> timestep 2p+1;  eps = chol(Sigma) z
// All float ops use explicit-rounding intrinsics so every kernel produces identical bits.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t &c0, uint32_t &c1, uint32_t &c2, uint32_t &c3,
                                              uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1;
        c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

__device__ __forceinline__ float u01_open(uint32_t r) {
    // ((r >> 9) + 0.5) * 2^-23, exact: [1,2) mantissa trick minus (1 - 2^-24)
    return __fadd_rn(__uint_as_float(0x3f800000u | (r >> 9)), -0.99999994f);
}

__device__ __forceinline__ void box_muller(uint32_t ra, uint32_t rb, float &z0, float &z1) {
    const float ua = u01_open(ra), ub = u01_open(rb);
    float rad;                                                                     // sqrt(-2 ln ua)
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(__fmul_rn(-1.3862943611198906f, __log2f(ua))));
    const float ang = __fmul_rn(6.2831853071795865f, __fadd_rn(ub, -0.5f));
    z0 = __fmul_rn(rad, __cosf(ang));
    z1 = __fmul_rn(rad, __sinf(ang));
}

// eps for timesteps 2p (e[0],e[1]) and 2p+1 (e[2],e[3]) of global sample k
// `tick_add`: tick offset supplied on the device (graph-captured closed loops read the running tick from memory)
__device__ __forceinline__ void philox_eps_pair(const TickArgs &a, uint32_t k, uint32_t p, uint32_t robot, float e[4], uint32_t tick_add = 0u) {
    uint32_t c0 = k, c1 = p, c2 = a.tick + tick_add, c3 = robot;
    philox4x32_10(c0, c1, c2, c3, a.seed_lo, a.seed_hi);
    float z0, z1, z2, z3;
    box_muller(c0, c1, z0, z1);
    box_muller(c2, c3, z2, z3);
    e[0] = __fmul_rn(a.chol[0], z0);
    e[1] = __fmaf_rn(a.chol[1], z0, __fmul_rn(a.chol[2], z1));
    e[2] = __fmul_rn(a.chol[0], z2);
    e[3] = __fmaf_rn(a.chol[1], z2, __fmul_rn(a.chol[2], z3));
}

#ifndef MPPI_KEYIDX_SMEM
#define MPPI_KEYIDX_SMEM 1      // index addends of the first-minimum key from shared memory (hoisted LDS.128) instead of 20
#endif                          // immediates re-materialised by MOVs in every loop iteration: 365 -> 349 instructions, +1.7 %
// ------------------------------------------------------------------------------------------
// shared-memory view of one robot's tick constants
// ------------------------------------------------------------------------------------------
struct TickSmem {
    float2 U[MPPI_MAX_T];                  // nominal
    float2 Q[MPPI_MAX_T];                  // gamma * Sigma^-1 applied to U[t] (row vector u^T Sigma^-1)
    __align__(16) float wx[MPPI_MAX_WINDOW];   // window SoA of NEGATED coordinates, padded with sentinels
    __align__(16) float wy[MPPI_MAX_WINDOW];   // to a multiple of 16 entries (static window 20: exactly 20)
    float2 wyv[MPPI_MAX_WINDOW];           // (yaw, v) of each window entry, for the lookup after the argmin
    float x0[4];
    int win_start, n_win16;                // absolute index of window entry 0; padded length / 16
    float4 cb[MPPI_MAX_WINDOW / 16];       // dynamic window: bounding circle (cx, cy, r) of every 16-entry chunk
    // static 20-entry window, expanded form (MPPI_WIN20_EXPANDED): coordinates relative to the window centre and their
    // squared norms, d_j - |p'|^2 = ec_j - 2 p'.(ex_j, ey_j)
    __align__(16) float ex[20];
    __align__(16) float ey[20];
    __align__(16) float ec[20];
    float c2x, c2y;                        // twice the centre
#if MPPI_KEYIDX_SMEM
    __align__(16) float kidx[20];          // 0..19: the index addends of the first-minimum key, read as LDS.128
#endif
};

// Fills the expanded-form arrays of the static window from the (already written) negated coordinates; entries past the
// path end (sentinels) get distance 1e30.  Call between the barriers of the prologue, any thread count.
__device__ __forceinline__ void fill_window_expanded(TickSmem &sm, int nw, int tid, int nthreads) {
    const int jc = nw > 10 ? 10 : nw - 1;
    const float cx = -sm.wx[jc], cy = -sm.wy[jc];
    for (int j = tid; j < 20; j += nthreads) {
        const float wx = __fsub_rn(-sm.wx[j], cx), wy = __fsub_rn(-sm.wy[j], cy);
        const bool valid = j < nw;
        sm.ex[j] = valid ? wx : 0.f;
        sm.ey[j] = valid ? wy : 0.f;
        sm.ec[j] = valid ? __fmaf_rn(wy, wy, __fmul_rn(wx, wx)) : 1e30f;
    }
    if (tid == 0) { sm.c2x = 2.f * cx; sm.c2y = 2.f * cy; }
#if MPPI_KEYIDX_SMEM
    for (int j = tid; j < 20; j += nthreads) sm.kidx[j] = (float)j;
#endif
}

// Bounding circle of the window entries path[first .. first + n_valid) (one 16-entry chunk of the dynamic window).
// nearest_wp<0> skips a chunk only when this circle proves every point in it farther than the best found so far,
// so the argmin stays exactly the reference's (first minimum over the whole window).
// Reads the window from SHARED memory (negated coordinates, already staged): 32 dependent global loads per thread here
// were several microseconds of every CTA's prologue, which is what a K = 16 384 tick is made of.
__device__ __forceinline__ float4 chunk_bound(const float *nwx, const float *nwy, int first, int n_valid) {
    float xmin = CUDART_INF_F, xmax = -CUDART_INF_F, ymin = CUDART_INF_F, ymax = -CUDART_INF_F;
#pragma unroll 4
    for (int j = 0; j < n_valid; ++j) {
        const float px = -nwx[first + j], py = -nwy[first + j];
        xmin = fminf(xmin, px); xmax = fmaxf(xmax, px); ymin = fminf(ymin, py); ymax = fmaxf(ymax, py);
    }
    const float cx = 0.5f * (xmin + xmax), cy = 0.5f * (ymin + ymax);
    float r2 = 0.f;
#pragma unroll 4
    for (int j = 0; j < n_valid; ++j) {
        const float dx = -nwx[first + j] - cx, dy = -nwy[first + j] - cy;
        r2 = fmaxf(r2, fmaf(dy, dy, dx * dx));
    }
    return make_float4(cx, cy, sqrtf(r2) * 1.00001f + 1e-6f, 0.f);
}

// ---- packed FP32 (Blackwell FADD2 / FMUL2 / FFMA2): two FP32 ops per issue slot ------------
__device__ __forceinline__ float2 f2_add(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b), rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b),
                       rc = *reinterpret_cast<unsigned long long *>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2 *>(&rd);
}

// First-min argmin over one chunk of CH window entries (CH % 4 == 0), branch-free and almost
// entirely on the FMA pipe:  d_j = (x-px_j)^2 + (y-py_j)^2 as FFMA2 pairs;  m = min_j d_j (FMNMX3);
// key_j = (d_j - m) * 2^100 + j, which is exactly j where d_j == m and >= 2^76 elsewhere, so
// min_j key_j is the FIRST index attaining the minimum (the d.index(min(d)) / np.argmin rule).
// The window arrays hold NEGATED coordinates so the differences are plain packed adds.
#ifndef MPPI_WP_CHUNK_ILP
#define MPPI_WP_CHUNK_ILP 1
#endif
#ifndef MPPI_WP_FULL
#define MPPI_WP_FULL 0          // 1: dynamic window without pruning (A/B: slower at every K, 70 -> 78 us at K = 1024)
#endif
#ifndef MPPI_WIN20_EXPANDED
#define MPPI_WIN20_EXPANDED 1   // static window distances as ec_j - 2 p'.w'_j: 2 packed FMAs per waypoint pair instead of 4 ops (0: direct form)
#endif
#ifndef MPPI_ARGMIN_KEY_SEL
#define MPPI_ARGMIN_KEY_SEL 0   // 1: first-min index by FSETP/SEL chains on the ALU pipe (A/B variant, see profiles/)
#endif
#ifndef MPPI_MIN_TREE
#define MPPI_MIN_TREE 1         // tree-shaped FMNMX3 reductions in the static-window argmin (0: chains of 10; +2.9 % on B200)
#endif
#ifndef MPPI_ARGMIN_PACK
#define MPPI_ARGMIN_PACK 2      // 2: all FP32 work packed (FFMA2); 1: differences scalar, rest packed; 0: all scalar
#endif
// Minimum of N register values as a tree of 3-input minima.  Compile-time recursion: every index is a constant after inlining, so
// the values stay in registers (a run-time `while (n > 1)` over the array, however unrollable it looks, sent the 16-entry chunks
// of the dynamic window through local memory: 91 registers + a stack frame instead of 126, race-car ticks 2.5x slower).
template <int N>
__device__ __forceinline__ float min_tree3(const float (&t)[N]) {
    if constexpr (N == 1) return t[0];
    else if constexpr (N == 2) return fminf(t[0], t[1]);
    else if constexpr (N == 3) return fminf(fminf(t[0], t[1]), t[2]);
    else {
        constexpr int N3 = N / 3, REM = N - 3 * N3, M = N3 + (REM ? 1 : 0);
        float u[M];
#pragma unroll
        for (int i = 0; i < N3; ++i) u[i] = fminf(fminf(t[3 * i], t[3 * i + 1]), t[3 * i + 2]);
        if constexpr (REM == 2) u[N3] = fminf(t[3 * N3], t[3 * N3 + 1]);
        else if constexpr (REM == 1) u[N3] = t[3 * N3];
        return min_tree3<M>(u);
    }
}
template <int CH>
__device__ __forceinline__ void chunk_argmin(const float4 *nwx4, const float4 *nwy4, float x, float y,
                                             float &m_out, float &key_out) {
    const float2 xx = make_float2(x, x), yy = make_float2(y, y);
    float2 d[CH / 2];
#pragma unroll
    for (int q = 0; q < CH / 4; ++q) {
        const float4 X = nwx4[q], Y = nwy4[q];
#if MPPI_ARGMIN_PACK == 2
        const float2 dxa = f2_add(xx, make_float2(X.x, X.y)), dya = f2_add(yy, make_float2(Y.x, Y.y));
        const float2 dxb = f2_add(xx, make_float2(X.z, X.w)), dyb = f2_add(yy, make_float2(Y.z, Y.w));
        d[2 * q] = f2_fma(dya, dya, f2_mul(dxa, dxa));
        d[2 * q + 1] = f2_fma(dyb, dyb, f2_mul(dxb, dxb));
#elif MPPI_ARGMIN_PACK == 1
        const float2 dxa = make_float2(x + X.x, x + X.y), dya = make_float2(y + Y.x, y + Y.y);
        const float2 dxb = make_float2(x + X.z, x + X.w), dyb = make_float2(y + Y.z, y + Y.w);
        d[2 * q] = f2_fma(dya, dya, f2_mul(dxa, dxa));
        d[2 * q + 1] = f2_fma(dyb, dyb, f2_mul(dxb, dxb));
#else
        float dx, dy;
        dx = x + X.x; dy = y + Y.x; d[2 * q].x = fmaf(dy, dy, dx * dx);
        dx = x + X.y; dy = y + Y.y; d[2 * q].y = fmaf(dy, dy, dx * dx);
        dx = x + X.z; dy = y + Y.z; d[2 * q + 1].x = fmaf(dy, dy, dx * dx);
        dx = x + X.w; dy = y + Y.w; d[2 * q + 1].y = fmaf(dy, dy, dx * dx);
#endif
    }
#if MPPI_MIN_TREE
    // minimum of the CH distances as a tree of 3-input minima (depth ~3) instead of a chain of CH/2 dependent ones
    float m;
    {
        float t[CH / 2];
#pragma unroll
        for (int i = 0; i < CH / 2; ++i) t[i] = fminf(d[i].x, d[i].y);
        m = min_tree3<CH / 2>(t);
    }
#else
    float m = fminf(d[0].x, d[0].y);
#pragma unroll
    for (int i = 1; i < CH / 2; ++i) m = fminf(fminf(m, d[i].x), d[i].y);
#endif
#if MPPI_ARGMIN_KEY_SEL
    // index of the first minimum on the ALU pipe: descending select chains (the lowest index is written last), four
    // independent chains of CH/4 entries; FSETP + SEL per entry instead of FADD2 + FFMA2 per pair on the FMA pipe
    {
        float k0 = (float)CH, k1 = (float)CH, k2 = (float)CH, k3 = (float)CH;
#pragma unroll
        for (int i = CH / 8 - 1; i >= 0; --i) {
            const int a0 = i, a1 = i + CH / 8, a2 = i + 2 * (CH / 8), a3 = i + 3 * (CH / 8);     // float2 slots of the 4 chains
            k0 = d[a0].y == m ? (float)(2 * a0 + 1) : k0; k0 = d[a0].x == m ? (float)(2 * a0) : k0;
            k1 = d[a1].y == m ? (float)(2 * a1 + 1) : k1; k1 = d[a1].x == m ? (float)(2 * a1) : k1;
            k2 = d[a2].y == m ? (float)(2 * a2 + 1) : k2; k2 = d[a2].x == m ? (float)(2 * a2) : k2;
            k3 = d[a3].y == m ? (float)(2 * a3 + 1) : k3; k3 = d[a3].x == m ? (float)(2 * a3) : k3;
        }
        if (CH % 8) {                                   // CH = 20: slots 8, 9 are left over by the 4 x 2 split
#pragma unroll
            for (int a = CH / 2 - 1; a >= 4 * (CH / 8); --a) {
                k3 = d[a].y == m ? (float)(2 * a + 1) : k3; k3 = d[a].x == m ? (float)(2 * a) : k3;
            }
            // chain 3 now covers slots 6, 7 (written earlier) and 8, 9 (written later): redo 6, 7 so the lower index wins
#pragma unroll
            for (int a = 4 * (CH / 8) - 1; a >= 3 * (CH / 8); --a) {
                k3 = d[a].y == m ? (float)(2 * a + 1) : k3; k3 = d[a].x == m ? (float)(2 * a) : k3;
            }
        }
        m_out = m;
        key_out = fminf(fminf(k0, k1), fminf(k2, k3));
        return;
    }
#endif
    const float2 nm = make_float2(-m, -m), huge = make_float2(1.2676506e30f, 1.2676506e30f);
#if MPPI_MIN_TREE
    float kt[CH / 2];
#pragma unroll
    for (int i = 0; i < CH / 2; ++i) {
        const float2 k2 = f2_fma(f2_add(d[i], nm), huge, make_float2((float)(2 * i), (float)(2 * i + 1)));
        kt[i] = fminf(k2.x, k2.y);
    }
    m_out = m;
    key_out = min_tree3<CH / 2>(kt);
#else
    float key = CUDART_INF_F;
#pragma unroll
    for (int i = 0; i < CH / 2; ++i) {
#if MPPI_ARGMIN_PACK >= 1
        const float2 k2 = f2_fma(f2_add(d[i], nm), huge, make_float2((float)(2 * i), (float)(2 * i + 1)));
#else
        const float2 k2 = make_float2(fmaf(d[i].x - m, 1.2676506e30f, (float)(2 * i)), fmaf(d[i].y - m, 1.2676506e30f, (float)(2 * i + 1)));
#endif
        key = fminf(fminf(key, k2.x), k2.y);
    }
    m_out = m;
    key_out = key;
#endif
}

// A8: first-min argmin of squared xy distance over the window
// (mppi_differential_drive.py:201-220, mppi_race_car_obstacle.py:173-191).
template <int WIN>
__device__ __forceinline__ int nearest_wp(const TickSmem &sm, float x, float y) {
    const float4 *nwx4 = reinterpret_cast<const float4 *>(sm.wx);
    const float4 *nwy4 = reinterpret_cast<const float4 *>(sm.wy);
    if (WIN == 20) {
#if MPPI_WIN20_EXPANDED
        // squared distances up to the common term |p'|^2, in coordinates relative to the window centre (|w'| <= ~1 m, so
        // the cancellation costs no more than the FP32 rounding of the absolute path coordinates does in the direct form)
        const float ax = fmaf(-2.f, x, sm.c2x), ay = fmaf(-2.f, y, sm.c2y);
        const float2 axx = make_float2(ax, ax), ayy = make_float2(ay, ay);
        const float4 *ex4 = reinterpret_cast<const float4 *>(sm.ex), *ey4 = reinterpret_cast<const float4 *>(sm.ey);
        const float4 *ec4 = reinterpret_cast<const float4 *>(sm.ec);
        float2 d[10];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            const float4 X = ex4[q], Y = ey4[q], C = ec4[q];
            d[2 * q] = f2_fma(make_float2(Y.x, Y.y), ayy, f2_fma(make_float2(X.x, X.y), axx, make_float2(C.x, C.y)));
            d[2 * q + 1] = f2_fma(make_float2(Y.z, Y.w), ayy, f2_fma(make_float2(X.z, X.w), axx, make_float2(C.z, C.w)));
        }
#if MPPI_MIN_TREE
        // the two 20-input minima as TREES of 3-input FMNMX3 (depth 3) instead of chains of 10 dependent ones: the
        // horizon recurrence leaves a sample no other work to hide ~80 cycles of chain latency per step behind
        const float m = fminf(fminf(fminf(fminf(d[0].x, d[0].y), d[1].x), fminf(fminf(d[1].y, d[2].x), d[2].y)),
                              fminf(fminf(fminf(fminf(d[3].x, d[3].y), d[4].x), fminf(fminf(d[4].y, d[5].x), d[5].y)),
                                    fminf(fminf(fminf(fminf(d[6].x, d[6].y), d[7].x), fminf(fminf(d[7].y, d[8].x), d[8].y)),
                                          fminf(d[9].x, d[9].y))));
        const float2 nm = make_float2(-m, -m), huge = make_float2(1.2676506e30f, 1.2676506e30f);
        const float4 *ki4 = reinterpret_cast<const float4 *>(sm.kidx);
        float2 kk[10];
#pragma unroll
        for (int i = 0; i < 10; i += 2) {
            const float4 ki = ki4[i >> 1];
            kk[i] = f2_fma(f2_add(d[i], nm), huge, make_float2(ki.x, ki.y));
            kk[i + 1] = f2_fma(f2_add(d[i + 1], nm), huge, make_float2(ki.z, ki.w));
        }
        const float key = fminf(fminf(fminf(fminf(kk[0].x, kk[0].y), kk[1].x), fminf(fminf(kk[1].y, kk[2].x), kk[2].y)),
                                fminf(fminf(fminf(fminf(kk[3].x, kk[3].y), kk[4].x), fminf(fminf(kk[4].y, kk[5].x), kk[5].y)),
                                      fminf(fminf(fminf(fminf(kk[6].x, kk[6].y), kk[7].x), fminf(fminf(kk[7].y, kk[8].x), kk[8].y)),
                                            fminf(kk[9].x, kk[9].y))));
        return __float2int_rn(key);
#else
        float m = fminf(d[0].x, d[0].y);
#pragma unroll
        for (int i = 1; i < 10; ++i) m = fminf(fminf(m, d[i].x), d[i].y);
        const float2 nm = make_float2(-m, -m), huge = make_float2(1.2676506e30f, 1.2676506e30f);
        float key = CUDART_INF_F;
#if MPPI_KEYIDX_SMEM
        const float4 *ki4 = reinterpret_cast<const float4 *>(sm.kidx);
#pragma unroll
        for (int i = 0; i < 10; i += 2) {
            const float4 ki = ki4[i >> 1];
            const float2 ka = f2_fma(f2_add(d[i], nm), huge, make_float2(ki.x, ki.y));
            const float2 kb = f2_fma(f2_add(d[i + 1], nm), huge, make_float2(ki.z, ki.w));
            key = fminf(fminf(key, ka.x), ka.y);
            key = fminf(fminf(key, kb.x), kb.y);
        }
#else
#pragma unroll
        for (int i = 0; i < 10; ++i) {
            const float2 k2 = f2_fma(f2_add(d[i], nm), huge, make_float2((float)(2 * i), (float)(2 * i + 1)));
            key = fminf(fminf(key, k2.x), k2.y);
        }
#endif
        return __float2int_rn(key);
#endif
#else
        float m, key;
        chunk_argmin<20>(nwx4, nwy4, x, y, m, key);
        return __float2int_rn(key);
#endif
    }
    // dynamic window: chunks of 16 entries (the window is padded with sentinels to a multiple of 16)
    float bm = CUDART_INF_F, sbm = CUDART_INF_F;      // best squared distance so far and its square root
    int bj = 0;
    const int nch = sm.n_win16;
    int c = 0;
#if MPPI_WP_FULL
    // A/B variant: every chunk evaluated, no pruning, four independent chunk chains per trip (block-uniform trip count)
    for (; c + 3 < nch; c += 4) {
        float m0, k0, m1, k1, m2, k2, m3, k3;
        chunk_argmin<16>(nwx4 + 4 * c, nwy4 + 4 * c, x, y, m0, k0);
        chunk_argmin<16>(nwx4 + 4 * c + 4, nwy4 + 4 * c + 4, x, y, m1, k1);
        chunk_argmin<16>(nwx4 + 4 * c + 8, nwy4 + 4 * c + 8, x, y, m2, k2);
        chunk_argmin<16>(nwx4 + 4 * c + 12, nwy4 + 4 * c + 12, x, y, m3, k3);
        const bool s01 = m1 < m0, s23 = m3 < m2;
        const float ma = s01 ? m1 : m0, mb = s23 ? m3 : m2;
        const float ka = s01 ? k1 + 16.f : k0, kb = s23 ? k3 + 48.f : k2 + 32.f;
        const bool sb = mb < ma;
        const float m = sb ? mb : ma;
        const int j = 16 * c + __float2int_rn(sb ? kb : ka);
        if (m < bm) { bm = m; bj = j; }
    }
    for (; c < nch; ++c) {
        float m, key;
        chunk_argmin<16>(nwx4 + 4 * c, nwy4 + 4 * c, x, y, m, key);
        if (m < bm) { bm = m; bj = 16 * c + __float2int_rn(key); }
    }
    (void)sbm;
    return bj;
#endif
    // |z - p| >= |z - centre| - r for every point p of a chunk: if that exceeds the best distance (with a 1e-4 relative
    // margin, three orders above FP32 rounding) no point of the chunk can be the minimum or tie with it
    auto far = [&](int ch) {
        const float4 cb = sm.cb[ch];
        const float ex = x - cb.x, ey = y - cb.y, R = sbm + cb.z;
        return fmaf(ey, ey, ex * ex) > R * R * 1.0002f;
    };
#if MPPI_WP_CHUNK_ILP
    // two chunks per trip: their (independent) distance / min / key chains overlap, which is what a latency-bound
    // small-K tick needs; the earlier chunk still wins ties
    for (; c + 1 < nch; c += 2) {
        if (far(c) && far(c + 1)) continue;
        float m0, k0, m1, k1;
        chunk_argmin<16>(nwx4 + 4 * c, nwy4 + 4 * c, x, y, m0, k0);
        chunk_argmin<16>(nwx4 + 4 * c + 4, nwy4 + 4 * c + 4, x, y, m1, k1);
        const bool second = m1 < m0;
        const float m = second ? m1 : m0;
        const int j = second ? 16 * c + 16 + __float2int_rn(k1) : 16 * c + __float2int_rn(k0);
        if (m < bm) { bm = m; bj = j; sbm = sqrtf(m); }
    }
#endif
    for (; c < nch; ++c) {
        if (far(c)) continue;
        float m, key;
        chunk_argmin<16>(nwx4 + 4 * c, nwy4 + 4 * c, x, y, m, key);
        if (m < bm) { bm = m; bj = 16 * c + __float2int_rn(key); sbm = sqrtf(m); }       // strict <: the earlier chunk wins ties
    }
    return bj;
}

__device__ __forceinline__ float4 window_ref(const TickSmem &sm, int j) {
    MPPI_DCHECK(j >= 0 && j < MPPI_MAX_WINDOW);
    const float2 yv = sm.wyv[j];
    return make_float4(-sm.wx[j], -sm.wy[j], yv.x, yv.y);
}

// sin and cos together, ~1.5 ulp for |x| < 1e4 (headings never leave that range): three-constant
// Cody-Waite reduction by pi/2 with the quadrant taken from the magic-number rounding (no F2I, no
// MUFU, no slow path), then the Cephes single-precision minimax polynomials on [-pi/4, pi/4].
// Replaces np.cos / np.sin in _state_transition (mppi_differential_drive.py:194-195).
__device__ __forceinline__ void sincos_cw(float x, float &s, float &c) {
    const float t = fmaf(x, 0.636619772f, 12582912.f);
    const int q = __float_as_int(t);
    const float k = t - 12582912.f;
    float r = fmaf(k, -1.5707963705062866f, x);          // pi/2 = hi + mid + lo (float32 pieces)
    r = fmaf(k, 4.371138828673793e-08f, r);
    r = fmaf(k, 1.7151245100058819e-15f, r);
    const float r2 = r * r;
    float sp = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = fmaf(sp, r2, -1.6666654611e-1f);
    sp = fmaf(sp * r2, r, r);
    float cp = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = fmaf(cp, r2, 4.166664568298827e-2f);
    cp = fmaf(cp, r2, -0.5f);
    cp = fmaf(cp, r2, 1.0f);
    const float ss = (q & 1) ? cp : sp, cc = (q & 1) ? sp : cp;
    s = __int_as_float(__float_as_int(ss) ^ ((q << 30) & 0x80000000));
    c = __int_as_float(__float_as_int(cc) ^ (((q + 1) << 30) & 0x80000000));
}

// exact (yaw + 2pi) mod 2pi with the sign of the divisor (race-car :151): the FMA remainder
// of a correctly chosen quotient is exactly representable, so this equals fmodf + fix-up.
__device__ __forceinline__ float wrap_2pi(float yaw) {
    const float b = 6.2831855f;
    const float y2 = yaw + b;
    const float q = floorf(y2 * 0.15915494f);
    float r = fmaf(-q, b, y2);
    if (r < 0.f) r += b;
    if (r >= b) r -= b;
    return r;
}

// A10: collision tests.  Returns true if the state collides with any obstacle.  The obstacles come from `sc`: the shared
// set in TickArgs (sc is `a`), or a robot's SceneRec in shared memory (scene instantiations).
// A per-robot obstacle set (SceneRec in shared memory): the same tests, walked one obstacle per trip -- its operands are
// shared-memory loads, and unrolled trips would hold several obstacles' worth of them in registers.
template <int MODEL, int COLL>
__device__ __forceinline__ bool collided_scene(const TickArgs &a, const SceneRec &sc, float x, float y, float cs, float sn) {
    bool hit = false;
    if constexpr (COLL == MPPI_COLLISION_CIRCLE) {
#pragma unroll 1
        for (int m = 0; m < sc.n_obs; ++m) {
            const float dx = x - sc.obs_x[m], dy = y - sc.obs_y[m];
            hit |= (dx * dx + dy * dy < sc.obs_r2[m]);
        }
    } else if constexpr (COLL == MPPI_COLLISION_FOOTPRINT) {
#pragma unroll 1
        for (int m = 0; m < sc.n_obs; ++m) {
            const float cx = x - sc.obs_x[m], cy = y - sc.obs_y[m];
            if (cx * cx + cy * cy >= sc.obs_far2[m]) continue;
            const float r2 = sc.obs_r2[m];
            const float ac = a.fp_hl * cs, as = a.fp_hl * sn, bc = a.fp_hw * cs, bs = a.fp_hw * sn;
            float px, py;
            px = cx - ac;      py = cy - as;      hit |= (px * px + py * py < r2);
            px = cx - ac - bs; py = cy - as + bc; hit |= (px * px + py * py < r2);
            px = cx - bs;      py = cy + bc;      hit |= (px * px + py * py < r2);
            px = cx + ac - bs; py = cy + as + bc; hit |= (px * px + py * py < r2);
            px = cx + ac;      py = cy + as;      hit |= (px * px + py * py < r2);
            px = cx + ac + bs; py = cy + as - bc; hit |= (px * px + py * py < r2);
            px = cx + bs;      py = cy - bc;      hit |= (px * px + py * py < r2);
            px = cx - ac + bs; py = cy - as - bc; hit |= (px * px + py * py < r2);
        }
    }
    return hit;
}

// A10: collision tests.  Returns true if the state collides with any obstacle.  The obstacles come from `sc`: the shared
// set in TickArgs (sc is `a`, constant-bank operands), or a robot's SceneRec in shared memory (scene instantiations).
template <int MODEL, int COLL, class SC>
__device__ __forceinline__ bool collided(const TickArgs &a, const SC &sc, float x, float y, float cs, float sn) {
    if constexpr (!std::is_same<SC, TickArgs>::value) return collided_scene<MODEL, COLL>(a, sc, x, y, cs, sn);
    bool hit = false;
    if constexpr (COLL == MPPI_COLLISION_NONE) {
        return false;
    } else if constexpr (COLL == MPPI_COLLISION_CIRCLE) {        // mppi_differential_drive_obs.py:301-313
        for (int m = 0; m < sc.n_obs; ++m) {
            const float dx = x - sc.obs_x[m], dy = y - sc.obs_y[m];
            hit |= (dx * dx + dy * dy < sc.obs_r2[m]);
        }
        return hit;
    } else {
    // footprint: 8 perimeter points of the (l*margin) x (w*margin) box rotated by the raw yaw
    // (mppi_race_car_obstacle.py:255-274)
    for (int m = 0; m < sc.n_obs; ++m) {
        const float ox = sc.obs_x[m], oy = sc.obs_y[m];
        const float cx = x - ox, cy = y - oy;
        if (cx * cx + cy * cy >= sc.obs_far2[m]) continue;      // conservative reject
        const float r2 = sc.obs_r2[m];
        const float ac = a.fp_hl * cs, as = a.fp_hl * sn, bc = a.fp_hw * cs, bs = a.fp_hw * sn;
        float px, py;
        px = cx - ac;      py = cy - as;      hit |= (px * px + py * py < r2);   // (-hl, 0)
        px = cx - ac - bs; py = cy - as + bc; hit |= (px * px + py * py < r2);   // (-hl, +hw)
        px = cx - bs;      py = cy + bc;      hit |= (px * px + py * py < r2);   // (0, +hw)
        px = cx + ac - bs; py = cy + as + bc; hit |= (px * px + py * py < r2);   // (+hl, +hw)
        px = cx + ac;      py = cy + as;      hit |= (px * px + py * py < r2);   // (+hl, 0)
        px = cx + ac + bs; py = cy + as - bc; hit |= (px * px + py * py < r2);   // (+hl, -hw)
        px = cx + bs;      py = cy - bc;      hit |= (px * px + py * py < r2);   // (0, -hw)
        px = cx - ac + bs; py = cy - as - bc; hit |= (px * px + py * py < r2);   // (-hl, -hw)
    }
    return hit;
    }
}

// A9: weighted squared error to a waypoint (mppi_differential_drive.py:222-249; race-car :147-171)
template <int MODEL>
__device__ __forceinline__ float tracking_cost(const float4 ref, const float z[4], float yaw_eff, const float w[4]) {
    const float dx = z[0] - ref.x, dy = z[1] - ref.y, dyaw = yaw_eff - ref.z;
    float c = w[0] * dx * dx + w[1] * dy * dy + w[2] * dyaw * dyaw;
    if (MODEL == MPPI_MODEL_BICYCLE) { const float dv = z[3] - ref.w; c += w[3] * dv * dv; }
    return c;
}

// The tick kernel's WIN template argument doubles as the cost-kind selector: 20 / 0 = path tracking with a static /
// dynamic waypoint window, negative = no reference path at all.
#define MPPI_WIN_GOAL (-1)
#define MPPI_WIN_TARGET (-2)

// Goal-point cost of test/mppi_differential_drive_obs.py:202-232: w0 * |xy - goal|^2 + w1 * wrap(atan2(dy, dx) - yaw)^2
// with (dx, dy) = xy - goal (the bearing FROM the goal, as the reference writes it) and wrap(a) =
// atan2(sin a, cos a) in (-pi, pi], evaluated as the FMA remainder a - 2pi*rint(a / 2pi) (only its square is used).
template <class SC>
__device__ __forceinline__ float goal_cost(const SC &sc, const float z[4], const float w[4]) {
    const float dx = z[0] - sc.goal[0], dy = z[1] - sc.goal[1];
    const float d2 = fmaf(dy, dy, dx * dx);
    const float diff = atan2f(dy, dx) - z[2];
    const float k = rintf(diff * 0.15915494309189535f);
    float r = fmaf(k, -6.2831854820251465f, diff);          // 2pi = hi + lo (float32 pieces)
    r = fmaf(k, 1.7484555314695172e-07f, r);
    return w[0] * d2 + w[1] * r * r;
}

// Running cost of test/test_mppi_diff_obs.py:44-66 for the state reached by horizon step t (time t*dt) under the
// clamped control (v0, v1): (z - target)^T Q (z - target) + v^T R v + W * sum_m exp(sd - d_m) [d_m < sd] with
// d_m the distance to obstacle m at pos_m + vel_m * t*dt (:14-20).  `full` = false: the quadratic pose error only.
template <class SC>
__device__ __forceinline__ float target_soft_cost(const TickArgs &a, const SC &sc, const float z[4], float v0, float v1, int t,
                                                  const float w[4], bool full) {
    const float ex = z[0] - sc.goal[0], ey = z[1] - sc.goal[1], eth = z[2] - sc.goal[2];
    float c = w[0] * ex * ex + w[1] * ey * ey + w[2] * eth * eth;
    if (full) {
        c += a.ctrl_w[0] * v0 * v0 + a.ctrl_w[1] * v1 * v1;
        const float tt = (float)t * a.dt;
        float soft = 0.f;
        for (int m = 0; m < sc.n_obs; ++m) {
            const float dx = z[0] - fmaf(sc.obs_vx[m], tt, sc.obs_x[m]), dy = z[1] - fmaf(sc.obs_vy[m], tt, sc.obs_y[m]);
            const float d = sqrtf(fmaf(dy, dy, dx * dx));
            if (d < a.soft_sd) soft += expf(a.soft_sd - d);
        }
        c = fmaf(a.soft_w, soft, c);
    }
    return c;
}

// A9 for every cost kind: the cost of state z reached by horizon step t with weights w.  For the path kinds the
// waypoint (ref, yaw_eff) found here is kept so the terminal cost of the same state can reuse it.
template <int MODEL, int WIN, class SC>
__device__ __forceinline__ float eval_state_cost(const TickArgs &a, const SC &sc, const TickSmem &sm, const float z[4], float v0,
                                                 float v1, int t, const float w[4], float4 &ref, float &yaw_eff) {
    if constexpr (WIN == MPPI_WIN_GOAL) {
        return goal_cost(sc, z, w);
    } else if constexpr (WIN == MPPI_WIN_TARGET) {
        return target_soft_cost(a, sc, z, v0, v1, t, w, true);
    } else {
        const int j = nearest_wp<WIN>(sm, z[0], z[1]);
        ref = window_ref(sm, j);
        yaw_eff = (MODEL == MPPI_MODEL_BICYCLE && a.yaw_wrap) ? wrap_2pi(z[2]) : z[2];
        return tracking_cost<MODEL>(ref, z, yaw_eff, w);
    }
}
// terminal cost of the SAME state the last stage cost was evaluated at (A9, :126)
template <int MODEL, int WIN, class SC>
__device__ __forceinline__ float eval_terminal_cost(const TickArgs &a, const SC &sc, const float z[4], const float4 ref, float yaw_eff) {
    if constexpr (WIN == MPPI_WIN_GOAL) return goal_cost(sc, z, a.tw);
    else if constexpr (WIN == MPPI_WIN_TARGET) return target_soft_cost(a, sc, z, 0.f, 0.f, 0, a.tw, false);
    else return tracking_cost<MODEL>(ref, z, yaw_eff, a.tw);
}

// A6 / A7: explicit-Euler dynamics; (cs, sn) = cos/sin of the CURRENT heading.
template <int MODEL>
__device__ __forceinline__ void dyn_step(const TickArgs &a, float z[4], float v0, float v1, float cs, float sn) {
    if (MODEL == MPPI_MODEL_BICYCLE) {          // mppi_race_car_obstacle.py:200-214, v = [steer, accel]
        const float vel = z[3];
        z[0] += vel * cs * a.dt;
        z[1] += vel * sn * a.dt;
        z[2] += vel * a.dt_over_L * tanf(v0);
        z[3] += v1 * a.dt;
    } else {                                    // mppi_differential_drive.py:182-198
        z[0] += v0 * cs * a.dt;
        z[1] += v0 * sn * a.dt;
        z[2] += v1 * a.dt;
    }
}

// The same step with tan(steer) supplied by the caller (time-parallel rollout: the tangent depends on the noise only, so it is
// taken off the recurrence's dependency chain, where its range test is the one branch that keeps the steps from overlapping).
template <int MODEL>
__device__ __forceinline__ void dyn_step_tan(const TickArgs &a, float z[4], float v0, float v1, float cs, float sn, float tan_v0) {
    if (MODEL == MPPI_MODEL_BICYCLE) {
        const float vel = z[3];
        z[0] += vel * cs * a.dt;
        z[1] += vel * sn * a.dt;
        z[2] += vel * a.dt_over_L * tan_v0;
        z[3] += v1 * a.dt;
    } else {
        dyn_step<MODEL>(a, z, v0, v1, cs, sn);
    }
}

__device__ __forceinline__ float clampf(float v, float lim) { return fminf(fmaxf(v, -lim), lim); }

// The rollouts of SPT samples of one thread (frozen window), advanced in LOCKSTEP: every stage is written as a loop over the
// thread's samples inside one basic block, so the instruction scheduler interleaves SPT independent dependency chains
// (the horizon recurrence makes a single chain latency-bound: ~220 cycles of dependent latency per step).  Sample s of
// the thread is chunk slot `slot0 + s * MPPI_BLOCK`.  Returns per sample the smooth cost and the number of collided
// evaluations separately so 1e10 * n never swallows the tracking cost (SURVEY.md section 7).
//
// The loop is also software-pipelined by hand: the noise of the NEXT timestep pair (Philox + Box-Muller:
// integer/ALU + MUFU work) is generated in the same straight-line block as the two dynamics/cost
// steps of the CURRENT pair (FMA-pipe work), so the ALU, MUFU and FMA pipes are busy at the same time.
template <int MODEL, int COLL, bool SUM, bool INJ, int WIN, int SPT, class SC>
__device__ __forceinline__ void rollout_samples(const TickArgs &a, const SC &sc, const TickSmem &sm, const uint32_t (&kg)[SPT], const int (&klocal)[SPT],
                                                uint32_t robot, const bool (&exploit)[SPT], float2 *stash, float (&smooth)[SPT], int (&ncoll)[SPT],
                                                uint32_t tick_add = 0u) {
    const int T = a.T;
    float z[SPT][4], cs[SPT], sn[SPT], acc[SPT], v0[SPT], v1[SPT], yaw_eff[SPT];
    int nc[SPT];
    float4 ref[SPT];
    bool hit[SPT];
    const float2 *eps_k[SPT];
#pragma unroll
    for (int s = 0; s < SPT; ++s) {
        z[s][0] = sm.x0[0]; z[s][1] = sm.x0[1]; z[s][2] = sm.x0[2]; z[s][3] = sm.x0[3];
        sincos_cw(z[s][2], sn[s], cs[s]);
        acc[s] = 0.f; nc[s] = 0; v0[s] = v1[s] = 0.f; yaw_eff[s] = 0.f; hit[s] = false;
        ref[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        eps_k[s] = INJ ? reinterpret_cast<const float2 *>(a.eps) + (size_t)klocal[s] * T : nullptr;
    }

    auto fetch = [&](int s, int tp, float e[4]) {
        if (INJ) {
            e[0] = e[1] = e[2] = e[3] = 0.f;
            if (tp < T) { const float2 ea = eps_k[s][tp]; e[0] = ea.x; e[1] = ea.y; }
            if (tp + 1 < T) { const float2 eb = eps_k[s][tp + 1]; e[2] = eb.x; e[3] = eb.y; }
        } else {
            philox_eps_pair(a, kg[s], (uint32_t)(tp >> 1), robot, e, tick_add);
        }
    };
    auto step = [&](int s, int t, float e0, float e1) {
        MPPI_DCHECK(t >= 0 && t < T);
        if (stash) stash[t * MPPI_CHUNK + s * MPPI_BLOCK] = make_float2(e0, e1);
        const float2 u = sm.U[t];
        v0[s] = clampf(exploit[s] ? __fadd_rn(u.x, e0) : e0, a.umax0);                   // A4, A5
        v1[s] = clampf(exploit[s] ? __fadd_rn(u.y, e1) : e1, a.umax1);
        dyn_step<MODEL>(a, z[s], v0[s], v1[s], cs[s], sn[s]);
        sincos_cw(z[s][2], sn[s], cs[s]);
        if (SUM) {
            const float c = eval_state_cost<MODEL, WIN>(a, sc, sm, z[s], v0[s], v1[s], t, a.sw, ref[s], yaw_eff[s]);
            const float2 q = sm.Q[t];                                                // zero when gamma == 0
            acc[s] += c + (q.x * v0[s] + q.y * v1[s]);
            hit[s] = collided<MODEL, COLL>(a, sc, z[s][0], z[s][1], cs[s], sn[s]);
            nc[s] += hit[s] ? 1 : 0;
        }
    };

    float e[SPT][4];
#pragma unroll
    for (int s = 0; s < SPT; ++s) fetch(s, 0, e[s]);
    // pairs of timesteps whose successor still needs noise run with the fetch of the NEXT pair interleaved; the last
    // pair (or the odd last step) runs alone, so no Philox call is wasted
    // (path-free cost kinds, WIN < 0, keep the surplus fetch: their step carries atan2f / expf bodies and a second inlined
    // copy of it costs more in instruction fetch than the one Philox call saves -- goal-point K = 1M: 0.472 vs 0.490 ms)
    const int n_fetch_pairs = WIN >= 0 ? (T - 1) >> 1 : T >> 1;   // pairs tp = 0, 2, ... for which a step tp + 2 exists (or all pairs)
    int tp = 0;
    for (int i = 0; i < n_fetch_pairs; ++i, tp += 2) {
        float en[SPT][4];
#pragma unroll
        for (int s = 0; s < SPT; ++s) fetch(s, tp + 2, en[s]);      // independent of the two steps below
#pragma unroll
        for (int s = 0; s < SPT; ++s) step(s, tp, e[s][0], e[s][1]);
#pragma unroll
        for (int s = 0; s < SPT; ++s) step(s, tp + 1, e[s][2], e[s][3]);
#pragma unroll
        for (int s = 0; s < SPT; ++s) { e[s][0] = en[s][0]; e[s][1] = en[s][1]; e[s][2] = en[s][2]; e[s][3] = en[s][3]; }
    }
#pragma unroll
    for (int s = 0; s < SPT; ++s) {
        if (WIN >= 0) {
            step(s, tp, e[s][0], e[s][1]);                  // tp = T - 2 (even T) or T - 1 (odd T)
            if (!(T & 1)) step(s, tp + 1, e[s][2], e[s][3]);
        } else if (T & 1) {
            step(s, T - 1, e[s][0], e[s][1]);
        }
        if (SUM) {                          // terminal cost: same state, same waypoint as the last stage cost (A9)
            acc[s] += eval_terminal_cost<MODEL, WIN>(a, sc, z[s], ref[s], yaw_eff[s]);
            nc[s] += hit[s] ? 1 : 0;
        } else {                            // Q1: only the last stage cost survives, plus terminal
            const float2 q = sm.Q[T - 1];
            acc[s] = eval_state_cost<MODEL, WIN>(a, sc, sm, z[s], v0[s], v1[s], T - 1, a.sw, ref[s], yaw_eff[s]) + (q.x * v0[s] + q.y * v1[s]);
            acc[s] += eval_terminal_cost<MODEL, WIN>(a, sc, z[s], ref[s], yaw_eff[s]);
            nc[s] = collided<MODEL, COLL>(a, sc, z[s][0], z[s][1], cs[s], sn[s]) ? 2 : 0;
        }
        smooth[s] = acc[s];
        ncoll[s] = nc[s];
    }
}

// ------------------------------------------------------------------------------------------
// Time-parallel rollout for SMALL sample counts (tick kernel instantiations with STASH == 2).
// With fewer samples than the GPU has lanes, one thread walking one sample through the horizon is bound by the
// latency of its own instruction chain (race-car K = 16 384, H = 50: 1.4 us per step whatever K is).  But only the
// dynamics are a recurrence over t: the noise of (k, t) is a pure function of its Philox counter, and the stage cost
// of step t (waypoint search, tracking terms, collision test -- 2/3 of a step's instructions) only READS state t.
// So a CTA that owns n <= MPPI_TPAR_SLOTS samples runs the horizon in four block-wide phases:
//   N  all threads: Philox + Box-Muller of every (sample, timestep pair) into the noise stash (rows of MPPI_TPAR_SLOTS
//      columns here, which K2's column sums read with that stride);
//   D  one thread per sample: clamp + Euler recurrence only, state of every step into `zbuf[t][slot]`;
//   C  all threads: stage (and terminal) cost + collision test of every (sample, t), written over the state it read --
//      started together with D and following it step by step (progress flags), so the six warps D does not need are not idle;
//   S  one thread per sample: the T costs added in horizon order -- the same sum, in the same order, as the serial loop.
// Two such CTAs are resident per SM (T * 64 * 24 B of shared memory each), so one CTA's serial phase D overlaps the other's
// wide phases.  Same device functions as rollout_samples, so a sample's result does not depend on which rollout ran it.
// All MPPI_BLOCK threads must call; threads tid < n return their sample, the others (inf, INT_MAX).  Shared scene only: the
// per-robot-scene instantiations have no time-parallel variant.
// ------------------------------------------------------------------------------------------
#define MPPI_TPAR_SLOTS 64
#ifndef MPPI_TPAR_PROBE
#define MPPI_TPAR_PROBE 0          // 1: block 0 / 77 print the cycles of each phase at tick 25 (measurement builds only)
#endif
#if MPPI_TPAR_PROBE
#include <cstdio>
#endif
struct TparSmem {
    int prog[MPPI_TPAR_SLOTS / 32];    // horizon steps whose state warp w has published
    int next;                          // next unclaimed cost item
};
template <int MODEL, int COLL, int WIN>
__device__ __forceinline__ void rollout_tpar(const TickArgs &a, const TickSmem &sm, TparSmem &ts, const int k_begin, const int n, const uint32_t robot,
                                             float2 *stash, float4 *zbuf, float &smooth, int &ncoll, const uint32_t tick_add) {
    const int T = a.T, tid = threadIdx.x;
    // item -> (row, slot) without an integer division per item (48 instructions of a ~500-instruction cost item): i / n as the high
    // word of i * ceil(2^32 / n), exact while i * n < 2^32 (here i < 2^13, n <= 64)
    const uint32_t inv_n = n > 1 ? (uint32_t)((0x100000000ull + (uint32_t)n - 1u) / (uint32_t)n) : 0u;
    auto div_n = [&](int i) { return n > 1 ? (int)__umulhi((uint32_t)i, inv_n) : i; };
    if (tid < MPPI_TPAR_SLOTS / 32) ts.prog[tid] = 0;      // (the previous chunk's consumers are past its last barrier)
    if (tid == 0) ts.next = 0;
    const uint32_t kg0 = (uint32_t)(a.k_offset + k_begin);
    MPPI_DCHECK(n >= 1 && n <= MPPI_TPAR_SLOTS && MPPI_TPAR_SLOTS <= MPPI_BLOCK);
#if MPPI_TPAR_PROBE
    long long pc[5];
#define MPPI_TPAR_STAMP(i) pc[i] = clock64()
#else
#define MPPI_TPAR_STAMP(i)
#endif
    MPPI_TPAR_STAMP(0);
    // ---- N: noise.  Item i = (pair p, slot): consecutive lanes take consecutive slots of one pair.
    {
        const int npairs = (T + 1) >> 1, items = n * npairs;
        for (int i = tid; i < items; i += MPPI_BLOCK) {
            const int p = div_n(i), slot = i - p * n;
            MPPI_DCHECK(p == i / n && 2 * p < T && slot >= 0 && slot < n);
            float e[4];
            philox_eps_pair(a, kg0 + (uint32_t)slot, (uint32_t)p, robot, e, tick_add);
            stash[(2 * p) * MPPI_TPAR_SLOTS + slot] = make_float2(e[0], e[1]);
            if (2 * p + 1 < T) stash[(2 * p + 1) * MPPI_TPAR_SLOTS + slot] = make_float2(e[2], e[3]);
            if (MODEL == MPPI_MODEL_BICYCLE) {          // tan(steer) of both steps, parked in the state slot phase D will overwrite
                const bool exploit = (int)(kg0 + (uint32_t)slot) < a.n_exploit;
                const float ua = sm.U[2 * p].x, ub = (2 * p + 1 < T) ? sm.U[2 * p + 1].x : 0.f;
                zbuf[(2 * p) * MPPI_TPAR_SLOTS + slot].x = tanf(clampf(exploit ? __fadd_rn(ua, e[0]) : e[0], a.umax0));
                if (2 * p + 1 < T) zbuf[(2 * p + 1) * MPPI_TPAR_SLOTS + slot].x = tanf(clampf(exploit ? __fadd_rn(ub, e[2]) : e[2], a.umax0));
            }
        }
        // chunk slots without a sample carry weight 0 in the column sums: their noise must be finite
        const int idle = MPPI_TPAR_SLOTS - n;
        for (int i = tid; i < idle * T; i += MPPI_BLOCK) {
            const int t = i / idle, slot = n + (i - t * idle);
            stash[t * MPPI_TPAR_SLOTS + slot] = make_float2(0.f, 0.f);
            zbuf[t * MPPI_TPAR_SLOTS + slot].x = 0.f;
        }
    }
    __syncthreads();
    MPPI_TPAR_STAMP(1);
    // ---- D and C overlapped.  The warps that own the samples (n_dw of them) run the recurrence (A4-A7) and publish, every four
    // steps, how far they are (`ts.prog[warp]`, release / acquire at CTA scope); every other warp -- and the D warps once they are
    // through -- takes batches of 32 cost items (t-major, so the batches follow the recurrence) from a shared counter and waits
    // for the state it needs.  The D warps never wait, so the consumers cannot deadlock.
    const int lane = tid & 31, warp = tid >> 5, n_dw = (n + 31) >> 5;
    if (warp < n_dw) {
        // (lanes past n in the last D warp roll out an idle slot -- zero noise, finite -- so the whole warp stays converged)
        const bool exploit = (int)(kg0 + (uint32_t)tid) < a.n_exploit;
        float z[4] = {sm.x0[0], sm.x0[1], sm.x0[2], sm.x0[3]}, cs, sn;
        sincos_cw(z[2], sn, cs);
        for (int t0 = 0; t0 < T; t0 += 4) {
            // four steps at a time: only the heading / speed updates are a true recurrence; the sin/cos of a step and the position
            // update that needs it overlap with the following steps' heading updates
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = t0 + j;
                if (t < T) {
                    const float2 e = stash[t * MPPI_TPAR_SLOTS + tid], u = sm.U[t];
                    const float v0 = clampf(exploit ? __fadd_rn(u.x, e.x) : e.x, a.umax0);
                    const float v1 = clampf(exploit ? __fadd_rn(u.y, e.y) : e.y, a.umax1);
                    const float tan_v0 = (MODEL == MPPI_MODEL_BICYCLE) ? zbuf[t * MPPI_TPAR_SLOTS + tid].x : 0.f;
                    dyn_step_tan<MODEL>(a, z, v0, v1, cs, sn, tan_v0);
                    sincos_cw(z[2], sn, cs);
                    zbuf[t * MPPI_TPAR_SLOTS + tid] = make_float4(z[0], z[1], z[2], z[3]);
                }
            }
            __syncwarp();
            if (lane == 0) {
                const int done = min(t0 + 4, T);
                asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(&ts.prog[warp])), "r"(done) : "memory");
            }
        }
    }
    MPPI_TPAR_STAMP(2);
    // costs of every (t, slot); the record (stage cost + control term, terminal cost, collided) replaces the state it was computed from
    {
        const int items = n * T;
        for (;;) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&ts.next, 32);
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base >= items) break;
            const int i = base + lane;
            if (i < items) {
                const int t = div_n(i), slot = i - t * n;
                MPPI_DCHECK(t == i / n && t < T && slot >= 0 && slot < n && (slot >> 5) < n_dw);
                {
                    const uint32_t flag = (uint32_t)__cvta_generic_to_shared(&ts.prog[slot >> 5]);
                    int done;
                    for (;;) {
                        asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(done) : "r"(flag) : "memory");
                        if (done > t) break;
                        __nanosleep(40);            // do not poll the recurrence warps out of their issue slots
                    }
                }
                const float4 z4 = zbuf[t * MPPI_TPAR_SLOTS + slot];
                const float z[4] = {z4.x, z4.y, z4.z, z4.w};
                const bool exploit = (int)(kg0 + (uint32_t)slot) < a.n_exploit;
                const float2 e = stash[t * MPPI_TPAR_SLOTS + slot], u = sm.U[t];
                const float v0 = clampf(exploit ? __fadd_rn(u.x, e.x) : e.x, a.umax0);
                const float v1 = clampf(exploit ? __fadd_rn(u.y, e.y) : e.y, a.umax1);
                float4 ref = make_float4(0.f, 0.f, 0.f, 0.f);
                float yaw_eff = 0.f;
                const float c = eval_state_cost<MODEL, WIN>(a, a, sm, z, v0, v1, t, a.sw, ref, yaw_eff);
                const float2 q = sm.Q[t];
                const float cc = c + (q.x * v0 + q.y * v1);
                bool hit = false;
                if constexpr (COLL != MPPI_COLLISION_NONE) {
                    float cs, sn;
                    sincos_cw(z[2], sn, cs);
                    hit = collided<MODEL, COLL>(a, a, z[0], z[1], cs, sn);
                }
                const float term = (t == T - 1) ? eval_terminal_cost<MODEL, WIN>(a, a, z, ref, yaw_eff) : 0.f;
                zbuf[t * MPPI_TPAR_SLOTS + slot] = make_float4(cc, term, hit ? 1.f : 0.f, 0.f);
            }
        }
    }
    __syncthreads();
    MPPI_TPAR_STAMP(3);
    // ---- S: horizon-order sum (A11), terminal cost and the terminal collision test of the same state (A9, A10)
    smooth = CUDART_INF_F; ncoll = INT_MAX;
    if (tid < n) {
        float acc = 0.f;
        int nc = 0;
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int t = 0; t < T; ++t) {
            r = zbuf[t * MPPI_TPAR_SLOTS + tid];
            acc += r.x;
            nc += (r.z != 0.f) ? 1 : 0;
        }
        acc += r.y;
        nc += (r.z != 0.f) ? 1 : 0;
        smooth = acc; ncoll = nc;
    }
#if MPPI_TPAR_PROBE
    MPPI_TPAR_STAMP(4);
    if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == 77) && a.tick == 25u)
        printf("tpar block %d n %d: N %lld D %lld C %lld S %lld cycles\n", (int)blockIdx.x, n, pc[1] - pc[0], pc[2] - pc[1], pc[3] - pc[2], pc[4] - pc[3]);
#endif
}
