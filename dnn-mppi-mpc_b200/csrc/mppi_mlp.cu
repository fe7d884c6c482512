// K3: learned-dynamics rollout for BASELINE config 3 -- unicycle + dnn/simple_mlp.py residual,
//     x+ = x + dt * ([v cos(th), v sin(th), w] + MLP(x))            (SURVEY.md 3.4)
// with MLP = Linear(3,512) -> tanh(Linear(512,512)) -> tanh(Linear(512,512)) -> Linear(512,3)
// (dnn/simple_mlp.py:10-23).
//
// sm_100a mapping (one persistent CTA per SM, clusters of two, each CTA owning 128-sample tiles for the whole horizon):
//   * the input layer has NO activation (simple_mlp.py:19), so Linear(3,512) and the first hidden
//     Linear(512,512) are folded on the host into one 3->512 map (W01 = W1 W0, b01 = W1 b0 + b1).  The compute warps evaluate it in
//     FP32 on the CUDA cores (three-input kernels) or read it back from a split-fp16 tcgen05 MMA (five-input ping-pong kernels),
//     apply tanh (MUFU), round ONCE to the half-precision operand type and store the A operand straight into
//     TENSOR MEMORY (tcgen05.st, 256 columns): the activations never touch shared memory, which leaves it to the weight stream;
//   * the remaining 512x512 layer is the GEMM: D[128x512] = A[128x512] (TMEM) x W2^T, issued by ONE thread as tcgen05.mma kind::f16
//     with the A operand in TMEM (N=128, K=16), W2 streamed from L2 by TMA (cp.async.bulk.tensor, 128B swizzle) through an mbarrier
//     ring that fills the 192 KB of shared memory.  The two CTAs of a cluster walk the weight stream in lockstep; in the ping-pong
//     kernels they are ONE MMA unit (cta_group::2, M = 256: rank 0 issues for both, each CTA holds half of every W2 box), otherwise
//     each CTA issues every other box with .multicast::cluster; the accumulator is produced in four 128-column quarters through two
//     TMEM buffers (2 x 128 columns), so the epilogue of one quarter overlaps the MMAs of the next;
//   * the epilogue warps read the accumulator with tcgen05.ld (32x32b.x32), add b2, apply tanh and
//     contract with the 512x3 output layer in FP32 registers -- the output layer never touches memory;
//   * the unicycle step, nearest-waypoint search and cost run in the same epilogue threads with the
//     state in registers across the horizon.
// Learned residuals with FIVE inputs (state + control, the shape of the reference's trained saved_models/mlp_diff*.pth:
// simulation/bullet_differential_drive_dnn.py:37-60, train/train_diff_mlp.py:13-36) run through the same kernel
// (template NIN = 5): the folded first layer takes (x, y, yaw, v, w), so the owner thread generates the control of step
// t+1 while the GEMM of step t runs and publishes it with the state.  StandardScaler pre/post-processing
// (test/test_diff_dyna_eval.py:54-56) is folded into the first / last layer on the host.
// Residuals with THREE tanh layers (train/train_diff_mlp.py:13-36, saved_models/mlp_diff_300x100_3l*.pth) need a second
// 512x512 GEMM whose A operand is the first GEMM's epilogue.  Tensor memory has no room for it (A 256 + two
// accumulator buffers 256 = all 512 columns), so the template NG = 2 keeps that second operand in SHARED memory: the
// epilogue of GEMM 1 (+bias, tanh, pack) writes the 128 x 512 tile in the K-major 128B-swizzled layout the UMMA
// descriptor expects (eight 16 KB K-chunks, 128 KB), fences it to the async proxy and GEMM 2 runs in the SS form; the
// weight ring shrinks to four 16 KB stages and carries both layers' boxes back to back.
// Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (both run converged, one elected lane issues), warps 2..17 = 16 compute
// warps (four per TMEM lane quarter; group g = (warp-2)/4 takes 32 columns of every 128-column part of the
// activations and of every accumulator quarter, so MMA start and epilogue tail are both short).
// Variants that were built, measured and rejected (mma.sync layer 1, register-tiled 16x256b layer 1 / epilogue, early layer 1,
// K-interleaved last quarters, output-layer records through the constant bank) are described in DESIGN.md 3.4 with the commits that hold them.
//
// THIS FILE IS COMPILED TWICE.  mppi_mlp_traj.cu includes it with MPPI_MLP_TRAJ_UNIT defined to instantiate the replay (TRAJ)
// kernels apart from the tick's (see mlp_traj_kernels below).  In that unit only the TRAJ table is emitted: everything that
// must exist once -- host functions, the tick's kernel table, any __device__ / __constant__ variable or other kernel -- belongs
// in the `#else` branch of the `#ifdef MPPI_MLP_TRAJ_UNIT` at the end, or behind a guard of its own.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "mppi_device.cuh"
#include "mppi_mlp.h"

namespace {

// Operand type of the hidden GEMM(s): fp16.  The A operand is a tanh output in [-1, 1] and trained weights are O(1), so half
// precision's 11-bit significand applies with no range problem -- 8x smaller rounding error than bf16 at the same tensor-core
// rate (weights beyond +-65504 are refused on the host).
typedef __half mlp_op_t;

// -DMPPI_MLP_PROBE=32 (never shipped, profiles/; 32 is its only bit): per-wait stall accounting (clock64 around every barrier wait of
// the MMA issuer and of compute warp 0, printed by CTA 0)
#ifndef MPPI_MLP_PROBE
#define MPPI_MLP_PROBE 0
#endif
#if MPPI_MLP_PROBE & 32
#define MLP_PROBE_DECL() long long pr_c = 0; const long long pr_begin = clock64(); unsigned long long *pr_t = reinterpret_cast<unsigned long long *>(sm.cb) + (warp == 1 ? 0 : 16);   /* static window: cb is unused */ (void)pr_c; \
    if ((threadIdx.x & 31) == 0 && (threadIdx.x >> 5) <= 2) for (int i_ = 0; i_ < 16; ++i_) pr_t[i_] = 0
#define MLP_TIC() pr_c = clock64()
#define MLP_TOC(i) do { const long long n_ = clock64(); if ((threadIdx.x & 31) == 0 && (threadIdx.x >> 5) <= 2) pr_t[(i)] += (unsigned long long)(n_ - pr_c); pr_c = n_; } while (0)
#define MLP_PROBE_PRINT(what, steps) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) printf("%s (cycles per tile-step, %d tile-steps, total %lld): %lld %lld %lld %lld | %lld %lld %lld %lld | %lld %lld %lld %lld | %lld %lld %lld %lld\n", what, (int)(steps), (clock64() - pr_begin) / max((int)(steps), 1), \
    (long long)pr_t[0] / max((int)(steps), 1), (long long)pr_t[1] / max((int)(steps), 1), (long long)pr_t[2] / max((int)(steps), 1), (long long)pr_t[3] / max((int)(steps), 1), (long long)pr_t[4] / max((int)(steps), 1), (long long)pr_t[5] / max((int)(steps), 1), (long long)pr_t[6] / max((int)(steps), 1), (long long)pr_t[7] / max((int)(steps), 1), \
    (long long)pr_t[8] / max((int)(steps), 1), (long long)pr_t[9] / max((int)(steps), 1), (long long)pr_t[10] / max((int)(steps), 1), (long long)pr_t[11] / max((int)(steps), 1), (long long)pr_t[12] / max((int)(steps), 1), (long long)pr_t[13] / max((int)(steps), 1), (long long)pr_t[14] / max((int)(steps), 1), (long long)pr_t[15] / max((int)(steps), 1)); } while (0)
#else
#define MLP_PROBE_DECL()
#define MLP_TIC()
#define MLP_TOC(i)
#define MLP_PROBE_PRINT(what, steps)
#endif

constexpr int HID = 512;
constexpr int TILE_M = 128;
constexpr int KCH = 64;                   // K elements per 128-byte swizzle span (fp16)

constexpr int N_MMA = 128;                // N per tcgen05.mma = one accumulator quarter
constexpr int N_QUARTERS = HID / N_MMA;
// Five-input ping-pong kernels: layer 1 ON THE tcgen05 TENSOR CORE.  The folded first layer needs FP32 accuracy, so inputs and
// weights are split into fp16 pieces, v = hi + lo, x.w ~= x_hi w_hi + x_hi w_lo + x_lo w_hi (three K slots per input + two for the bias: K = 16 | 32).  Its A
// operand (128 sample rows x K) and B operand (512 hidden units x K) live in shared memory in the same K-major 128B-swizzled layout as
// the weight boxes (rows padded to 128 B), and each 128-column part is ONE (two for 5 inputs) M128 x N128 x K16 MMA in the SS form.
// The pre-activations of a part pass through accumulator buffer 0, which is idle between the drain of quarter 2 and the next GEMM's
// quarter 0: the issuer slips the part-p MMA in right behind the K-part-p MMAs of the running GEMM's quarter 3 (the tensor pipe executes
// in order, so the part's commit also proves that quarter 3 is done with A part p), the compute warps read it back (tcgen05.ld), apply
// tanh, round once to fp16 and store it into A part p.  That replaces a broadcast LDS.128 + 3 (5) FMAs per (row, column) -- the work the
// compute warps' chain is made of (profiles/r2_mlp_stall_accounting.txt) -- by one tcgen05.ld of 32 columns per thread and part.
constexpr int KCH_PER_STAGE = 4;          // K chunks (TMA boxes) per ring stage: one barrier wait + one commit per 16 MMAs,
                                          // otherwise the single issuing thread (try_wait ~90 cycles) paces the tensor core
constexpr int B_STAGES = 3;
constexpr int B_BOX_BYTES = N_MMA * KCH * 2;       // 16 KB per TMA box
constexpr int B_TILE_BYTES = KCH_PER_STAGE * B_BOX_BYTES;   // 64 KB per stage
constexpr int RING_BYTES = 12 * B_BOX_BYTES;        // the 1024-aligned operand region at the start of dynamic shared memory (192 KB)
constexpr int A2_BYTES = TILE_M * HID * 2;          // NG = 2: second GEMM's A operand in shared memory (128 KB)
constexpr int B2_STAGES = (RING_BYTES - A2_BYTES) / B_BOX_BYTES;   // NG = 2: one-box stages in what is left (4)
static_assert(B2_STAGES >= 2, "NG = 2 ring");
static_assert(B_STAGES * B_TILE_BYTES <= RING_BYTES && (HID / KCH) % KCH_PER_STAGE == 0 && KCH_PER_STAGE % 2 == 0, "NG = 1 ring");
// The other ping-pong kernels: the hidden GEMM as PAIR MMAs, tcgen05.mma.cta_group::2 with M = 256 -- the two CTAs of a cluster
// (which already walk the weight stream in lockstep) become one MMA unit: rank 0 issues for both, each CTA keeps its own 128 rows of A and
// D in its tensor memory and only HALF of every W2 box (64 of the 128 rows) in its shared memory.  Per SM that halves the TMA writes and the
// B-operand reads (2 x 256 KB instead of 2 x 512 KB per tile-step), which share the shared-memory bandwidth with the compute warps'
// broadcast LDS.128 (profiles/r2_mlp_stall_accounting.txt).  The ring keeps its 192 KB: six 32 KB stages instead of three 64 KB ones.
constexpr int CG2_BOX_BYTES = B_BOX_BYTES / 2;                    // 64 W2 rows x 64 K halves
constexpr int RING_SLOTS = 12;                                    // barrier pairs: enough for every ring geometry (asserted in the kernel)
constexpr int L1_KS_MAX = 32;                       // tcgen05 layer 1: K slots (halves) per row, 16 (3 inputs) or 32 (5 inputs)
// tcgen05 layer 1 operands: K-major, SWIZZLE_32B -- rows of 16 halves (one K = 16 MMA step), 8-row atoms of 256 B, 16-byte chunk c of row
// r stored at c ^ ((r / 4) % 2).  Five inputs take two K steps: two such tiles ("K blocks") per operand.
constexpr int B1TC_KB_BYTES = HID * 32, A1TC_KB_BYTES = TILE_M * 32;     // one K block of B (16 KB: 4 parts of 4 KB) / of A (4 KB)
constexpr int B1TC_BYTES = 2 * B1TC_KB_BYTES;       // B operand, 512 hidden units (32 KB)
constexpr int A1TC_BYTES = 2 * A1TC_KB_BYTES;       // A operand, 128 sample rows (8 KB)
// which ping-pong kernels use what (shared by the kernel and the launcher): the tcgen05 layer 1 for the five-input kernels (where it
// wins: their CUDA-core layer 1 costs two LDS + five FMAs per column); pair MMAs for the others (the tcgen05 layer 1 issues
// cta_group::1, and one kernel may use only one group size)
__host__ __device__ constexpr bool mlp_use_l1tc(int nin, bool pp, int ng) { return pp && ng == 1 && nin == 5; }
__host__ __device__ constexpr bool mlp_use_cg2(int nin, bool pp, int ng) { return pp && ng == 1 && !mlp_use_l1tc(nin, pp, ng); }
constexpr int TMEM_A_COL = 0;             // A operand: 512 fp16 per row = 256 packed 32-bit columns
constexpr int TMEM_D_COL = 256;           // two accumulator buffers of 128 FP32 columns
constexpr int N_GROUPS = 4;                // compute-warp groups: group g owns accumulator quarter g (128 columns)
constexpr int N_COMPUTE = 128 * N_GROUPS;  // 16 compute warps: 4 per TMEM lane quarter
constexpr int MLP_THREADS = 64 + N_COMPUTE;
constexpr int N_ARRIVE = N_COMPUTE / 32;   // arrivals per compute-warp hand-off (see compute_arrive)


struct MlpSmem {                          // after the 1024-aligned A / B regions
    float4 w01[HID];                      // (W01[j][0], W01[j][1], W01[j][2], b01[j])   (unused when layer 1 runs on the tensor core)
    __align__(16) float2 w01u[HID];       // NIN = 5: (W01[j][3], W01[j][4]) -- the control columns
    union {
        float xw[TILE_M];                 // NIN = 5: second control component of each row (the first rides in xs.w)
        struct { unsigned long long a1_ready, d1_full, d1_empty; };   // tcgen05 layer 1 (never together with xw): input rows
    };                                                                // written / part in buffer 0 / part read back
    float4 w3[HID];                       // (b2[j], W3[0][j], W3[1][j], W3[2][j])
    float4 xs[TILE_M];                    // current state of each row for the partner thread
    float res[N_GROUPS - 1][3][TILE_M];   // partners' partial output-layer sums (SoA: 4.5 KB instead of 6 KB as float4)
    unsigned long long b_full[RING_SLOTS], b_empty[RING_SLOTS], a_ready[N_QUARTERS], d_full[2], d_empty[2];   // ring barriers: every geometry
    unsigned long long a_free[N_QUARTERS];   // ping-pong mode: the last accumulator quarter has consumed this K part of A
    unsigned long long key[8];
    unsigned long long a2_ready[N_QUARTERS];   // NG = 2: second-operand parts
    uint32_t tmem_base;
    float b3[3];
};

constexpr size_t MLP_DYN_SMEM = RING_BYTES + sizeof(TickSmem) + sizeof(MlpSmem);
static_assert(MLP_DYN_SMEM + 1024 <= 232448, "K3 shared memory exceeds the 227 KB per-CTA limit of sm_100a");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra.uni WAIT_DONE;\n\t"
        "bra.uni WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// Compute warps signal "my part of the operand is written" / "my part of the accumulator is read".  One arrival per WARP:
// every lane has waited for its tcgen05.st / tcgen05.ld and fenced, __syncwarp orders that before lane 0's releasing arrive -- 16
// shared-memory barrier operations per hand-off instead of 512.
__device__ __forceinline__ void mbar_arrive_rank0(unsigned long long *bar);
template <bool TO_RANK0 = false>                               // pair MMAs: both CTAs report to rank 0's barrier
__device__ __forceinline__ void compute_arrive(unsigned long long *bar) {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) { if constexpr (TO_RANK0) mbar_arrive_rank0(bar); else mbar_arrive(bar); }
}

// non-blocking: has the phase with this parity completed?  (warp-uniform: lane 0's answer)
__device__ __forceinline__ bool mbar_test_warp(unsigned long long *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return __shfl_sync(0xffffffffu, ok, 0) != 0;
}

// warp-level wait: one lane polls the barrier (every try_wait is a shared-memory operation -- 16 compute warps polling
// with all 32 lanes loaded the same data pipe the weight LDS, the UMMA B reads and the TMA writes go through), the rest
// of the warp joins at __syncwarp, which also orders the polling lane's acquire before the other lanes' later accesses
__device__ __forceinline__ void mbar_wait_warp(unsigned long long *bar, uint32_t parity) {
    if ((threadIdx.x & 31) == 0) mbar_wait(bar, parity);
    __syncwarp();
}

__device__ __forceinline__ void tma_load_2d_mc(void *dst, const CUtensorMap *map, unsigned long long *bar, int c0, int c1, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// UMMA shared-memory descriptor: K-major, SWIZZLE_128B, 8-row x 128-byte atoms 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);              // start address
    d |= (uint64_t)0 << 16;                              // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)((1024 >> 4) & 0x3FFF) << 32;         // stride byte offset
    d |= (uint64_t)1 << 46;                              // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                              // SWIZZLE_128B
    return d;
}

// same for SWIZZLE_32B operands (tcgen05 layer 1): 8-row x 32-byte atoms 256 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((256 >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)6 << 61;                              // SWIZZLE_32B
    return d;
}

// kind::f16 instruction descriptor: F16 x F16 -> F32 (A and B format fields 0), K-major A and B, M=128, N=128
constexpr uint32_t UMMA_IDESC = (1u << 4) | ((uint32_t)(N_MMA >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);

// A operand in tensor memory (128 lanes x 8 packed f16x2 columns per K=16 step), B in shared memory
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(UMMA_IDESC), "r"(accumulate), "r"(0u) : "memory");
}
// both operands in shared memory (NG = 2, second GEMM)
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(UMMA_IDESC), "r"(accumulate), "r"(0u) : "memory");
}
// ---- pair MMAs (cta_group::2): rank 0 issues M = 256 MMAs over both CTAs' tensor memory and shared memory ----
constexpr uint32_t UMMA_IDESC_2SM = (1u << 4) | ((uint32_t)(N_MMA >> 3) << 17) | ((uint32_t)((2 * TILE_M) >> 4) << 24);
__device__ __forceinline__ void umma_f16_ts_2sm(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(UMMA_IDESC_2SM), "r"(accumulate), "r"(0u) : "memory");
}
// arrive on the barrier at this offset in every CTA of the mask once the pair MMAs issued so far retire
__device__ __forceinline__ void umma_commit_2sm_mc(unsigned long long *bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
// this CTA's half of a W2 box into its own ring; the bytes are counted on RANK 0's barrier (peer bit of the address cleared)
__device__ __forceinline__ void tma_load_2d_2sm(void *dst, const CUtensorMap *map, unsigned long long *bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1) : "memory");
}
// arrive on rank 0's copy of a barrier, from either CTA of the pair.  Default semantics (release at CTA scope), as CUTLASS's
// ClusterBarrier::arrive does for the same hand-off: what travels between the CTAs is tensor memory, ordered by tcgen05.wait +
// tcgen05.fence::before_thread_sync on this side and fence::after_thread_sync on the issuer's; a release at CLUSTER scope here
// measured ~700 cycles per arrival (profiles/r2_mlp_stall_accounting.txt)
__device__ __forceinline__ void mbar_arrive_rank0(unsigned long long *bar) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, 0;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned long long *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on the same barrier in every CTA of the cluster mask once the MMAs issued so far retire
__device__ __forceinline__ void umma_commit_mc(unsigned long long *bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// two FP32 values -> packed half-precision operand pair (lo in the low half)
__device__ __forceinline__ uint32_t pack_op2(float lo, float hi) {
    uint32_t p;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(p) : "f"(hi), "f"(lo));
    return p;
}
// tanh of two FP32 pre-activations -> packed operand pair: FP32 MUFU.TANH on the unrounded pre-activation, ONE rounding at
// the end
__device__ __forceinline__ uint32_t tanh_op2(float lo, float hi) {
    return pack_op2(tanh_approx(lo), tanh_approx(hi));
}
// v = hi + lo in half precision, packed (hi in the low half)
__device__ __forceinline__ void split_half(float v, unsigned short &hi, unsigned short &lo) {
    const __half h = __float2half_rn(v);
    const __half l = __float2half_rn(v - __half2float(h));
    hi = __half_as_ushort(h); lo = __half_as_ushort(l);
}
// tcgen05 layer 1: the split input row of one sample -- slots 3c..3c+2 = (hi, hi, lo) of input c, then (1, 1) for the bias, zeros behind --
// in the K-major 32B-swizzled operand layout (row r at (r / 8) * 256 B + (r % 8) * 32 B,
// 16-byte chunk c at position c ^ ((r / 4) % 2); halves 16..31 in the second K block)
template <int NIN>
__device__ __forceinline__ void write_a1tc_row(unsigned char *a1, int r, const float (&x)[5]) {
    constexpr int KS = NIN == 3 ? 16 : 32;
    unsigned short h[KS];
#pragma unroll
    for (int i = 0; i < KS; ++i) h[i] = 0;
#pragma unroll
    for (int c = 0; c < NIN; ++c) {
        unsigned short hi, lo;
        split_half(x[c], hi, lo);
        h[3 * c] = hi; h[3 * c + 1] = hi; h[3 * c + 2] = lo;
    }
    h[3 * NIN] = 0x3C00; h[3 * NIN + 1] = 0x3C00;                       // 1.0
    unsigned char *rowp = a1 + (r >> 3) * 256 + (r & 7) * 32;
#pragma unroll
    for (int i = 0; i < KS / 8; ++i)
        *reinterpret_cast<uint4 *>(rowp + (i >> 1) * A1TC_KB_BYTES + (((i & 1) ^ ((r >> 2) & 1)) << 4)) =
            make_uint4((uint32_t)h[8 * i] | ((uint32_t)h[8 * i + 1] << 16), (uint32_t)h[8 * i + 2] | ((uint32_t)h[8 * i + 3] << 16),
                       (uint32_t)h[8 * i + 4] | ((uint32_t)h[8 * i + 5] << 16), (uint32_t)h[8 * i + 6] | ((uint32_t)h[8 * i + 7] << 16));
}
// one lane of a CONVERGED warp (elect.sync): the MMA / TMA issue loops run warp-converged with the issuing
// instructions predicated on this, so ptxas emits each UTCHMMA once with uniform-register operands instead of the
// elect / execute / retire loop it needs inside a divergent `if (lane == 0)` region (8 SASS instructions and ~80
// cycles per MMA there, more than the 64 cycles the MMA itself takes)
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Order in which a tile-step's weight stages (accumulator quarter nq, K block kb2 of KCH_PER_STAGE chunks) are streamed and issued.
template <int SPQ>
__device__ __forceinline__ void mlp_stage_map(int s, int &nq, int &kb2) { nq = s / SPQ; kb2 = s % SPQ; }

// ---- hand-off of a split quad / pair between neighbouring clusters (balanced schedule) ----
// Records live at hand[tile slot][6][128] (x, y, yaw, cost so far, previous control), tile slot = ((consumer cluster * 2 +
// rank) * 2 + ping-pong slot); flags at hand_flag[consumer cluster * 2 + rank] hold the epoch of the launch that published.
// Producer: every owner thread stores its row (st.global.cg), fences, the owner groups meet at named barrier 2 and one thread
// releases the flag.  Consumer: one lane per warp polls with ld.acquire.gpu (guarded, ~4 s: never hang the device; a missing
// record turns the cost into NaN instead of garbage), then every thread reads its row past L1 (ld.global.cg).
__device__ __forceinline__ void handoff_give(float *hand, unsigned int *hand_flag, unsigned int epoch, int tile_slot, int flag_idx,
                                             int row, bool signaller, int n_owner_threads, const float (&z)[4], float acc, float vp0, float vp1) {
    MPPI_DCHECK(tile_slot >= 0 && flag_idx >= 0 && row >= 0 && row < TILE_M);
    float *rec = hand + (size_t)tile_slot * 6 * TILE_M + row;
    __stcg(rec, z[0]); __stcg(rec + TILE_M, z[1]); __stcg(rec + 2 * TILE_M, z[2]);
    __stcg(rec + 3 * TILE_M, acc); __stcg(rec + 4 * TILE_M, vp0); __stcg(rec + 5 * TILE_M, vp1);
    __threadfence();
    named_bar_sync(2, n_owner_threads);
    if (signaller) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(hand_flag + flag_idx), "r"(epoch) : "memory");
}
__device__ __forceinline__ void handoff_take(const float *hand, unsigned int *hand_flag, unsigned int *fault, unsigned int epoch, int tile_slot,
                                             int flag_idx, int row, int lane, float (&z)[4], float &acc, float &vp0, float &vp1) {
    unsigned int seen = epoch;
    if (lane == 0) {
        long long spins = 0;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(hand_flag + flag_idx) : "memory");
            if (seen != epoch) __nanosleep(200);
        } while (seen != epoch && ++spins < 20000000ll);
    }
    const bool handed = __shfl_sync(0xffffffffu, seen == epoch ? 1 : 0, 0) != 0;
    const float *rec = hand + (size_t)tile_slot * 6 * TILE_M + row;
    z[0] = __ldcg(rec); z[1] = __ldcg(rec + TILE_M); z[2] = __ldcg(rec + 2 * TILE_M);
    acc = __ldcg(rec + 3 * TILE_M); vp0 = __ldcg(rec + 4 * TILE_M); vp1 = __ldcg(rec + 5 * TILE_M);
    if (!handed) {                                        // never garbage: NaN costs make finalize_tick refuse the tick, and the
        acc = CUDART_NAN_F;                               // fault word tells the host why (MPPI_E_NUMERIC, "hand-off was missed")
        if (lane == 0) atomicExch(fault, epoch);
    }
}

// TRAJ (replays for the trajectory viewers): behind the K costs, S_out also receives the state after every Euler step, (K, T, 3),
// stored by the owner thread of each row from whichever cluster runs the step.
__device__ __forceinline__ void store_state(float *S_out, int K, int T, int k, int t, const float (&z)[4]) {
    float *xo = S_out + K + ((size_t)k * T + t) * 3;
    xo[0] = z[0]; xo[1] = z[1]; xo[2] = z[2];
}

template <int NIN, bool PP, int NG, bool TRAJ = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MLP_THREADS, 1)
mppi_mlp_rollout_kernel(const __grid_constant__ TickArgs a, const __grid_constant__ CUtensorMap w2_map,
                        const float4 *__restrict__ g_w01, const float2 *__restrict__ g_w01u, const float4 *__restrict__ g_w3,
                        const float *__restrict__ g_b3, const float *__restrict__ g_bh, float *__restrict__ S_out, int n_tiles,
                        float *__restrict__ hand, unsigned int *__restrict__ hand_flag, unsigned int *__restrict__ fault,
                        unsigned int epoch, int balanced, const __half *__restrict__ g_b1
                        ) {
    static_assert(NG == 1 || (NG == 2 && !PP), "two GEMMs per step run the one-tile schedule");
    // 1024-byte alignment is what SWIZZLE_128B needs; keeping every pointer derived from this symbol (no
    // integer round-trips) lets the compiler emit LDS/STS instead of generic LD/ST
    extern __shared__ __align__(1024) unsigned char dyn[];
    unsigned char *smB = dyn + (NG == 2 ? A2_BYTES : 0);          // weight ring, 1024-aligned (NG = 2: after the A2 tile)
    unsigned char *smA2 = dyn;                                    // NG = 2: 8 K-chunks x [128 rows x 128 B], 128B swizzle
    TickSmem &sm = *reinterpret_cast<TickSmem *>(dyn + RING_BYTES);
    MlpSmem &ms = *reinterpret_cast<MlpSmem *>(dyn + RING_BYTES + sizeof(TickSmem));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int T = a.T;
    // clusters of two CTAs advance in lockstep: cluster c owns tile pairs c, c + n_clusters, ...; both CTAs run
    // the same number of tile-steps even when the last pair is half empty
    const uint32_t cta_rank = cluster_ctarank();
    const int n_clusters = (int)gridDim.x / 2, cluster_id = (int)blockIdx.x / 2;
    const int n_pairs = (n_tiles + 1) / 2;
    const int my_tiles = (n_pairs - cluster_id + n_clusters - 1) / n_clusters;
    // ping-pong mode walks the CTA's tiles two at a time (an odd count is padded with an empty tile)
    const int my_slots = PP ? 2 * ((my_tiles + 1) / 2) : my_tiles;
    // BALANCED ping-pong schedule.  A cluster's unit of work is a quad (2 CTAs x 2 tiles) x one timestep; n_quads * T of
    // them rarely divide by the cluster count (K = 65 536: 128 quads over 74 clusters -- whole quads leave 13.5 % of the
    // SM-time idle).  Cluster c takes the contiguous range [bal_b0, bal_b1) of the quad-major step sequence, cut at even
    // timesteps: the TAIL of one quad (steps t0..T-1), whole quads, and the HEAD of another (steps 0..t1-1).  It runs the
    // head FIRST and publishes the 128 x 6-float state record per tile (x, y, yaw, cost so far, previous control) with a
    // release flag; the next cluster runs that quad's tail LAST, so the record is ready long before it is needed.
    // (one-tile schedule, NG = 2: the unit is a PAIR -- 2 CTAs x 1 tile -- x one timestep, same rule)
    const int n_quads = PP ? (n_tiles + 3) / 4 : (n_tiles + 1) / 2;
    const int bal_b0 = balanced ? mlp_bal_cut(cluster_id, n_clusters, n_quads, T) : 0;
    const int bal_b1 = balanced ? mlp_bal_cut(cluster_id + 1, n_clusters, n_quads, T) : 0;
    const int my_tile_steps = balanced ? (PP ? 2 : 1) * (bal_b1 - bal_b0) : my_slots * T;    // tile-steps of this CTA

    // ---- one-time setup: constants, barriers, TMEM, step-1 index + window (same rule as the tick kernel)
    constexpr bool L1TC = mlp_use_l1tc(NIN, PP, NG);          // layer 1 on the tcgen05 tensor core
    constexpr bool CG2 = mlp_use_cg2(NIN, PP, NG);            // pair MMAs (cta_group::2, M = 256)
    // ring geometry of the one-GEMM kernels: K chunks per stage, stages, stages per accumulator quarter / per tile-step.  The tcgen05
    // layer 1 follows quarter 3 K part by K part (one 128-column part = two K chunks per stage) and keeps 40 KB for its own operands
    constexpr int KPS = L1TC ? 2 : KCH_PER_STAGE;
    constexpr int NSTG = L1TC ? 4 : (CG2 ? RING_BYTES / (KPS * CG2_BOX_BYTES) : B_STAGES);
    constexpr int SPQ = HID / KCH / KPS, SPS = N_QUARTERS * SPQ;
    constexpr int B1_OFF = NSTG * KPS * B_BOX_BYTES;           // tcgen05 layer-1 operands behind the ring
    static_assert(NSTG <= RING_SLOTS && (!L1TC || B1_OFF + B1TC_BYTES + A1TC_BYTES <= RING_BYTES), "ring geometry");
    unsigned char *smA1 = dyn + B1_OFF + B1TC_BYTES;                  // its A operand (this step's split input rows)
    for (int j = tid; j < HID; j += MLP_THREADS) {
        ms.w3[j] = g_w3[j];
        if (!L1TC) {
            ms.w01[j] = g_w01[j];
            if (NIN == 5) ms.w01u[j] = g_w01u[j];
        }
    }
    if (L1TC) {                                               // B operand as the host laid it out (swizzled); A rows start as zeros
        for (int i = tid; i < B1TC_BYTES / 16; i += MLP_THREADS)
            reinterpret_cast<uint4 *>(dyn + B1_OFF)[i] = reinterpret_cast<const uint4 *>(g_b1)[i];
        for (int i = tid; i < A1TC_BYTES / 16; i += MLP_THREADS) reinterpret_cast<uint4 *>(smA1)[i] = make_uint4(0u, 0u, 0u, 0u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (tid < 3) ms.b3[tid] = g_b3[tid];
    if (tid < 4) sm.x0[tid] = a.x0[tid];
    if (tid == 0) {
        // multicast TMA: a slot is free when BOTH CTAs' MMAs have read it (2); pair MMAs: one commit frees each CTA's own half (1).
        // Pair MMAs: the compute warps of both CTAs report to rank 0's a_ready / d_empty
        for (int s = 0; s < RING_SLOTS; ++s) { mbar_init(&ms.b_full[s], 1); mbar_init(&ms.b_empty[s], CG2 ? 1 : 2); }
        for (int pa = 0; pa < N_QUARTERS; ++pa) { mbar_init(&ms.a_ready[pa], CG2 ? 2 * N_ARRIVE : N_ARRIVE); mbar_init(&ms.a_free[pa], 1); }
        for (int bf = 0; bf < 2; ++bf) { mbar_init(&ms.d_full[bf], 1); mbar_init(&ms.d_empty[bf], CG2 ? 2 * N_ARRIVE : N_ARRIVE); }
        for (int pa = 0; pa < N_QUARTERS; ++pa) mbar_init(&ms.a2_ready[pa], N_ARRIVE);
        if (L1TC) { mbar_init(&ms.a1_ready, N_ARRIVE / N_GROUPS); mbar_init(&ms.d1_full, 1); mbar_init(&ms.d1_empty, N_ARRIVE); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if constexpr (CG2) {                                  // the same warp of both CTAs allocates the pair's tensor memory
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ms.tmem_base)), "r"(512));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ms.tmem_base)), "r"(512));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        }
    }
    __syncthreads();
    {
        const int s_old = max(0, min(a.idx[0], a.n_path - 1));
        unsigned long long key = ~0ull;
        for (int j = tid; j < a.window && s_old + j < a.n_path; j += MLP_THREADS) {
            const float4 p = a.path[s_old + j];
            const float dx = sm.x0[0] - p.x, dy = sm.x0[1] - p.y;
            const unsigned long long kj = ((unsigned long long)__float_as_uint(dx * dx + dy * dy) << 32) | (unsigned)j;
            key = kj < key ? kj : key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other < key ? other : key;
        }
        if (lane == 0 && warp < 8) ms.key[warp] = key;
        __syncthreads();
        if (warp >= 8) {                                     // warps 8,9 fold their candidates in serially
            if (lane == 0) atomicMin(&ms.key[0], key);
        }
        __syncthreads();
        key = ms.key[0];
#pragma unroll
        for (int w = 1; w < 8; ++w) key = ms.key[w] < key ? ms.key[w] : key;
        const int s_new = s_old + (int)(key & 0xffffffffu);
        int nw = a.n_path - s_new; nw = nw < a.window ? nw : a.window;
        const int fill = (a.window == 20) ? 20 : ((nw + 15) & ~15);
        for (int j = tid; j < fill; j += MLP_THREADS) {
            if (j < nw) {
                const float4 p = a.path[s_new + j];
                sm.wx[j] = -p.x; sm.wy[j] = -p.y; sm.wyv[j] = make_float2(p.z, p.w);
            } else {
                sm.wx[j] = -MPPI_SENTINEL; sm.wy[j] = -MPPI_SENTINEL; sm.wyv[j] = make_float2(0.f, 0.f);
            }
        }
        if (tid == 0) { sm.win_start = s_new; sm.n_win16 = fill >> 4; }
        if (a.window == 20) { __syncthreads(); fill_window_expanded(sm, nw, tid, MLP_THREADS); }
        if (a.window != 20) {
            __syncthreads();
            for (int c = tid; c < (fill >> 4); c += MLP_THREADS) sm.cb[c] = chunk_bound(sm.wx, sm.wy, 16 * c, min(16, nw - 16 * c));
        }
        for (int t = tid; t < T; t += MLP_THREADS) {
            const float u0 = a.U[2 * t], u1 = a.U[2 * t + 1];
            sm.U[t] = make_float2(u0, u1);
            sm.Q[t] = make_float2(u0 * a.gq[0] + u1 * a.gq[2], u0 * a.gq[1] + u1 * a.gq[3]);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();                                   // the peer's barriers exist before anything is multicast
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = ms.tmem_base;

    if (warp == 0) {
        // ===== TMA producer: the same 16 W2 boxes every timestep, through a NSTG ring =====
        const bool leader = elect_one_sync();
        if constexpr (NG == 2) {
            // two layers' weights back to back: per step 2 GEMMs x 4 quarters x 8 K-chunks, one 16 KB box per stage;
            // the tensor map stacks the layers, rows [512 g, 512 g + 512)
            const int total = my_tile_steps * NG * N_QUARTERS * (HID / KCH);
            int stage = 0; uint32_t phase = 0;
            for (int it = 0; it < total; ++it) {
                const int kc = it % (HID / KCH), nq = (it / (HID / KCH)) % N_QUARTERS, g = (it / (HID / KCH * N_QUARTERS)) % NG;
                mbar_wait(&ms.b_empty[stage], phase ^ 1);
                if (leader) {
                    mbar_expect_tx(&ms.b_full[stage], B_BOX_BYTES);
                    if ((uint32_t)(it & 1) == cta_rank)
                        tma_load_2d_mc(smB + stage * B_BOX_BYTES, &w2_map, &ms.b_full[stage], kc * KCH, g * HID + nq * N_MMA, (uint16_t)3);
                }
                __syncwarp();
                if (++stage == B2_STAGES) { stage = 0; phase ^= 1; }
            }
        } else {
        const int total = my_tile_steps * SPS;
        int stage = 0; uint32_t phase = 0;
        for (int it = 0; it < total; ++it) {
            int nq, kb2;
            mlp_stage_map<SPQ>(it % SPS, nq, kb2);
            mbar_wait(&ms.b_empty[stage], phase ^ 1);               // both CTAs are done with this slot
            if constexpr (CG2) {
                // pair MMAs: every CTA loads ITS half of the box rows (64 of 128) into its own ring; all bytes of the pair are
                // counted on rank 0's barrier, which rank 0 arms for both halves
                if (leader) {
                    if (cta_rank == 0) mbar_expect_tx(&ms.b_full[stage], 2 * (KPS * CG2_BOX_BYTES));
#pragma unroll
                    for (int j = 0; j < KPS; ++j)
                        tma_load_2d_2sm(smB + stage * (KPS * CG2_BOX_BYTES) + j * CG2_BOX_BYTES, &w2_map, &ms.b_full[stage],
                                        (kb2 * KPS + j) * KCH, nq * N_MMA + (int)cta_rank * (N_MMA / 2));
                }
                __syncwarp();
                if (++stage == NSTG) { stage = 0; phase ^= 1; }
                continue;
            }
            if (leader) {
                mbar_expect_tx(&ms.b_full[stage], (KPS * B_BOX_BYTES));    // every CTA arms its own barrier ...
                if ((uint32_t)(it & 1) == cta_rank) {                // ... and issues every other stage for both
#pragma unroll
                    for (int j = 0; j < KPS; ++j)
                        tma_load_2d_mc(smB + stage * (KPS * B_BOX_BYTES) + j * B_BOX_BYTES, &w2_map, &ms.b_full[stage],
                                       (kb2 * KPS + j) * KCH, nq * N_MMA, (uint16_t)3);
                }
            }
            __syncwarp();
            if (++stage == NSTG) { stage = 0; phase ^= 1; }
        }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one elected lane of the converged warp drives the tensor core =====
        const bool leader = elect_one_sync();
        int stage = 0; uint32_t phase = 0, a_phase = 0;
        MLP_PROBE_DECL();
        if constexpr (NG == 2) {
            uint32_t quarter = 0;
            for (int step = 0; step < my_tile_steps; ++step) {
                for (int g = 0; g < NG; ++g) {
                    for (int nq = 0; nq < N_QUARTERS; ++nq, ++quarter) {
                        const uint32_t buf = quarter & 1;
                        mbar_wait(&ms.d_empty[buf], ((quarter >> 1) & 1) ^ 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t d_tmem = tmem + TMEM_D_COL + buf * N_MMA;
                        for (int kc = 0; kc < HID / KCH; ++kc) {
                            // the first quarter of each GEMM chases its A operand part by part (a part = two K-chunks):
                            // GEMM 1 reads the layer-1 activations from tensor memory, GEMM 2 the tile GEMM 1's epilogue
                            // wrote to shared memory
                            if (nq == 0 && (kc & 1) == 0) mbar_wait(g == 0 ? &ms.a_ready[kc >> 1] : &ms.a2_ready[kc >> 1], a_phase);
                            mbar_wait(&ms.b_full[stage], phase);
                            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            const uint64_t b_desc0 = umma_desc_sw128(smem_u32(smB + stage * B_BOX_BYTES));
                            const uint64_t a_desc0 = umma_desc_sw128(smem_u32(smA2 + kc * B_BOX_BYTES));
                            const uint32_t a_col0 = tmem + TMEM_A_COL + kc * (KCH / 16) * 8;
                            if (leader) {
#pragma unroll
                                for (int k = 0; k < KCH / 16; ++k) {
                                    if (g == 0) umma_f16_ts(d_tmem, a_col0 + k * 8, b_desc0 + (uint64_t)((k * 32) >> 4), (kc | k) ? 1u : 0u);
                                    else umma_f16_ss(d_tmem, a_desc0 + (uint64_t)((k * 32) >> 4), b_desc0 + (uint64_t)((k * 32) >> 4), (kc | k) ? 1u : 0u);
                                }
                                umma_commit_mc(&ms.b_empty[stage], (uint16_t)3);
                            }
                            __syncwarp();
                            if (++stage == B2_STAGES) { stage = 0; phase ^= 1; }
                        }
                        if (leader) umma_commit(&ms.d_full[buf]);
                        __syncwarp();
                    }
                }
                a_phase ^= 1;
            }
        } else {
        // tcgen05 layer 1 (L1TC): evaluation #n feeds GEMM #n.  #0 is issued on its own; #(n+1) is slipped into GEMM #n's quarter 3 (see
        // the order below).  A part waits for its inputs (part 0: a1_ready, and quarter 2 read out of buffer 0) or for the previous
        // part to have been read back (d1_empty)
        uint32_t l1_n = 0, l1_parts = 0, d1e_n = 0;          // evaluation being issued, its parts issued so far, d1_empty phases consumed
        bool l1_inline = false; (void)l1_inline;
        auto l1_issue_part = [&]() {
            if (l1_parts == 0) {
                mbar_wait(&ms.a1_ready, l1_n & 1);
                if (l1_n > 0) mbar_wait(&ms.d_empty[0], 1u);            // quarter 2 of the running GEMM has been read out of buffer 0
            } else {
                mbar_wait(&ms.d1_empty, d1e_n & 1);
                ++d1e_n;
            }
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (leader) {
                const uint64_t a_desc = umma_desc_sw32(smem_u32(smA1));
                const uint64_t b_desc = umma_desc_sw32(smem_u32(dyn + B1_OFF + (int)l1_parts * (N_MMA * 32)));
                umma_f16_ss(tmem + TMEM_D_COL, a_desc, b_desc, 0u);
                if (NIN == 5) umma_f16_ss(tmem + TMEM_D_COL, a_desc + (uint64_t)(A1TC_KB_BYTES >> 4), b_desc + (uint64_t)(B1TC_KB_BYTES >> 4), 1u);   // second K block
                umma_commit(&ms.d1_full);
            }
            __syncwarp();
            if (++l1_parts == N_QUARTERS) { l1_parts = 0; ++l1_n; }
        };
        if constexpr (L1TC) {
            if (my_tile_steps > 0) for (int p = 0; p < N_QUARTERS; ++p) l1_issue_part();
        }
        for (int step = 0; step < ((!CG2 || cta_rank == 0) ? my_tile_steps : 0); ++step) {      // pair MMAs: rank 0 issues for both CTAs
            for (int s = 0; s < SPS; ++s) {
                int nq, kb2;
                mlp_stage_map<SPQ>(s, nq, kb2);
                // quarter Q = 4 step + nq of this CTA runs in buffer Q & 1 = nq & 1; its previous user was quarter Q - 2
                const uint32_t buf = (uint32_t)nq & 1u;
                MLP_TIC();
                if (kb2 == 0) {
                    mbar_wait(&ms.d_empty[buf], (((uint32_t)nq >> 1) & 1u) ^ 1u);      // epilogue drained this buffer
                    if (L1TC && nq == 0) { mbar_wait(&ms.d1_empty, d1e_n & 1); ++d1e_n; }      // ... and layer 1's last part has left it
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                MLP_TOC(nq);
                const uint32_t d_tmem = tmem + TMEM_D_COL + buf * N_MMA;
                // the activations arrive in four 128-column parts (a stage spans KPS / 2 of them); the first
                // quarter's K loop chases them
                if (nq == 0) {
#pragma unroll
                    for (int pa = 0; pa < KPS / 2; ++pa) mbar_wait(&ms.a_ready[kb2 * (KPS / 2) + pa], a_phase);
                }
                MLP_TOC(4 + (kb2 * KPS / 2 & 3));
                mbar_wait(&ms.b_full[stage], phase);
                MLP_TOC(8 + nq);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                // one descriptor per stage; the K-steps only bump its 14-bit start-address field
                constexpr int BOX_B = CG2 ? CG2_BOX_BYTES : B_BOX_BYTES, TILE_B = KPS * BOX_B;
                const uint64_t b_desc0 = umma_desc_sw128(smem_u32(smB + stage * TILE_B));
                const uint32_t a_col0 = tmem + TMEM_A_COL + kb2 * KPS * (KCH / 16) * 8;
                if (leader) {
#pragma unroll
                    for (int k = 0; k < KPS * (KCH / 16); ++k) {
                        const uint64_t b_desc = b_desc0 + (uint64_t)(((k / (KCH / 16)) * BOX_B + (k % (KCH / 16)) * 32) >> 4);
                        if constexpr (CG2) umma_f16_ts_2sm(d_tmem, a_col0 + k * 8, b_desc, (kb2 | k) ? 1u : 0u);
                        else umma_f16_ts(d_tmem, a_col0 + k * 8, b_desc, (kb2 | k) ? 1u : 0u);
                        // ping-pong: quarter 3 is the last reader of A -- release each 128-column part as soon as its MMAs
                        // retire so the other tile's layer 1 can overwrite it
                        if (PP && !L1TC && nq == N_QUARTERS - 1 && (k & 7) == 7) {
                            if constexpr (CG2) umma_commit_2sm_mc(&ms.a_free[kb2 * (KPS / 2) + (k >> 3)], (uint16_t)3);
                            else umma_commit(&ms.a_free[kb2 * (KPS / 2) + (k >> 3)]);
                        }
                    }
                    if constexpr (CG2) {
                        umma_commit_2sm_mc(&ms.b_empty[stage], (uint16_t)3);           // frees each CTA's half of the slot
                        if (kb2 == SPQ - 1) umma_commit_2sm_mc(&ms.d_full[buf], (uint16_t)3);
                    } else {
                        umma_commit_mc(&ms.b_empty[stage], (uint16_t)3);   // frees the W2 slot in BOTH CTAs when these MMAs retire
                        if (kb2 == SPQ - 1) umma_commit(&ms.d_full[buf]);         // this accumulator quarter is complete
                    }
                }
                __syncwarp();
                if (++stage == NSTG) { stage = 0; phase ^= 1; }
                if (L1TC && nq == N_QUARTERS - 1 && step + 1 < my_tile_steps) {
                    // Issue order K0 K1 [L1 p0] K2 [L1 p1] K3 [L1 p2] [L1 p3]: a part is issued one K part of quarter 3 late, so the
                    // wait for its buffer (quarter 2 drained / previous part read back) is covered by MMAs already queued.  Only if
                    // the inputs are there by K1 (always, inside a segment: they are published at the start of the slot); at a
                    // segment boundary the next tile's inputs come after this GEMM's epilogue -- waiting here would deadlock -- so
                    // the whole evaluation follows the quarter.
                    if (kb2 == 1) l1_inline = mbar_test_warp(&ms.a1_ready, l1_n & 1);
                    if (l1_inline && kb2 >= 1) l1_issue_part();
                    if (kb2 == SPQ - 1) { while ((int)l1_n == step + 1) l1_issue_part(); l1_inline = false; }
                }
            }
            a_phase ^= 1;
        }
        }
        MLP_PROBE_PRINT("issuer: wait d_empty q0-3 | a_ready p0-3 | b_full q0-3", my_tile_steps);
    } else {
        // ===== compute warps: rows = TMEM lanes 32*(warp%4)..+31, column group grp =====
        if constexpr (PP) {
        // ---- ping-pong mode: two tiles X, Y per CTA.  While the tensor core runs the GEMM of one tile, the compute
        // warps finish the other tile's previous step (last epilogue quarter, Euler), generate its next control and
        // evaluate its layer 1 into the A region part by part as the running GEMM's LAST quarter releases the parts
        // (a_free).  Tile X is owned (state, cost, noise) by column group 0, tile Y by group 1; every group helps with
        // the layer-1 columns and the epilogue of both.  GEMM order: X(0) Y(0) X(1) Y(1) ... ; L1 #l feeds GEMM #l.
        const int cw = warp - 2;
        const int q = warp & 3, grp = cw >> 2;
        const int row = q * 32 + lane;
        const bool owner = grp < 2;
        uint32_t d_phase[2] = {0, 0};
        uint32_t l1_count = 0, d1_phase = 0;
        MLP_PROBE_DECL();
        // segments of this CTA: static = tile pairs over the whole horizon; balanced = [head], whole quads, [tail]
        const int g_first = balanced ? bal_b0 / T : 0;
        const int n_nat = balanced ? (bal_b1 > bal_b0 ? (bal_b1 - 1) / T - g_first + 1 : 0) : my_slots / 2;
        const bool head_first = balanced && n_nat > 1 && (bal_b1 % T) != 0;
        for (int pr = 0; pr < n_nat; ++pr) {
            int tile, t0 = 0, t1 = T;
            bool valid = true;
            if (balanced) {
                // natural order j = 0 (maybe a tail) .. n_nat-1 (maybe a head); run order: the head, the middle ones, j = 0 last
                const int j = pr == n_nat - 1 ? 0 : head_first ? (pr == 0 ? n_nat - 1 : pr) : pr + 1;
                const int g = g_first + j;
                t0 = max(bal_b0 - g * T, 0); t1 = min(bal_b1 - g * T, T);
                tile = 4 * g + 2 * (grp & 1) + (int)cta_rank;
            } else {
                const int tl = 2 * pr + (grp & 1);
                tile = 2 * (cluster_id + tl * n_clusters) + (int)cta_rank;
                valid = tl < my_tiles;
            }
            const int k = tile * TILE_M + row;
            const bool active = owner && valid && k < a.K;
            const uint32_t kg = (uint32_t)(a.k_offset + k);
            const bool exploit = (int)kg < a.n_exploit;
            float z[4] = {sm.x0[0], sm.x0[1], sm.x0[2], 0.f};
            float acc = 0.f, e[4] = {0.f, 0.f, 0.f, 0.f}, sn = 0.f, cs = 1.f;
            float vp0 = 0.f, vp1 = 0.f, vc0 = 0.f, vc1 = 0.f;          // controls of steps t-1 and t
            if (t0 > 0 && owner)                                   // tail of a split quad: the previous cluster's record
                handoff_take(hand, hand_flag, fault, epoch, (cluster_id * 2 + (int)cta_rank) * 2 + (grp & 1), 2 * cluster_id + (int)cta_rank,
                             row, lane, z, acc, vp0, vp1);
            float4 ref = make_float4(0.f, 0.f, 0.f, 0.f);
            const float2 *eps_k = a.eps ? reinterpret_cast<const float2 *>(a.eps) + (size_t)(active ? k : 0) * T : nullptr;
            // owner: stage cost of the state reached by step t-1, noise + clamped control of step t, heading sin/cos
            auto prep = [&](int t) {
                if (t > 0 && (a.flags & F_COST_SUM)) {
                    const int j = a.window == 20 ? nearest_wp<20>(sm, z[0], z[1]) : nearest_wp<0>(sm, z[0], z[1]);
                    ref = window_ref(sm, j);
                    const float2 qq = sm.Q[t - 1];
                    acc += tracking_cost<MPPI_MODEL_DIFFDRIVE>(ref, z, z[2], a.sw) + (qq.x * vp0 + qq.y * vp1);
                }
                if (eps_k) { const float2 ee = eps_k[t]; e[2 * (t & 1)] = ee.x; e[2 * (t & 1) + 1] = ee.y; }
                else if ((t & 1) == 0) philox_eps_pair(a, kg, (uint32_t)(t >> 1), 0u, e);
                const float2 u = sm.U[t];
                vc0 = clampf(exploit ? __fadd_rn(u.x, e[2 * (t & 1)]) : e[2 * (t & 1)], a.umax0);
                vc1 = clampf(exploit ? __fadd_rn(u.y, e[2 * (t & 1) + 1]) : e[2 * (t & 1) + 1], a.umax1);
                sincos_cw(z[2], sn, cs);
            };
            // layer 1 of the tile owned by group og -> A region (L1 #l1_count, consumed by GEMM #l1_count)
            // tcgen05 layer 1, compute side.  l1_publish: the owner group writes its tile's split input rows (as soon as the state is
            // known -- the issuer slips the MMAs into the running GEMM's last quarter only if they are there in time);
            // l1_collect: every group reads its 32 columns of each part back from accumulator buffer 0, applies tanh, rounds once and
            // stores the operand into A part p (the part's commit also proves the running GEMM is done with that part of A)
            auto l1_publish = [&](int og) {
                if (grp == og) {
                    const float xin[5] = {z[0], z[1], z[2], vc0, vc1};
                    write_a1tc_row<NIN>(smA1, row, xin);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> the tensor core's reads
                    compute_arrive(&ms.a1_ready);
                }
            };
            auto l1_collect = [&]() {
#pragma unroll 1
                for (int part = 0; part < N_QUARTERS; ++part) {
                    MLP_TIC();
                    mbar_wait_warp(&ms.d1_full, d1_phase); d1_phase ^= 1;
                    MLP_TOC(4 + part);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    uint32_t v[32];
                    tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(TMEM_D_COL + grp * 32), v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    compute_arrive(&ms.d1_empty);
#pragma unroll
                    for (int c8 = 0; c8 < 4; ++c8) {
                        uint32_t pk[4];
#pragma unroll
                        for (int pp = 0; pp < 4; ++pp) pk[pp] = tanh_op2(__uint_as_float(v[8 * c8 + 2 * pp]), __uint_as_float(v[8 * c8 + 2 * pp + 1]));
                        tmem_st4(tmem + ((uint32_t)(q * 32) << 16) + TMEM_A_COL + (uint32_t)((part * N_MMA + grp * 32 + c8 * 8) >> 1), pk[0], pk[1], pk[2], pk[3]);
                    }
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    compute_arrive<CG2>(&ms.a_ready[part]);
                    MLP_TOC(8 + part);
                }
                ++l1_count;
            };
            auto layer1 = [&](int og) {
                if constexpr (L1TC) { l1_publish(og); l1_collect(); return; }
                if (grp == og) {
                    ms.xs[row] = make_float4(z[0], z[1], z[2], vc0);
                    if (NIN == 5) ms.xw[row] = vc1;
                }
                MLP_TIC();
                named_bar_sync(1, N_COMPUTE);
                MLP_TOC(13);
                const float4 st = ms.xs[row];
                const float su1 = NIN == 5 ? ms.xw[row] : 0.f;
#pragma unroll 1
                for (int part = 0; part < N_QUARTERS; ++part) {
                    MLP_TIC();
                    if (l1_count > 0) {                                   // GEMM #(l1_count-1) is done with this part of A
                        mbar_wait_warp(&ms.a_free[part], (l1_count - 1) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    }
                    MLP_TOC(4 + part);
#pragma unroll 2
                    for (int c8 = 0; c8 < 4; ++c8) {
                        const int col = part * N_MMA + grp * 32 + c8 * 8;
                        uint32_t pk[4];
#pragma unroll
                        for (int p = 0; p < 4; ++p) {
                            const float4 wa = ms.w01[col + 2 * p], wb = ms.w01[col + 2 * p + 1];
                            float pa = fmaf(wa.x, st.x, fmaf(wa.y, st.y, fmaf(wa.z, st.z, wa.w)));
                            float pb = fmaf(wb.x, st.x, fmaf(wb.y, st.y, fmaf(wb.z, st.z, wb.w)));
                            if (NIN == 5) {
                                const float4 wu = *reinterpret_cast<const float4 *>(&ms.w01u[col + 2 * p]);
                                pa = fmaf(wu.x, st.w, fmaf(wu.y, su1, pa));
                                pb = fmaf(wu.z, st.w, fmaf(wu.w, su1, pb));
                            }
                            pk[p] = tanh_op2(pa, pb);
                        }
                        tmem_st4(tmem + ((uint32_t)(q * 32) << 16) + TMEM_A_COL + (uint32_t)(col >> 1), pk[0], pk[1], pk[2], pk[3]);
                    }
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    compute_arrive<CG2>(&ms.a_ready[part]);
                    MLP_TOC(8 + part);
                }
                ++l1_count;
            };
            // one accumulator quarter: D -> +b2 -> tanh -> partial contraction with the 512x3 output layer
            auto epilogue = [&](int nq, float &r0, float &r1, float &r2) {
                const int col = nq * N_MMA + grp * 32;
                const int buf = nq & 1;
                MLP_TIC();
                mbar_wait_warp(&ms.d_full[buf], d_phase[buf]); d_phase[buf] ^= 1;
                MLP_TOC(nq);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                uint32_t v[32];
                tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(TMEM_D_COL + buf * N_MMA + grp * 32), v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                compute_arrive<CG2>(&ms.d_empty[buf]);
                MLP_TOC(12);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float4 w = ms.w3[col + i];
                    const float h = tanh_approx(__uint_as_float(v[i]) + w.x);
                    r0 = fmaf(w.y, h, r0); r1 = fmaf(w.z, h, r1); r2 = fmaf(w.w, h, r2);
                }
                MLP_TOC(15);
            };
            // the step of the tile owned by group og is complete: gather the partial sums, Euler step with the residual
            auto finish = [&](int og, float r0, float r1, float r2) {
                const int rel = (grp - og) & 3;
                if (rel) { ms.res[rel - 1][0][row] = r0; ms.res[rel - 1][1][row] = r1; ms.res[rel - 1][2][row] = r2; }
                MLP_TIC();
                named_bar_sync(1, N_COMPUTE);
                MLP_TOC(14);
                if (grp == og) {
                    // partial sums added in ascending GROUP order whichever group owns the tile, so a sample's result does not
                    // depend on the slot (X / Y) the schedule puts it in: the static and the balanced walk agree bit for bit
                    float t0s = 0.f, t1s = 0.f, t2s = 0.f;
#pragma unroll
                    for (int g = 0; g < N_GROUPS; ++g) {
                        const int rel = (g - og) & 3;
                        const float p0 = rel ? ms.res[rel - 1][0][row] : r0, p1 = rel ? ms.res[rel - 1][1][row] : r1,
                                    p2 = rel ? ms.res[rel - 1][2][row] : r2;
                        t0s = g ? t0s + p0 : p0; t1s = g ? t1s + p1 : p1; t2s = g ? t2s + p2 : p2;
                    }
                    r0 = t0s + ms.b3[0]; r1 = t1s + ms.b3[1]; r2 = t2s + ms.b3[2];
                    z[0] = fmaf(fmaf(vc0, cs, r0), a.dt, z[0]);
                    z[1] = fmaf(fmaf(vc0, sn, r1), a.dt, z[1]);
                    z[2] = fmaf(vc1 + r2, a.dt, z[2]);
                    vp0 = vc0; vp1 = vc1;
                }
            };

            if (owner) prep(t0);
            layer1(0);                                               // L1(X, t0)
            float r0, r1, r2;
            float s0 = 0.f, s1 = 0.f, s2 = 0.f;                      // partial sums of the tile whose GEMM ran one slot ago
            for (int t = t0; t < t1; ++t) {
                // ---- slot X(t): the tensor core runs GEMM X(t)
                if (t > t0) {
                    epilogue(3, s0, s1, s2);                         // Y(t-1), last quarter
                    finish(1, s0, s1, s2);
                    if constexpr (TRAJ) { if (grp == 1 && active) store_state(S_out, a.K, T, k, t - 1, z); }
                    if (grp == 1) prep(t);
                }
                if constexpr (L1TC) l1_publish(1);                   // inputs of L1(Y, t): the evaluation before it is long done
                r0 = r1 = r2 = 0.f;
                epilogue(0, r0, r1, r2); epilogue(1, r0, r1, r2); epilogue(2, r0, r1, r2);      // X(t)
                if constexpr (L1TC) l1_collect(); else layer1(1);    // L1(Y, t) chases X(t)'s last quarter
                // ---- slot Y(t): the tensor core runs GEMM Y(t)
                epilogue(3, r0, r1, r2);                             // X(t), last quarter
                finish(0, r0, r1, r2);
                if constexpr (TRAJ) { if (grp == 0 && active) store_state(S_out, a.K, T, k, t, z); }
                if (grp == 0 && t + 1 < t1) prep(t + 1);
                if constexpr (L1TC) { if (t + 1 < t1) l1_publish(0); }
                s0 = s1 = s2 = 0.f;
                epilogue(0, s0, s1, s2); epilogue(1, s0, s1, s2); epilogue(2, s0, s1, s2);      // Y(t)
                if (t + 1 < t1) { if constexpr (L1TC) l1_collect(); else layer1(0); }           // L1(X, t+1) chases Y(t)'s last quarter
            }
            epilogue(3, s0, s1, s2);                                 // Y(t1-1), last quarter
            finish(1, s0, s1, s2);
            if constexpr (TRAJ) { if (grp == 1 && active) store_state(S_out, a.K, T, k, t1 - 1, z); }
            if (warp == 2 && pr == n_nat - 1) MLP_PROBE_PRINT("compute warp 0: wait d_full q0-3 | a_free p0-3 | L1 work p0-3 | tmem ld, L1 bar, finish bar, epilogue math", my_tile_steps / 2);
            if (t1 < T) {
                // head of a split quad: publish the state after step t1-1 for the next cluster's tail
                if (owner)
                    handoff_give(hand, hand_flag, epoch, ((cluster_id + 1) * 2 + (int)cta_rank) * 2 + (grp & 1),
                                 2 * (cluster_id + 1) + (int)cta_rank, row, cw == 0 && lane == 0, 256, z, acc, vp0, vp1);
            } else if (active) {
                const int j = a.window == 20 ? nearest_wp<20>(sm, z[0], z[1]) : nearest_wp<0>(sm, z[0], z[1]);
                ref = window_ref(sm, j);
                const float2 qq = sm.Q[T - 1];
                const float last = tracking_cost<MPPI_MODEL_DIFFDRIVE>(ref, z, z[2], a.sw) + (qq.x * vp0 + qq.y * vp1) +
                                   tracking_cost<MPPI_MODEL_DIFFDRIVE>(ref, z, z[2], a.tw);
                acc = (a.flags & F_COST_SUM) ? acc + last : last;
                S_out[k] = acc;
            }
        }
        } else {
        const int cw = warp - 2;
        const int q = warp & 3, grp = cw >> 2;          // TMEM lane quarter (hardware: warp % 4), column group
        const int row = q * 32 + lane;
        const bool owner = grp == 0;
        uint32_t d_phase[2] = {0, 0};
        // segments: static = this CTA's tiles over the whole horizon; balanced = [head], whole pairs, [tail] (see above)
        const int g_first = balanced ? bal_b0 / T : 0;
        const int n_nat = balanced ? (bal_b1 > bal_b0 ? (bal_b1 - 1) / T - g_first + 1 : 0) : my_tiles;
        const bool head_first = balanced && n_nat > 1 && (bal_b1 % T) != 0;
        for (int tl = 0; tl < n_nat; ++tl) {
            int tile, t0 = 0, t1 = T;
            if (balanced) {
                const int j = tl == n_nat - 1 ? 0 : head_first ? (tl == 0 ? n_nat - 1 : tl) : tl + 1;
                const int g = g_first + j;
                t0 = max(bal_b0 - g * T, 0); t1 = min(bal_b1 - g * T, T);
                tile = 2 * g + (int)cta_rank;
            } else {
                tile = 2 * (cluster_id + tl * n_clusters) + (int)cta_rank;
            }
            const int k = tile * TILE_M + row;
            const bool active = k < a.K;
            const uint32_t kg = (uint32_t)(a.k_offset + k);
            const bool exploit = (int)kg < a.n_exploit;
            float z[4] = {sm.x0[0], sm.x0[1], sm.x0[2], 0.f};
            float acc = 0.f, e[4] = {0.f, 0.f, 0.f, 0.f}, sn = 0.f, cs = 1.f;
            float vp0 = 0.f, vp1 = 0.f, vc0 = 0.f, vc1 = 0.f, vn0 = 0.f, vn1 = 0.f;    // controls of steps t-1, t, t+1
            if (t0 > 0 && owner)                                   // tail of a split pair: the previous cluster's record
                handoff_take(hand, hand_flag, fault, epoch, (cluster_id * 2 + (int)cta_rank) * 2, 2 * cluster_id + (int)cta_rank,
                             row, lane, z, acc, vp0, vp1);
            float4 ref = make_float4(0.f, 0.f, 0.f, 0.f);
            const float2 *eps_k = a.eps ? reinterpret_cast<const float2 *>(a.eps) + (size_t)(active ? k : 0) * T : nullptr;
            // noise + clamped control of step t (A3-A5); called for t = 0, 1, 2, ... in order (a Philox call yields two steps)
            auto control = [&](int t, float &o0, float &o1) {
                if (eps_k) { const float2 ee = eps_k[t]; e[2 * (t & 1)] = ee.x; e[2 * (t & 1) + 1] = ee.y; }
                else if ((t & 1) == 0) philox_eps_pair(a, kg, (uint32_t)(t >> 1), 0u, e);
                const float2 u = sm.U[t];
                o0 = clampf(exploit ? __fadd_rn(u.x, e[2 * (t & 1)]) : e[2 * (t & 1)], a.umax0);
                o1 = clampf(exploit ? __fadd_rn(u.y, e[2 * (t & 1) + 1]) : e[2 * (t & 1) + 1], a.umax1);
            };
            if (owner) control(t0, vc0, vc1);
            for (int t = t0; t < t1; ++t) {
                // (1) owner publishes the state (and, for the 5-input residual, this step's control); every group
                //     evaluates its 128 columns of tanh(W01 [x; u] + b01)
                if (owner) {
                    ms.xs[row] = make_float4(z[0], z[1], z[2], vc0);
                    if (NIN == 5) ms.xw[row] = vc1;
                }
                named_bar_sync(1, N_COMPUTE);
                const float4 st = ms.xs[row];
                const float su1 = NIN == 5 ? ms.xw[row] : 0.f;
#pragma unroll 1
                for (int part = 0; part < N_QUARTERS; ++part) {      // 128-column parts of A, each signalled on its own
#pragma unroll 2
                    for (int c8 = 0; c8 < 4; ++c8) {                 // this group's 32 columns of the part, 8 at a time
                        const int col = part * N_MMA + grp * 32 + c8 * 8;
                        uint32_t pk[4];
#pragma unroll
                        for (int p = 0; p < 4; ++p) {
                            const float4 wa = ms.w01[col + 2 * p], wb = ms.w01[col + 2 * p + 1];
                            float pa = fmaf(wa.x, st.x, fmaf(wa.y, st.y, fmaf(wa.z, st.z, wa.w)));
                            float pb = fmaf(wb.x, st.x, fmaf(wb.y, st.y, fmaf(wb.z, st.z, wb.w)));
                            if (NIN == 5) {
                                const float4 wu = *reinterpret_cast<const float4 *>(&ms.w01u[col + 2 * p]);
                                pa = fmaf(wu.x, st.w, fmaf(wu.y, su1, pa));
                                pb = fmaf(wu.z, st.w, fmaf(wu.w, su1, pb));
                            }
                            pk[p] = tanh_op2(pa, pb);
                        }
                        tmem_st4(tmem + ((uint32_t)(q * 32) << 16) + TMEM_A_COL + (uint32_t)(col >> 1), pk[0], pk[1], pk[2], pk[3]);
                    }
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    compute_arrive(&ms.a_ready[part]);
                }
                // (2) owner overlaps with the GEMM: stage cost of the state reached by the previous step, then the
                //     noise and clamped control of the NEXT step
                if (owner) {
                    if (t > 0 && (a.flags & F_COST_SUM)) {
                        const int j = a.window == 20 ? nearest_wp<20>(sm, z[0], z[1]) : nearest_wp<0>(sm, z[0], z[1]);
                        ref = window_ref(sm, j);
                        const float2 qq = sm.Q[t - 1];
                        acc += tracking_cost<MPPI_MODEL_DIFFDRIVE>(ref, z, z[2], a.sw) + (qq.x * vp0 + qq.y * vp1);
                    }
                    if (t + 1 < t1) control(t + 1, vn0, vn1);
                    sincos_cw(z[2], sn, cs);
                }
                // (2b) three tanh layers: epilogue of GEMM 1 = the A operand of GEMM 2.  D -> +bias -> tanh -> fp16, stored
                //      to shared memory in the K-major 128B-swizzled layout (row r of K-chunk c at c*16 KB + (r/8)*1 KB +
                //      (r%8)*128 B, 16-byte units XORed with r%8): conflict-free, a quarter-warp covers all 32 banks
                if constexpr (NG == 2) {
#pragma unroll 1
                    for (int nq = 0; nq < N_QUARTERS; ++nq) {
                        const int col = nq * N_MMA + grp * 32;
                        const int buf = nq & 1;
                        mbar_wait_warp(&ms.d_full[buf], d_phase[buf]); d_phase[buf] ^= 1;
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        uint32_t v[32];
                        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(TMEM_D_COL + buf * N_MMA + grp * 32), v);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        compute_arrive(&ms.d_empty[buf]);
                        unsigned char *dst = smA2 + (col >> 6) * B_BOX_BYTES + (row >> 3) * 1024 + (row & 7) * 128;
                        const int c16 = (col & 63) >> 3;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            // (shared memory is full: the 2 KB bias vector is read through L1, warp-uniform addresses)
                            const float4 ba = __ldg(reinterpret_cast<const float4 *>(g_bh + col + 8 * c));
                            const float4 bb = __ldg(reinterpret_cast<const float4 *>(g_bh + col + 8 * c + 4));
                            uint4 pk;
                            pk.x = pack_op2(tanh_approx(__uint_as_float(v[8 * c + 0]) + ba.x), tanh_approx(__uint_as_float(v[8 * c + 1]) + ba.y));
                            pk.y = pack_op2(tanh_approx(__uint_as_float(v[8 * c + 2]) + ba.z), tanh_approx(__uint_as_float(v[8 * c + 3]) + ba.w));
                            pk.z = pack_op2(tanh_approx(__uint_as_float(v[8 * c + 4]) + bb.x), tanh_approx(__uint_as_float(v[8 * c + 5]) + bb.y));
                            pk.w = pack_op2(tanh_approx(__uint_as_float(v[8 * c + 6]) + bb.z), tanh_approx(__uint_as_float(v[8 * c + 7]) + bb.w));
                            *reinterpret_cast<uint4 *>(dst + (((c16 + c) ^ (row & 7)) << 4)) = pk;
                        }
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> the tensor core's reads
                        compute_arrive(&ms.a2_ready[nq]);
                    }
                }
                // (3) epilogue: D -> +b2 -> tanh -> FP32 contraction with the 512x3 output layer
                float r0 = 0.f, r1 = 0.f, r2 = 0.f;
#pragma unroll 1
                for (int nq = 0; nq < N_QUARTERS; ++nq) {         // every group takes 32 columns of EACH quarter, so the
                    const int col = nq * N_MMA + grp * 32;        // work exposed after the last MMA is 32 columns, not 128
                    const int buf = nq & 1;
                    mbar_wait_warp(&ms.d_full[buf], d_phase[buf]); d_phase[buf] ^= 1;
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    uint32_t v[32];
                    tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(TMEM_D_COL + buf * N_MMA + grp * 32), v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    compute_arrive(&ms.d_empty[buf]);                // values are in registers: the buffer may be overwritten
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const float4 w = ms.w3[col + i];
                        const float h = tanh_approx(__uint_as_float(v[i]) + w.x);
                        r0 = fmaf(w.y, h, r0); r1 = fmaf(w.z, h, r1); r2 = fmaf(w.w, h, r2);
                    }
                }
                if (!owner) { ms.res[grp - 1][0][row] = r0; ms.res[grp - 1][1][row] = r1; ms.res[grp - 1][2][row] = r2; }
                named_bar_sync(1, N_COMPUTE);
                // (4) owner: Euler step with the learned residual
                if (owner) {
#pragma unroll
                    for (int g = 0; g < N_GROUPS - 1; ++g) { r0 += ms.res[g][0][row]; r1 += ms.res[g][1][row]; r2 += ms.res[g][2][row]; }
                    r0 += ms.b3[0]; r1 += ms.b3[1]; r2 += ms.b3[2];
                    z[0] = fmaf(fmaf(vc0, cs, r0), a.dt, z[0]);
                    z[1] = fmaf(fmaf(vc0, sn, r1), a.dt, z[1]);
                    z[2] = fmaf(vc1 + r2, a.dt, z[2]);
                    vp0 = vc0; vp1 = vc1; vc0 = vn0; vc1 = vn1;
                    if constexpr (TRAJ) { if (active) store_state(S_out, a.K, T, k, t, z); }
                }
            }
            if (t1 < T) {
                if (owner)                                        // head of a split pair: hand the state to the next cluster
                    handoff_give(hand, hand_flag, epoch, ((cluster_id + 1) * 2 + (int)cta_rank) * 2, 2 * (cluster_id + 1) + (int)cta_rank,
                                 row, cw == 0 && lane == 0, 128, z, acc, vp0, vp1);
            } else if (owner && active) {
                // cost of the final state: last stage cost (+ terminal); in `last` mode nothing else survives (Q1)
                const int j = a.window == 20 ? nearest_wp<20>(sm, z[0], z[1]) : nearest_wp<0>(sm, z[0], z[1]);
                ref = window_ref(sm, j);
                const float2 qq = sm.Q[T - 1];
                const float last = tracking_cost<MPPI_MODEL_DIFFDRIVE>(ref, z, z[2], a.sw) + (qq.x * vp0 + qq.y * vp1) +
                                   tracking_cost<MPPI_MODEL_DIFFDRIVE>(ref, z, z[2], a.tw);
                acc = (a.flags & F_COST_SUM) ? acc + last : last;
                S_out[k] = acc;
            }
        }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();                                   // no CTA leaves while its peer may still signal its barriers
    if (warp == 1) {
        if constexpr (CG2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
    }
}

#ifdef MPPI_MLP_TRAJ_UNIT
typedef decltype(&mppi_mlp_rollout_kernel<3, false, 1, true>) MlpKernel;
#else
typedef decltype(&mppi_mlp_rollout_kernel<3, false, 1>) MlpKernel;
#endif

typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

// The instantiations, indexed by the (n_in, ping-pong, GEMMs per step) variant (n_in 3 / 5 alternate): the tick's here, the
// replays' (TRAJ) in mppi_mlp_traj.cu, which compiles this file with MPPI_MLP_TRAJ_UNIT.  Instantiated in this translation unit,
// the TRAJ kernels change how the device compiler numbers the shared code of <5, true, 1> and with it that kernel's machine
// code; apart, the tick's six compile exactly as they did without them.
extern const MlpKernel mlp_traj_kernels[6];
#ifdef MPPI_MLP_TRAJ_UNIT
const MlpKernel mlp_traj_kernels[6] = {
    mppi_mlp_rollout_kernel<3, false, 1, true>, mppi_mlp_rollout_kernel<5, false, 1, true>, mppi_mlp_rollout_kernel<3, true, 1, true>,
    mppi_mlp_rollout_kernel<5, true, 1, true>,  mppi_mlp_rollout_kernel<3, false, 2, true>, mppi_mlp_rollout_kernel<5, false, 2, true>};
#else
static const MlpKernel mlp_kernels[6] = {
    mppi_mlp_rollout_kernel<3, false, 1>, mppi_mlp_rollout_kernel<5, false, 1>, mppi_mlp_rollout_kernel<3, true, 1>,
    mppi_mlp_rollout_kernel<5, true, 1>,  mppi_mlp_rollout_kernel<3, false, 2>, mppi_mlp_rollout_kernel<5, false, 2>};
static MlpKernel mlp_kernel(int variant, bool traj) { return traj ? mlp_traj_kernels[variant] : mlp_kernels[variant]; }

struct MlpState {
    int K = 0, T = 0, n_sm = 148;
    mlp_op_t *d_w2 = nullptr;             // n_gemm x [512 out][512 in] fp16, K-major B operand (layers stacked along the rows)
    float4 *d_w01 = nullptr, *d_w3 = nullptr;
    float2 *d_w01u = nullptr;             // control columns of the folded first layer (n_in = 5)
    float *d_b3 = nullptr;
    __half *d_b1 = nullptr;               // layer-1 MMA B operand: [512 hidden, tile order][16 | 32] split-fp16 weight slots
    float *d_bh = nullptr;                // n_hidden = 3: bias of the layer the first GEMM evaluates
    float *d_hand = nullptr;              // balanced schedule: state records of split quads [cluster][rank][slot][6][128]
    unsigned int *d_hand_flag = nullptr;  // [cluster][rank]: epoch of the launch that published the record; then one fault word
    int max_clusters[12] = {};            // co-resident 2-CTA clusters per instantiation (cudaOccupancyMaxActiveClusters), TRAJ at 6..11
    unsigned int epoch = 0;
    int n_in = 3, n_gemm = 1;
    CUtensorMap w2_map;
    CUtensorMap w2_map_half;              // 64-row boxes: each CTA's half of a W2 box under pair MMAs
    bool ready = false;
};

MlpState *mlp_create(int K, int T) {
    MlpState *m = new (std::nothrow) MlpState();
    if (!m) return nullptr;
    m->K = K; m->T = T;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&m->n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (cudaMalloc(&m->d_w2, sizeof(mlp_op_t) * 2 * HID * HID) != cudaSuccess ||
        cudaMalloc(&m->d_bh, sizeof(float) * HID) != cudaSuccess ||
        cudaMalloc(&m->d_hand, sizeof(float) * ((size_t)(m->n_sm / 2 + 1) * 2 * 2 * 6 * TILE_M + 64)) != cudaSuccess ||
        cudaMemset(m->d_hand + (size_t)(m->n_sm / 2 + 1) * 2 * 2 * 6 * TILE_M, 0xA5, sizeof(float) * 64) != cudaSuccess ||
        cudaMalloc(&m->d_hand_flag, sizeof(unsigned int) * ((size_t)(m->n_sm / 2 + 1) * 2 + 1)) != cudaSuccess ||
        cudaMemset(m->d_hand_flag, 0, sizeof(unsigned int) * ((size_t)(m->n_sm / 2 + 1) * 2 + 1)) != cudaSuccess ||
        cudaMalloc(&m->d_w01, sizeof(float4) * HID) != cudaSuccess ||
        cudaMalloc(&m->d_w3, sizeof(float4) * HID) != cudaSuccess ||
        cudaMalloc(&m->d_w01u, sizeof(float2) * HID) != cudaSuccess ||
        cudaMalloc(&m->d_b3, sizeof(float) * 4) != cudaSuccess ||
        cudaMalloc(&m->d_b1, (size_t)B1TC_BYTES) != cudaSuccess) { mlp_destroy(m); return nullptr; }
    for (int v = 0; v < 12; ++v)
        if (cudaFuncSetAttribute(mlp_kernel(v % 6, v >= 6), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MLP_DYN_SMEM) != cudaSuccess) {
            mlp_destroy(m); return nullptr;
        }
    return m;
}

void mlp_destroy(MlpState *m) {
    if (!m) return;
    cudaFree(m->d_w2); cudaFree(m->d_bh); cudaFree(m->d_hand); cudaFree(m->d_hand_flag); cudaFree(m->d_w01); cudaFree(m->d_w01u); cudaFree(m->d_w3); cudaFree(m->d_b3); cudaFree(m->d_b1);
    delete m;
}

// Weights arrive as nn.Linear tensors [out][in] (dnn/simple_mlp.py:10-13; 5-input variant
// simulation/bullet_differential_drive_dnn.py:41-48).  Layer 0 has no activation, so it is folded into layer 1 here
// (FP64 accumulation): W01 = W1 W0, b01 = W1 b0 + b1.  StandardScaler pre/post-processing of the trained models,
// in = (raw - in_mean) / in_scale and out_raw = out * out_scale + out_mean (train/train_diff_mlp.py:72-103,
// test/test_diff_dyna_eval.py:54-56), is folded into W0 / b0 and W3 / b3 first; null pointers mean identity.
// n_hidden = 2: W / b hold 4 layers (one GEMM per step); n_hidden = 3 (train/train_diff_mlp.py:13-36): 5 layers, the two
// inner 512x512 layers are the two GEMMs, the first one still folds the input layer.
cudaError_t mlp_set_weights(MlpState *m, int n_in, int n_hidden, const float *const *W, const float *const *b, const double *in_mean,
                            const double *in_scale, const double *out_mean, const double *out_scale, cudaStream_t st) {
    if ((n_in != 3 && n_in != 5) || (n_hidden != 2 && n_hidden != 3)) return cudaErrorInvalidValue;
    const int n_gemm = n_hidden - 1, l_last = n_hidden, l_out = n_hidden + 1;     // last tanh layer, output layer
    std::vector<double> W0((size_t)HID * n_in), b0(HID);
    for (int i = 0; i < HID; ++i) {
        double bb = b[0][i];
        for (int c = 0; c < n_in; ++c) {
            const double sc = in_scale ? in_scale[c] : 1.0, mu = in_mean ? in_mean[c] : 0.0;
            const double w = (double)W[0][(size_t)i * n_in + c] / sc;
            W0[(size_t)i * n_in + c] = w;
            bb -= w * mu;
        }
        b0[i] = bb;
    }
    std::vector<float4> w01(HID), w3(HID);
    std::vector<float2> w01u(HID, make_float2(0.f, 0.f));
    std::vector<__half> b1((size_t)B1TC_BYTES / 2, __float2half_rn(0.f));
    for (int j = 0; j < HID; ++j) {
        double s[5] = {0, 0, 0, 0, 0}, bb = b[1][j];
        for (int i = 0; i < HID; ++i) {
            const double w1 = W[1][(size_t)j * HID + i];
            for (int c = 0; c < n_in; ++c) s[c] += w1 * W0[(size_t)i * n_in + c];
            bb += w1 * b0[i];
        }
        w01[j] = make_float4((float)s[0], (float)s[1], (float)s[2], (float)bb);
        w01u[j] = make_float2((float)s[3], (float)s[4]);
        {   // the same folded row as the tcgen05 layer 1's B operand: per input (w_hi, w_lo, w_hi) against the input row's
            // (x_hi, x_hi, x_lo), then (b_hi, b_lo) against (1, 1)
            const int KS = n_in == 3 ? 16 : 32;
            const int part = j / N_MMA;
            __half slot[L1_KS_MAX];
            for (int i = 0; i < L1_KS_MAX; ++i) slot[i] = __float2half_rn(0.f);
            auto split = [](double w, __half &hi, __half &lo) {
                hi = __float2half_rn((float)w);
                lo = __float2half_rn((float)(w - (double)__half2float(hi)));
            };
            for (int c = 0; c < n_in; ++c) {
                if (!(std::fabs(s[c]) <= 65504.0)) return cudaErrorInvalidValue;
                __half hi, lo;
                split(s[c], hi, lo);
                slot[3 * c] = hi; slot[3 * c + 1] = lo; slot[3 * c + 2] = hi;
            }
            if (!(std::fabs(bb) <= 65504.0)) return cudaErrorInvalidValue;
            split(bb, slot[3 * n_in], slot[3 * n_in + 1]);
            // plain unit order, K-major 32B-swizzled rows of 16 halves (unit r of a part at (r / 8) * 256 B + (r % 8) * 32 B,
            // 16-byte chunk c at position c ^ ((r / 4) % 2)), parts 4 KB apart, the second K block (halves 16..31) 16 KB behind the first
            const int r = j % N_MMA;
            __half *row = &b1[((size_t)part * N_MMA * 32 + (size_t)(r >> 3) * 256 + (size_t)(r & 7) * 32) / 2];
            for (int i = 0; i < KS; ++i) row[(size_t)(i >> 4) * (B1TC_KB_BYTES / 2) + (((((i >> 3) & 1) ^ ((r >> 2) & 1))) << 3) + (i & 7)] = slot[i];
        }
        const double o0 = out_scale ? out_scale[0] : 1.0, o1 = out_scale ? out_scale[1] : 1.0, o2 = out_scale ? out_scale[2] : 1.0;
        w3[j] = make_float4(b[l_last][j], (float)(W[l_out][0 * HID + j] * o0), (float)(W[l_out][1 * HID + j] * o1), (float)(W[l_out][2 * HID + j] * o2));
    }
    std::vector<mlp_op_t> w2((size_t)n_gemm * HID * HID);
    for (int g = 0; g < n_gemm; ++g)
        for (size_t i = 0; i < (size_t)HID * HID; ++i) {
            const float w = W[2 + g][i];
            if (!(std::fabs(w) <= 65504.f)) return cudaErrorInvalidValue;      // outside half precision's range (or NaN)
            w2[(size_t)g * HID * HID + i] = __float2half_rn(w);
        }
    float b3[4] = {0.f, 0.f, 0.f, 0.f};
    for (int c = 0; c < 3; ++c) b3[c] = (float)((double)b[l_out][c] * (out_scale ? out_scale[c] : 1.0) + (out_mean ? out_mean[c] : 0.0));
    cudaError_t e;
    if ((e = cudaMemcpyAsync(m->d_w01, w01.data(), sizeof(float4) * HID, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(m->d_w3, w3.data(), sizeof(float4) * HID, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(m->d_w01u, w01u.data(), sizeof(float2) * HID, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(m->d_b3, b3, sizeof(b3), cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(m->d_b1, b1.data(), sizeof(__half) * b1.size(), cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(m->d_w2, w2.data(), sizeof(mlp_op_t) * w2.size(), cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if (n_gemm == 2 && (e = cudaMemcpyAsync(m->d_bh, b[2], sizeof(float) * HID, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    // TMA descriptor of W2: inner dim = K (512 fp16, contiguous), outer dim = N (512 rows); 64 x 256 boxes, 128B swizzle
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if ((e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres)) != cudaSuccess) return e;
    if (!fn || qres != cudaDriverEntryPointSuccess) return cudaErrorNotSupported;
    const cuuint64_t dims[2] = {HID, (cuuint64_t)n_gemm * HID};
    const cuuint64_t strides[1] = {HID * sizeof(mlp_op_t)};
    const cuuint32_t box[2] = {KCH, N_MMA};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = ((PFN_encodeTiled)fn)(&m->w2_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, m->d_w2, dims, strides, box, estr,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    const cuuint32_t box_half[2] = {KCH, N_MMA / 2};
    r = ((PFN_encodeTiled)fn)(&m->w2_map_half, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, m->d_w2, dims, strides, box_half, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    m->n_in = n_in;
    m->n_gemm = n_gemm;
    m->ready = true;
    return cudaSuccess;
}

// Co-resident 2-CTA clusters of one instantiation on an otherwise idle device.  The balanced schedule makes a cluster
// wait for a record its neighbour publishes inside the same launch, so every cluster of the grid has to be resident.
template <typename Kern>
static int mlp_max_active_clusters(Kern kern, int n_sm) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n_sm & ~1), 1, 1);
    cfg.blockDim = dim3(MLP_THREADS, 1, 1);
    cfg.dynamicSmemBytes = MLP_DYN_SMEM;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// One rollout launch over a.K rows: costs into `out` (K), with `traj` followed by the states after every step (K, T, 3).
static int mlp_launch(MlpState *m, const TickArgs &a, bool traj, float *out, unsigned int *fault, cudaStream_t st) {
    const int n_tiles = (a.K + TILE_M - 1) / TILE_M;
    int grid = std::min(((n_tiles + 1) / 2) * 2, m->n_sm & ~1);       // whole clusters of 2
    // two tiles per CTA in flight (ping-pong) whenever a CTA owns more than one tile
    const bool pp = n_tiles > grid && m->n_gemm == 1;
    const int variant = (m->n_gemm == 2 ? 4 : (pp ? 2 : 0)) + (m->n_in == 5 ? 1 : 0), slot = (traj ? 6 : 0) + variant;
    // never launch more clusters than the device keeps resident at once (fused-off SMs, MPS partitions): the grid is
    // persistent, so a smaller one only means more tiles per cluster
    if (m->max_clusters[slot] == 0) {
        const int n = mlp_max_active_clusters(mlp_kernel(variant, traj), m->n_sm);
        m->max_clusters[slot] = n > 0 ? n : -1;                       // -1: the query failed, keep the SM-count grid
    }
    if (m->max_clusters[slot] > 0) grid = std::min(grid, 2 * m->max_clusters[slot]);
    // balanced (horizon-split) walk when whole quads do not divide over the clusters and every cluster still gets more
    // than one horizon of steps; MPPI_MLP_BALANCED=0 forces whole quads (A/B measurements)
    const char *bal_env = std::getenv("MPPI_MLP_BALANCED");               // read per launch: tests flip it in-process
    const bool allow_bal = !(bal_env && bal_env[0] == '0');
    const bool one_tile_bal = !pp && m->n_gemm == 2 && n_tiles > grid;     // three-layer residuals: pairs x timesteps
    const int n_quads = pp ? (n_tiles + 3) / 4 : (n_tiles + 1) / 2, n_clusters = grid / 2;
    const int balanced = ((pp || one_tile_bal) && allow_bal && n_clusters > 0 && (n_quads % n_clusters) != 0 &&
                          (long long)n_quads * a.T / n_clusters >= a.T + 2) ? 1 : 0;
    const unsigned int epoch = ++m->epoch;
    mlp_kernel(variant, traj)<<<grid, MLP_THREADS, MLP_DYN_SMEM, st>>>(a, mlp_use_cg2(m->n_in, pp, m->n_gemm) ? m->w2_map_half : m->w2_map,
                                                                       m->d_w01, m->d_w01u, m->d_w3, m->d_b3, m->d_bh, out, n_tiles, m->d_hand,
                                                                       m->d_hand_flag, fault, epoch, balanced, m->d_b1);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int mlp_rollout_costs(MlpState *m, const TickArgs &args, bool sum, const float *d_eps, float *d_S, cudaStream_t st) {
    if (!m || !m->ready) return -2;
    TickArgs a = args;
    a.eps = d_eps;
    a.flags = sum ? F_COST_SUM : 0;
    return mlp_launch(m, a, false, d_S, m->d_hand_flag + (size_t)(m->n_sm / 2 + 1) * 2, st);
}

int mlp_rollout_states(MlpState *m, const TickArgs &args, const float *d_ctl, float *d_out, unsigned int *d_fault, cudaStream_t st) {
    if (!m || !m->ready) return -2;
    TickArgs a = args;
    a.eps = d_ctl;
    a.n_exploit = 0; a.k_offset = 0;
    a.flags = 0;
    return mlp_launch(m, a, true, d_out, d_fault, st);
}

int mlp_check_guards(MlpState *m) {
    if (!m || !m->d_hand) return 0;
    unsigned char g[256];
    if (cudaMemcpy(g, m->d_hand + (size_t)(m->n_sm / 2 + 1) * 2 * 2 * 6 * TILE_M, 256, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    for (int i = 0; i < 256; ++i) if (g[i] != 0xA5) return 1;
    return 0;
}

bool mlp_take_fault(MlpState *m, cudaStream_t st) {
    if (!m || !m->d_hand_flag) return false;
    unsigned int *fault = m->d_hand_flag + (size_t)(m->n_sm / 2 + 1) * 2, v = 0;
    if (cudaMemcpyAsync(&v, fault, sizeof(v), cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) return false;
    if (v) cudaMemsetAsync(fault, 0, sizeof(v), st);
    return v != 0;
}
#endif  // MPPI_MLP_TRAJ_UNIT
