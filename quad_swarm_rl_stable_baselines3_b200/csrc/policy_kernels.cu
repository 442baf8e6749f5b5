// policy_kernels.cu -- fused two-tower policy forward for the quadrotor-swarm rollouts on sm_100a (SURVEY.md 8 f1).
//
// What it replaces: the per-step forward of the reference's `ActorCriticPolicyCustomSeparateWeights`
// (swarm_rl/models/ActorCriticPolicyCustom.py:284-556) with one `QuadMultiEncoder` per tower
// (swarm_rl/models/quad_multi_model.py:250-354): self-observation MLP S -> 256 -> 256 (tanh), deep-sets neighbour encoder
// phi(nbr_j) = W -> 256 -> 256 (tanh) averaged over the V visible neighbours (quad_multi_model.py:23-41), feed-forward
// 512 -> 512 (tanh), then the action-mean head (512 -> A) of the actor tower and the value head (512 -> 1) of the critic tower.
// This is the one dense contraction of the system: ~3.06 MFLOP per drone row, 1.6 TFLOP per 65536 x 8 step.
//
// Design (persistent, one CTA per SM, 128-row tiles, 10 warps with fixed roles):
//   * warps 0-7  EPILOGUE: thread = (row, column half).  tcgen05.ld the fp32 accumulator, + bias, tanh (MUFU), then either pack to bf16
//                and tcgen05.st it into the TMEM region the next layer's MMA reads as its A operand, or add it to the running sum
//                over neighbours (128 fp32 registers per thread), or fold it into the heads (CUDA-core FMAs);
//   * warp 8     MMA ISSUER (one lane): `tcgen05.mma.cta_group::1.kind::f16` (bf16 x bf16 -> fp32), M = 128, N = 128 per instruction
//                group; first layers read A from shared memory (the 128 x 32 observation tile), every other layer reads A from
//                TENSOR MEMORY -- activations never touch shared or global memory;
//   * warp 9     WEIGHT PRODUCER (one lane): `cp.async.bulk` + mbarrier complete_tx.  The neighbour encoder's weights (144 KB, used
//                V times per tile) are loaded once per tower and stay resident in shared memory; the self-encoder and feed-forward
//                weights (656 KB per tile) stream from L2 through a 3-stage ring of 16 KB chunk images.
//   TMEM map (512 columns): two "streams", each an accumulator of 128 fp32 columns + an activation region of 128 columns (256 bf16).
//   The V neighbour passes alternate between the streams, so that the tensor core works on one neighbour's next half-layer while the
//   epilogue warps run tanh over the other's -- the pass is bound by the epilogue (MUFU: 16 tanh/clk/SM, TMEM read: 64 B/clk/SM;
//   both 2048 clk per 128 x 256 layer, the MMA 2048 clk as well), not by their sum.  Feed-forward: four N = 128 quarters ping-pong
//   between the two accumulators; A = [self-encoder output | neighbour mean] in the two activation regions.
//   Weight images are pre-packed on the device (qp_set_weights) into the canonical no-swizzle K-major core-matrix layout (8 rows x 16
//   bytes), in the order the kernel consumes them.  The first layers share one 128 x 32 observation tile per stream, K laid out
//   [self (24) | neighbour (8)]: the self encoder's image has zeros in the neighbour slots and the neighbour encoder's in the self slots,
//   so the self part is written once per tile and each neighbour pass rewrites one 16-byte chunk per row.
//   Obstacle encoder (the OB instantiation, qp_config.obst_dim > 0; quad_multi_model.py's obstacle MLP, O -> 256 -> 256): runs after the self
//   encoder on stream 1's x tile, whose self slots then hold the O obstacle columns; the feed-forward (K = 768) has one accumulator, ACC0.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "../../include/quadpolicy.h"

namespace qp {

constexpr int H = 256;                      // hidden width of every encoder layer
constexpr int FF = 512;                     // feed-forward width
constexpr int TILE_M = 128;
constexpr int NH = 128;                     // N of one MMA group (half an encoder layer, a quarter of the feed-forward)
constexpr int CHUNK = 16 * 1024;            // one (N = 128) x (K = 64) bf16 weight image
constexpr int CHUNK1 = 8 * 1024;            // one (N = 128) x (K = 32) image (first layers)
constexpr int STAGGER_CLK = 0;                // start offset between neighbouring blocks (tuning knob QP_STAGGER; measured: no gain, see below)
constexpr int STAGES = 12;                  // ring slots of one 16 KB chunk: 9 hold the neighbour encoder during its passes, all 12 stream otherwise
constexpr int MAX_ACT = 8;
constexpr int SELF_PAD = 24, NBR_PAD = 8;   // K layout of the first layers: [self | neighbour]
constexpr int EPI_WARPS = 8, EPI_THREADS = 32 * EPI_WARPS, THREADS = EPI_THREADS + 128;   // + one warpgroup: MMA issuer, producer, 2 idle warps (setmaxnreg acts on warpgroups)
constexpr int RES_BYTES = 2 * CHUNK1 + 8 * CHUNK;                    // neighbour-encoder weights: 147456 = 9 chunks
constexpr int RES_CHUNKS = RES_BYTES / CHUNK;
constexpr int STREAM_BYTES = 2 * CHUNK1 + 8 * CHUNK + 32 * CHUNK;    // streamed per tile: self L1, self L2, feed-forward
constexpr int STREAM_CHUNKS = STREAM_BYTES / CHUNK;                  // 41
// obstacle encoder (compile-time variant): its inputs take the self slots of stream 1's x tile, so O <= SELF_PAD; streamed per tile on top:
// obstacle L1, obstacle L2, the feed-forward's third K block (4 quarters x 4 chunks)
constexpr int MAX_OBST = SELF_PAD;
constexpr int OBST_BYTES = 2 * CHUNK1 + 8 * CHUNK + 16 * CHUNK;
constexpr int OBST_CHUNKS = OBST_BYTES / CHUNK;                      // 25
constexpr size_t tower_img_bytes(int obst_dim) { return (size_t)(RES_BYTES + STREAM_BYTES + (obst_dim > 0 ? OBST_BYTES : 0)); }   // 819200 / 1228800

// fp32 side parameters of one tower
struct TowerParams {
    float bias[4 * H + FF];                 // b_self1, b_self2, b_nbr1, b_nbr2, b_ff
    float head_wt[FF * MAX_ACT];            // [512][8]: transposed nn.Linear.weight, zero-padded
    float head_b[MAX_ACT];
    float obst_bias[2 * H];                 // b_obst1, b_obst2 (read through L1: shared memory has no room left)
};
constexpr int B_SELF1 = 0, B_SELF2 = H, B_NBR1 = 2 * H, B_NBR2 = 3 * H, B_FF = 4 * H, N_BIAS = 4 * H + FF;

struct Args {
    const float *obs; int n, stride, S, W, V, A;
    const uint8_t *wimg[2];                 // per tower: [resident block | streamed block]
    const TowerParams *params[2];
    float *mean, *value;                    // [n, A], [n]
    int stagger;                            // clocks between the start of neighbouring blocks (0 = off)
    long long *trace;                       // debug (qp_debug_trace): clock64 stamps of block 0's second tile, tower 0; null = off
};
// arguments of the obstacle variant: a type of its own, so that the plain kernel's parameter block (copied to its stack) stays as it is
struct ArgsOb : Args {
    int O;                                  // obstacle columns, at S + V * W
};
template <bool OB> using KernelArgs = typename std::conditional<OB, ArgsOb, Args>::type;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier / bulk copy ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
// Bounded wait: a protocol error (a commit or a copy that never arrives) traps after ~2 s instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    const uint32_t addr = smem_u32(bar);
    long long t0 = 0;
    for (uint32_t spin = 0;; ++spin) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
        if ((spin & 1023u) == 1023u) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) __trap();
        }
    }
}
// hot-path form: one probe first (the common case on the issuer's ring: the chunk landed long ago), then the bounded loop
__device__ __forceinline__ void mbar_wait_fast(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (!done) mbar_wait(bar, parity);
}
__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 ---------------------------------------------------------------------------------------------------------
// exactly one lane of a converged warp (the compiler then moves MMA operands to uniform registers without a waterfall loop)
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T, M = 128, N = 128, K = 16, bf16 x bf16 -> fp32
__device__ __forceinline__ void mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T
__device__ __forceinline__ void mma_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major, no swizzle: core matrix = 8 rows x 16 bytes (128 B contiguous); LBO = distance between the two K-halves of one MMA,
// SBO = distance between 8-row groups (cute/atom/mma_traits_sm100.hpp, "LayoutType::INTERLEAVE ((8,n),2):((1,SBO),LBO)")
__device__ __forceinline__ void commit_one(uint64_t *bar) { if (elect_one()) tc_commit(bar); __syncwarp(); }
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;                                              // descriptor version (Blackwell)
    return d;                                                            // base offset 0, layout type 0 (no swizzle)
}
// descriptor without the start address (added as (addr >> 4): shared-memory addresses are below 2^18, the field holds 14 bits)
__host__ __device__ constexpr uint64_t desc_hi(uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
constexpr uint64_t DESC_W64 = desc_hi(128u, 1024u);      // weight chunk, K = 64 per row group
constexpr uint64_t DESC_W32 = desc_hi(128u, 512u);       // weight chunk, K = 32
constexpr uint64_t DESC_X = desc_hi(2048u, 128u);        // x tile

constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NH >> 3) << 17) | ((128u >> 4) << 24);   // F32 acc, bf16 x bf16, K-major, N 128, M 128

// The issuing thread is one lane: every instruction it spends per MMA is serial latency in front of the tensor pipe.  These groups are
// fully unrolled, descriptors advance by an immediate (K = 16 -> 256 B -> +16 in the address field).
// one (N = 128) x (K = 64) weight chunk against 32 TMEM columns of A
template <bool FIRST>
__device__ __noinline__ void issue_chunk_ts(uint32_t acc, uint32_t a_col, uint32_t w_addr)
{
    const uint64_t bd = DESC_W64 | (uint64_t)(w_addr >> 4);
    if (elect_one()) {
        mma_ts(acc, a_col, bd, IDESC, FIRST ? 0u : 1u);
        mma_ts(acc, a_col + 8u, bd + 16u, IDESC, 1u);
        mma_ts(acc, a_col + 16u, bd + 32u, IDESC, 1u);
        mma_ts(acc, a_col + 24u, bd + 48u, IDESC, 1u);
    }
    __syncwarp();
}
// first layers: the 128 x 32 x tile (shared memory) against an (N = 128) x (K = 32) image
__device__ __noinline__ void issue_l1_ss(uint32_t acc, uint32_t x_addr, uint32_t w_addr)
{
    const uint64_t ad = DESC_X | (uint64_t)(x_addr >> 4), bd = DESC_W32 | (uint64_t)(w_addr >> 4);
    if (elect_one()) {
        mma_ss(acc, ad, bd, IDESC, 0u);
        mma_ss(acc, ad + 256u, bd + 16u, IDESC, 1u);       // next K-half of the x tile: 2 chunks of 2048 B
    }
    __syncwarp();
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t *v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t *v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t *v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
                 "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
                 "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
                 : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t *v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float tanh_fast(float x)
{
#ifdef QP_NO_TANH
    return x * 0.25f;                                                    // profiling aid: how long is an epilogue item without the MUFU work?
#else
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#endif
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));      // upper half <- first source
    return r;
}


// shared-memory map (226.1 KB)
struct Smem {
    uint8_t ring[STAGES][CHUNK];           // weight chunks in stream order; the neighbour encoder's 9 stay pinned during its passes
    uint8_t xbuf[2][TILE_M * 32 * 2];      // per stream: the 128 x 32 bf16 first-layer input, K-chunk-major core matrices
    float bias[N_BIAS];
    float xchg[TILE_M][MAX_ACT];           // head partial sums of the upper column half
    float4 headw[FF];                      // head weights of outputs 0..3, transposed (outputs 4..7 are read through L1)
    uint64_t full[STAGES], empty[STAGES], acc_full[2], epi_done[2], x_ready, mean_ready;
    uint32_t tmem_base;
};

static_assert(sizeof(Smem) <= 232448, "shared-memory map exceeds the 227 KB a block can opt into");

// element (row, k) of an x tile: K-chunk (8 elements, 16 B) major, then 8-row groups of 128 B: LBO = 2048, SBO = 128
__device__ __forceinline__ uint32_t xoff(int row, int kchunk) { return (uint32_t)(kchunk * 2048 + (row >> 3) * 128 + (row & 7) * 16); }

// OB: with the obstacle encoder (a compile-time variant, so that the plain kernel keeps its register allocation and code layout)
template <bool OB>
__global__ void __launch_bounds__(THREADS, 1) policy_forward_kernel(const KernelArgs<OB> a)
{
    extern __shared__ __align__(128) uint8_t smem_raw[];
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    if (t == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&sm.acc_full[s], 1); mbar_init(&sm.epi_done[s], EPI_WARPS); }
        mbar_init(&sm.x_ready, EPI_WARPS);
        mbar_init(&sm.mean_ready, EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    for (int i = t; i < (int)sizeof(sm.xbuf) / 16; i += THREADS) reinterpret_cast<uint4 *>(sm.xbuf)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    // Optional start offset between blocks (off).  The feed-forward phase streams 512 KB per tile and runs at ~42 B/clk per SM (97 clk per MMA
    // instead of 64); de-phasing the blocks does not change that (QP_STAGGER = 7000 / 14000 / 28000: 2.00 / 2.10 / 2.48 ms vs 1.93 ms) and a
    // one-block grid streams at the same rate -- it is the per-SM L2 -> shared-memory rate, not contention.
    if (a.stagger > 0 && gridDim.x > 4 && (blockIdx.x & 3) != 0) {
        const long long until = clock64() + (long long)(blockIdx.x & 3) * a.stagger;
        while (clock64() < until) __nanosleep(256);
    }
    constexpr uint32_t ACC0 = 0, ACC1 = 128, R10 = 256, R11 = 384;      // TMEM columns: stream accumulators, stream activation regions
    // Feed-forward input [self | neighbour mean | obstacle]: R10 | R11 | -- without obstacles (the quarters ping-pong between ACC0 and ACC1);
    // R10 | ACC1 | R11 with them: the three 256-wide activations leave one accumulator, ACC0, for all four quarters
    constexpr uint32_t R_MEAN = OB ? ACC1 : R11;
    const int S = a.S, W = a.W, V = a.V, A = a.A;
    const int n_tiles = (a.n + TILE_M - 1) / TILE_M;
    // phase bookkeeping, advanced identically by every role: items issued per stream, tiles, ring chunks
    uint32_t n_it0 = 0u, n_it1 = 0u, n_tile = 0u, n_chunk = 0u;
#define N_ITEM(s) ((s) ? n_it1 : n_it0)
#define N_ITEM_INC(s) do { if (s) n_it1 += 1; else n_it0 += 1; } while (0)
    // every role runs its own loop over the two towers and meets the others at one block-wide barrier per tower (TOWER_SYNC): all chunks
    // consumed and all accumulators read, so the resident weights, the biases and the head weights may be replaced
#define TOWER_SYNC() do { tc_fence_before(); __syncthreads(); tc_fence_after(); } while (0)

    if (warp >= EPI_WARPS) {
        // the producer / issuer warpgroup gives its registers to the epilogue warps (which hold 128 running sums per thread)
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
        if (warp == 9) {
            for (int tower = 0; tower < 2; ++tower) {
                // the whole tower image, in consumption order, once per tile: [neighbour encoder (9 chunks, skipped without neighbours) |
                // self L1 | self L2 x 8 | (OB: obstacle L1 | obstacle L2 x 8) | feed-forward x 32 (OB: x 48)]
                if (lane == 0) {
                    const uint8_t *img = a.wimg[tower] + (V > 0 ? 0 : RES_BYTES);
                    const int n_loads = (V > 0 ? RES_CHUNKS : 0) + STREAM_CHUNKS + (OB ? OBST_CHUNKS : 0);
                    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                        for (int i = 0; i < n_loads; ++i) {
                            const uint32_t slot = n_chunk % STAGES;
                            mbar_wait(&sm.empty[slot], ((n_chunk / STAGES) & 1u) ^ 1u);      // the MMAs that read this slot have completed
                            mbar_expect_tx(&sm.full[slot], CHUNK);
                            bulk_load(sm.ring[slot], img + (size_t)i * CHUNK, CHUNK, &sm.full[slot]);
                            n_chunk += 1;
                        }
                    }
                }
                __syncwarp();
                TOWER_SYNC();
            }
        } else if (warp == 8) {
            for (int tower = 0; tower < 2; ++tower) {
                // =========================== MMA ISSUER ===========================
                {                                                            // the whole warp runs the role (uniform control flow and addresses); one elected lane issues
                    const uint32_t ring0 = smem_u32(sm.ring[0]), xb0 = smem_u32(sm.xbuf[0]), xb1 = smem_u32(sm.xbuf[1]);
                    bool tr = false;
                    int tm = 256;
                    auto wait_prev = [&](int s) {                            // the epilogue of the stream's previous item has drained its accumulator
                        if (N_ITEM(s) > 0) { mbar_wait(&sm.epi_done[s], (N_ITEM(s) - 1u) & 1u); tc_fence_after(); }
                        if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                    };
                    auto ring_take = [&]() -> uint32_t {                     // next streamed chunk has landed
                        const uint32_t slot = n_chunk % STAGES;
                        mbar_wait_fast(&sm.full[slot], (n_chunk / STAGES) & 1u);
                        tc_fence_after();
                        return slot;
                    };
                    auto ring_release = [&](uint32_t slot) { commit_one(&sm.empty[slot]); n_chunk += 1; };
                    // grouped form: take 4 chunks one by one, release them with 4 commits back to back (a commit between two MMA groups costs
                    // the tensor pipe ~180 clk; grouped, that is paid once per 16 MMAs)
                    uint32_t held[4];
                    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                        mbar_wait(&sm.x_ready, n_tile & 1u);
                        n_tile += 1;
                        tc_fence_after();
                        tr = a.trace != nullptr && tower == 0 && blockIdx.x == 0 && tile == (int)gridDim.x;
                        // ---- the neighbour encoder's 9 chunks have landed; they stay in their slots until the last neighbour MMA has been issued
                        const uint32_t nbr0 = n_chunk;
                        if (V > 0) {
                            for (uint32_t i = 0; i < (uint32_t)RES_CHUNKS; ++i) mbar_wait(&sm.full[(nbr0 + i) % STAGES], ((nbr0 + i) / STAGES) & 1u);
                            tc_fence_after();
                            n_chunk += RES_CHUNKS;
                        }
                        uint32_t nbr_w[RES_CHUNKS];                           // shared-memory addresses of the pinned chunks
#pragma unroll
                        for (uint32_t i = 0; i < (uint32_t)RES_CHUNKS; ++i) nbr_w[i] = ring0 + ((nbr0 + i) % STAGES) * (uint32_t)CHUNK;
                        // ---- neighbour passes, two at a time on the two streams
                        for (int j0 = 0; j0 < V; j0 += 2) {
                            const int nact = (V - j0) < 2 ? (V - j0) : 2;
                            for (int it = 0; it < 4; ++it)
                                for (int s = 0; s < nact; ++s) {
                                    const uint32_t acc = tmem + (s ? ACC1 : ACC0);
                                    const int h = it & 1;
                                    wait_prev(s);
                                    if (it < 2) {                            // layer 1: A = the stream's x tile (shared memory), K = 32
                                        issue_l1_ss(acc, s ? xb1 : xb0, nbr_w[0] + (uint32_t)h * CHUNK1);
                                    } else {                                 // layer 2: A = the stream's hidden activations (tensor memory), K = 256
                                        const uint32_t r1 = tmem + (s ? R11 : R10);
                                        const uint32_t *w = nbr_w + 1 + h * 4;
                                        issue_chunk_ts<true>(acc, r1, w[0]);
                                        issue_chunk_ts<false>(acc, r1 + 32u, w[1]);
                                        issue_chunk_ts<false>(acc, r1 + 64u, w[2]);
                                        issue_chunk_ts<false>(acc, r1 + 96u, w[3]);
                                    }
                                    commit_one(&sm.acc_full[s]);
                                    N_ITEM_INC(s);
                                    if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                                }
                        }
                        if (V > 0)
                            for (uint32_t i = 0; i < (uint32_t)RES_CHUNKS; ++i) commit_one(&sm.empty[(nbr0 + i) % STAGES]);      // free once those MMAs complete
                        // ---- self encoder layer 1: halves on the two accumulators, A = x tile of stream 0 (its neighbour chunk meets zero weights)
                        {
                            const uint32_t slot = ring_take();
                            for (int s = 0; s < 2; ++s) {
                                wait_prev(s);
                                issue_l1_ss(tmem + (s ? ACC1 : ACC0), xb0, ring0 + slot * (uint32_t)CHUNK + (uint32_t)s * CHUNK1);
                                commit_one(&sm.acc_full[s]);
                                N_ITEM_INC(s);
                                if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                            }
                            ring_release(slot);
                        }
                        // ---- self encoder layer 2: A = R11 (hidden, written by both layer-1 epilogues), output goes to R10 -- no in-place hazard,
                        //      so the epilogue of half 0 runs under the MMA of half 1
                        wait_prev(0);
                        wait_prev(1);
                        for (int s = 0; s < 2; ++s) {
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const uint32_t slot = ring_take();
                                if (c == 0) issue_chunk_ts<true>(tmem + (s ? ACC1 : ACC0), tmem + R11, ring0 + slot * (uint32_t)CHUNK);
                                else issue_chunk_ts<false>(tmem + (s ? ACC1 : ACC0), tmem + R11 + (uint32_t)c * 32u, ring0 + slot * (uint32_t)CHUNK);
                                held[c] = slot;
                                n_chunk += 1;
                            }
#pragma unroll
                            for (int c = 0; c < 4; ++c) commit_one(&sm.empty[held[c]]);
                            commit_one(&sm.acc_full[s]);
                            N_ITEM_INC(s);
                            if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                        }
                        if constexpr (OB) {
                            // ---- obstacle encoder layer 1: halves on the two accumulators, A = x tile of stream 1 (the obstacle inputs sit in its self
                            //      slots; the neighbour images have zeros there, this image zeros in the neighbour slots)
                            {
                                const uint32_t slot = ring_take();
                                for (int s = 0; s < 2; ++s) {
                                    wait_prev(s);
                                    issue_l1_ss(tmem + (s ? ACC1 : ACC0), xb1, ring0 + slot * (uint32_t)CHUNK + (uint32_t)s * CHUNK1);
                                    commit_one(&sm.acc_full[s]);
                                    N_ITEM_INC(s);
                                    if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                                }
                                ring_release(slot);
                            }
                            // ---- obstacle encoder layer 2: A = R11 (hidden), output back into R11 -- the epilogue writes it once BOTH halves have
                            //      completed (in-place: every MMA of this layer reads all of R11)
                            wait_prev(0);
                            wait_prev(1);
                            for (int s = 0; s < 2; ++s) {
#pragma unroll
                                for (int c = 0; c < 4; ++c) {
                                    const uint32_t slot = ring_take();
                                    if (c == 0) issue_chunk_ts<true>(tmem + (s ? ACC1 : ACC0), tmem + R11, ring0 + slot * (uint32_t)CHUNK);
                                    else issue_chunk_ts<false>(tmem + (s ? ACC1 : ACC0), tmem + R11 + (uint32_t)c * 32u, ring0 + slot * (uint32_t)CHUNK);
                                    held[c] = slot;
                                    n_chunk += 1;
                                }
#pragma unroll
                                for (int c = 0; c < 4; ++c) commit_one(&sm.empty[held[c]]);
                                commit_one(&sm.acc_full[s]);
                                N_ITEM_INC(s);
                                if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                            }
                        }
                        // ---- feed-forward: four quarters of 128 outputs, K = 512 (OB: 768): chunks 0-3 read R10 (self encoder), chunks 4-7 R_MEAN
                        //      (neighbour mean, written by the epilogue warps while the first half of quarter 0 runs), OB: chunks 8-11 R11 (obstacle)
                        constexpr int FF_CHUNKS = OB ? 12 : 8;
                        for (int qtr = 0; qtr < 4; ++qtr) {
                            const int s = OB ? 0 : (qtr & 1);
                            wait_prev(s);
                            if (qtr == 0) wait_prev(1);
#pragma unroll
                            for (int c = 0; c < FF_CHUNKS; ++c) {
                                const uint32_t slot = ring_take();
                                const uint32_t acol = tmem + (c < 4 ? R10 + (uint32_t)c * 32u : c < 8 ? R_MEAN + (uint32_t)(c - 4) * 32u : R11 + (uint32_t)(c - 8) * 32u);
                                if (c == 4 && qtr == 0) { mbar_wait(&sm.mean_ready, (n_tile - 1u) & 1u); tc_fence_after(); }
                                if (c == 0) issue_chunk_ts<true>(tmem + (s ? ACC1 : ACC0), acol, ring0 + slot * (uint32_t)CHUNK);
                                else issue_chunk_ts<false>(tmem + (s ? ACC1 : ACC0), acol, ring0 + slot * (uint32_t)CHUNK);
                                held[c & 3] = slot;
                                n_chunk += 1;
                                if ((c & 3) == 3) {
#pragma unroll
                                    for (int r = 0; r < 4; ++r) commit_one(&sm.empty[held[r]]);
                                }
                            }
                            commit_one(&sm.acc_full[s]);
                            N_ITEM_INC(s);
                            if (tr) { if (lane == 0) a.trace[tm] = clock64(); tm += 1; }
                        }
                    }
                }
                __syncwarp();
                TOWER_SYNC();
            }
        } else {
            for (int tower = 0; tower < 2; ++tower) TOWER_SYNC();
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
        for (int tower = 0; tower < 2; ++tower) {
            const TowerParams *P = a.params[tower];
            for (int i = t; i < N_BIAS; i += EPI_THREADS) sm.bias[i] = P->bias[i];
            for (int i = t; i < FF; i += EPI_THREADS) sm.headw[i] = *reinterpret_cast<const float4 *>(P->head_wt + (size_t)i * MAX_ACT);
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
            // =========================== EPILOGUE WARPS ===========================
            const int row_l = 32 * (warp & 3) + lane, q = warp >> 2;     // this thread: one row, one half (64) of an accumulator's 128 columns
            const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
            const int n_out = tower == 0 ? A : 1;
            float nsum[128];                                             // running sum over neighbours: [layer half][64 columns of this thread]
#pragma unroll
            for (int i = 0; i < 128; ++i) nsum[i] = 0.f;

            bool tr = false;                                             // this thread records the traced tile (qp_debug_trace)
            int te = 0;
            auto wait_acc = [&](int s) {
                mbar_wait(&sm.acc_full[s], N_ITEM(s) & 1u);
                tc_fence_after();
                if (tr) a.trace[te++] = clock64();
            };
            auto item_done = [&](int s) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.epi_done[s]);
                N_ITEM_INC(s);
                if (tr) a.trace[te++] = clock64();
            };
            // accumulator -> + bias -> tanh -> packed bf16 -> activation region `dst` (columns of layer half h, this thread's 64); `bias`: the
            // layer's 256 biases (shared memory, or global for the obstacle encoder)
            auto epi_to_tmem = [&](uint32_t acc, const float *bias, int h, uint32_t dst) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {                            // 16 columns at a time (register budget: the 128 running sums stay live)
                    uint32_t v[16], u[8];
                    tmem_ld16(lane_addr + acc + (uint32_t)(q * 64 + b * 16), v);
                    const float4 *bp = reinterpret_cast<const float4 *>(bias + h * 128 + q * 64 + b * 16);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 bb = bp[i];
                        u[2 * i] = pack_bf16(tanh_fast(__uint_as_float(v[4 * i]) + bb.x), tanh_fast(__uint_as_float(v[4 * i + 1]) + bb.y));
                        u[2 * i + 1] = pack_bf16(tanh_fast(__uint_as_float(v[4 * i + 2]) + bb.z), tanh_fast(__uint_as_float(v[4 * i + 3]) + bb.w));
                    }
                    tmem_st8(lane_addr + dst + (uint32_t)(h * 64 + q * 32 + b * 8), u);
                }
                tmem_st_wait();
            };

            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int row = tile * TILE_M + row_l;
                const bool live = row < a.n;
                tr = a.trace != nullptr && t == 0 && tower == 0 && blockIdx.x == 0 && tile == (int)gridDim.x;
                const float *orow = a.obs + (size_t)(live ? row : 0) * a.stride;
                // the 16-byte neighbour chunk (K 24..31) of neighbour j
                auto nbr_chunk = [&](int j) -> uint4 {
                    float f[NBR_PAD];
#pragma unroll
                    for (int i = 0; i < NBR_PAD; ++i) f[i] = (live && i < W) ? __ldg(orow + S + j * W + i) : 0.f;
                    return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
                };
                // ---- x tiles of the new tile: the previous tile's MMAs have all completed (its last accumulator was waited for)
                if (q == 0) {
#pragma unroll
                    for (int kc = 0; kc < 3; ++kc) {
                        float f[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) f[i] = (live && kc * 8 + i < S) ? __ldg(orow + kc * 8 + i) : 0.f;
                        const uint4 u = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
                        *reinterpret_cast<uint4 *>(sm.xbuf[0] + xoff(row_l, kc)) = u;
                        if constexpr (!OB) *reinterpret_cast<uint4 *>(sm.xbuf[1] + xoff(row_l, kc)) = u;
                    }
                } else {
                    if (V > 0) *reinterpret_cast<uint4 *>(sm.xbuf[0] + xoff(row_l, 3)) = nbr_chunk(0);
                    if (V > 1) *reinterpret_cast<uint4 *>(sm.xbuf[1] + xoff(row_l, 3)) = nbr_chunk(1);
                    if constexpr (OB) {                                  // the obstacle inputs (columns S + V W ..) in the self slots of stream 1's tile
                        const float *orow_o = orow + S + V * W;
#pragma unroll 1
                        for (int kc = 0; kc < 3; ++kc) {                 // one chunk at a time: 24 loads in flight beside the 128 running sums spill
                            float f[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) f[i] = (live && kc * 8 + i < a.O) ? __ldg(orow_o + kc * 8 + i) : 0.f;
                            *reinterpret_cast<uint4 *>(sm.xbuf[1] + xoff(row_l, kc)) =
                                make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
                        }
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.x_ready);

                // ---- neighbour passes
                for (int j0 = 0; j0 < V; j0 += 2) {
                    const int nact = (V - j0) < 2 ? (V - j0) : 2;
                    const float keep = j0 == 0 ? 0.f : 1.f;              // the first pair of passes starts the running sum
                    for (int s = 0; s < nact; ++s) { wait_acc(s); epi_to_tmem(s ? ACC1 : ACC0, sm.bias + B_NBR1, 0, s ? R11 : R10); item_done(s); }
                    for (int s = 0; s < nact; ++s) {
                        wait_acc(s);                                     // both layer-1 MMAs of this pass have read the x tile
                        if (q == s && j0 + s + 2 < V) {
                            *reinterpret_cast<uint4 *>(sm.xbuf[s] + xoff(row_l, 3)) = nbr_chunk(j0 + s + 2);
                            fence_proxy_async();
                        }
                        epi_to_tmem(s ? ACC1 : ACC0, sm.bias + B_NBR1, 1, s ? R11 : R10);
                        item_done(s);
                    }
#pragma unroll
                    for (int h = 0; h < 2; ++h)
                        for (int s = 0; s < nact; ++s) {
                            wait_acc(s);
                            const float kp = (s == 0) ? keep : 1.f;
#pragma unroll
                            for (int b = 0; b < 4; ++b) {                // 16 columns at a time: the 128 running sums leave few registers
                                uint32_t v[16];
                                tmem_ld16(lane_addr + (s ? ACC1 : ACC0) + (uint32_t)(q * 64 + b * 16), v);
                                const float4 *bp = reinterpret_cast<const float4 *>(sm.bias + B_NBR2 + h * 128 + q * 64 + b * 16);
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    const float4 bb = bp[i];
                                    float *ns = nsum + h * 64 + b * 16 + 4 * i;
                                    ns[0] = fmaf(ns[0], kp, tanh_fast(__uint_as_float(v[4 * i]) + bb.x));
                                    ns[1] = fmaf(ns[1], kp, tanh_fast(__uint_as_float(v[4 * i + 1]) + bb.y));
                                    ns[2] = fmaf(ns[2], kp, tanh_fast(__uint_as_float(v[4 * i + 2]) + bb.z));
                                    ns[3] = fmaf(ns[3], kp, tanh_fast(__uint_as_float(v[4 * i + 3]) + bb.w));
                                }
                            }
                            item_done(s);
                        }
                }
                // ---- self encoder layer 1 (halves on the two accumulators) -> hidden in R11 (stream 1's last MMAs have completed)
                for (int s = 0; s < 2; ++s) { wait_acc(s); epi_to_tmem(s ? ACC1 : ACC0, sm.bias + B_SELF1, s, R11); item_done(s); }
                // ---- self encoder layer 2 -> R10
                for (int s = 0; s < 2; ++s) { wait_acc(s); epi_to_tmem(s ? ACC1 : ACC0, sm.bias + B_SELF2, s, R10); item_done(s); }
                if constexpr (OB) {
                    // ---- obstacle encoder layer 1 -> hidden in R11 (the self encoder's layer-2 MMAs, R11's last readers, have completed)
                    for (int s = 0; s < 2; ++s) { wait_acc(s); epi_to_tmem(s ? ACC1 : ACC0, P->obst_bias, s, R11); item_done(s); }
                    // ---- obstacle encoder layer 2 -> R11 in place: both halves' MMAs must have completed before either half is written
                    wait_acc(0);
                    wait_acc(1);
                    for (int s = 0; s < 2; ++s) { epi_to_tmem(s ? ACC1 : ACC0, P->obst_bias + H, s, R11); item_done(s); }
                    // the neighbour mean goes to ACC1: every epilogue warp has finished reading it (a row's two column halves are in two warps)
                    tc_fence_before();
                    asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
                    tc_fence_after();
                }
                // ---- neighbour mean -> R_MEAN (no neighbours: zeros, like an absent encoder half).  Its last readers (R11: the self encoder's
                //      layer-2 MMAs; OB, ACC1: the epilogue above) are done; the feed-forward reads it from its 5th K chunk on
                {
                    const float inv = V > 0 ? 1.0f / (float)V : 0.f;
#pragma unroll
                    for (int h = 0; h < 2; ++h)
#pragma unroll
                        for (int b = 0; b < 2; ++b) {
                            uint32_t u[16];
#pragma unroll
                            for (int i = 0; i < 16; ++i) u[i] = pack_bf16(nsum[h * 64 + b * 32 + 2 * i] * inv, nsum[h * 64 + b * 32 + 2 * i + 1] * inv);
                            tmem_st16(lane_addr + R_MEAN + (uint32_t)(h * 64 + q * 32 + b * 16), u);
                        }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sm.mean_ready);
                }
                // ---- feed-forward quarters with the head folded in
                float head[MAX_ACT];
#pragma unroll
                for (int o = 0; o < MAX_ACT; ++o) head[o] = 0.f;
                for (int qtr = 0; qtr < 4; ++qtr) {
                    const int s = OB ? 0 : (qtr & 1);
                    wait_acc(s);
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        uint32_t v[32];
                        tmem_ld32(lane_addr + (s ? ACC1 : ACC0) + (uint32_t)(q * 64 + b * 32), v);
                        const int c0 = qtr * 128 + q * 64 + b * 32;
                        const float4 *bp = reinterpret_cast<const float4 *>(sm.bias + B_FF + c0);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 bb = bp[i];
                            const float y[4] = { tanh_fast(__uint_as_float(v[4 * i]) + bb.x), tanh_fast(__uint_as_float(v[4 * i + 1]) + bb.y),
                                                 tanh_fast(__uint_as_float(v[4 * i + 2]) + bb.z), tanh_fast(__uint_as_float(v[4 * i + 3]) + bb.w) };
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const float4 w0 = sm.headw[c0 + 4 * i + e];
                                head[0] = fmaf(y[e], w0.x, head[0]); head[1] = fmaf(y[e], w0.y, head[1]);
                                head[2] = fmaf(y[e], w0.z, head[2]); head[3] = fmaf(y[e], w0.w, head[3]);
                            }
                            if (n_out > 4) {                             // wide action spaces: outputs 4..7 straight from L1
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const float4 w1 = __ldg(reinterpret_cast<const float4 *>(P->head_wt + (size_t)(c0 + 4 * i + e) * MAX_ACT) + 1);
                                    head[4] = fmaf(y[e], w1.x, head[4]); head[5] = fmaf(y[e], w1.y, head[5]);
                                    head[6] = fmaf(y[e], w1.z, head[6]); head[7] = fmaf(y[e], w1.w, head[7]);
                                }
                            }
                        }
                    }
                    item_done(s);
                }
                // ---- the two column halves of a row meet in shared memory; the lower half writes the outputs
                if (q == 1) {
#pragma unroll
                    for (int o = 0; o < MAX_ACT; ++o) sm.xchg[row_l][o] = head[o];
                }
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
                if (q == 0 && live) {
#pragma unroll
                    for (int o = 0; o < MAX_ACT; ++o)
                        if (o < n_out) {
                            const float r = head[o] + sm.xchg[row_l][o] + __ldg(P->head_b + o);
                            if (tower == 0) a.mean[(size_t)row * A + o] = r;
                            else a.value[row] = r;
                        }
                }
            }
            TOWER_SYNC();
        }
    }
#undef N_ITEM
#undef N_ITEM_INC
#undef TOWER_SYNC
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// ---- weight packing: nn.Linear weight [out, in] fp32 -> chunk images (bf16, canonical K-major core-matrix layout) ----------------
// image of rows n0 .. n0+127 and kc input slots of W: byte offset of element (n, k) = (n / 8) * SBO + (k / 8) * 128 + (n % 8) * 16 +
// (k % 8) * 2, SBO = (kc / 8) * 128.  Slot k reads input column k0 + k, or -- first layers, `split` > 0 -- column k for k < split and
// column len1 + (k - split) behind it (the [self | neighbour] K layout); columns beyond the matrix are zero.
__global__ void pack_chunk_kernel(const float *w, int out_dim, int in_dim, int n0, int k0, int kc, int split, int len1, uint8_t *img)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= NH * kc) return;
    const int n = idx / kc, k = idx % kc;
    const int gn = n0 + n;
    int gk = k0 + k;
    if (split > 0) gk = k < split ? (k < len1 ? k : -1) : len1 + (k - split);
    const float v = (gn < out_dim && gk >= 0 && gk < in_dim) ? w[(size_t)gn * in_dim + gk] : 0.f;
    const size_t off = (size_t)(n / 8) * ((size_t)(kc / 8) * 128) + (size_t)(k / 8) * 128 + (size_t)(n % 8) * 16 + (size_t)(k % 8) * 2;
    *reinterpret_cast<__nv_bfloat16 *>(img + off) = __float2bfloat16_rn(v);
}

// head weights [n_out, 512] -> transposed, zero-padded [512][8]
__global__ void pack_head_kernel(const float *w, int n_out, float *wt)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= FF * MAX_ACT) return;
    const int c = idx / MAX_ACT, o = idx % MAX_ACT;
    wt[idx] = o < n_out ? w[(size_t)o * FF + c] : 0.f;
}

// ---- generalised advantage estimation over a rollout (SB3 RolloutBuffer.compute_returns_and_advantage, buffers.py: the recursion
// last = delta_t + gamma * lambda * nonterminal_t * last, delta_t = r_t + gamma * V_{t+1} * nonterminal_t - V_t, backwards in time).
// One thread per agent row, [T, n] arrays row-major: every step's loads and stores are coalesced across the warp.
__global__ void gae_kernel(const float *rew, const float *val, const uint8_t *done, const float *last_val, int T, int n, float gamma, float lam,
                           float *adv, float *ret)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float next_v = last_val[i], last = 0.f;
    for (int t = T - 1; t >= 0; --t) {
        const size_t k = (size_t)t * n + i;
        const float nonterminal = done[k] ? 0.f : 1.f, v = val[k];
        const float delta = rew[k] + gamma * next_v * nonterminal - v;
        last = delta + gamma * lam * nonterminal * last;
        adv[k] = last;
        ret[k] = last + v;
        next_v = v;
    }
}

// ---- fused bias + tanh of a dense layer and its backward (the PPO update's elementwise work around the cuBLAS GEMMs) -------------------
// forward:  y = tanh(z + b)            z, y [n, h] (bf16 under autocast, else fp32), b [h] fp32
// backward: gz = gy * (1 - y^2),  gb[c] += sum_rows gz[., c]   -- one pass instead of tanh_backward + a separate column reduction
// (eager autograd: 27 % of the update's device time, profiles/r2_ppo_update_kernels.md).  Block = h / 2 threads, one column pair per thread,
// grid-stride over rows: every row is one contiguous, coalesced segment.
template <typename T> struct Pair;
template <> struct Pair<float> {
    static __device__ __forceinline__ float2 ld(const float *p) { return *reinterpret_cast<const float2 *>(p); }
    static __device__ __forceinline__ void st(float *p, float2 v) { *reinterpret_cast<float2 *>(p) = v; }
};
template <> struct Pair<__nv_bfloat16> {
    static __device__ __forceinline__ float2 ld(const __nv_bfloat16 *p) { return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(p)); }
    static __device__ __forceinline__ void st(__nv_bfloat16 *p, float2 v) { *reinterpret_cast<__nv_bfloat162 *>(p) = __float22bfloat162_rn(v); }
};
template <typename T>
__global__ void bias_tanh_kernel(const T *z, const float *b, int n, int h, T *y)
{
    const int c = 2 * threadIdx.x;
    if (c >= h) return;
    const float b0 = b[c], b1 = b[c + 1];
    for (int r = blockIdx.x; r < n; r += gridDim.x) {
        const float2 v = Pair<T>::ld(z + (size_t)r * h + c);
        Pair<T>::st(y + (size_t)r * h + c, make_float2(tanhf(v.x + b0), tanhf(v.y + b1)));
    }
}
template <typename T>
__global__ void bias_tanh_bwd_kernel(const T *gy, const T *y, int n, int h, T *gz, float *gb)
{
    const int c = 2 * threadIdx.x;
    if (c >= h) return;
    float a0 = 0.f, a1 = 0.f;
    for (int r = blockIdx.x; r < n; r += gridDim.x) {
        const float2 g = Pair<T>::ld(gy + (size_t)r * h + c), t = Pair<T>::ld(y + (size_t)r * h + c);
        const float2 o = make_float2(g.x * (1.f - t.x * t.x), g.y * (1.f - t.y * t.y));
        Pair<T>::st(gz + (size_t)r * h + c, o);
        a0 += o.x; a1 += o.y;
    }
    atomicAdd(gb + c, a0);
    atomicAdd(gb + c + 1, a1);
}

// 16-byte form (h % 8 == 0): a thread owns 8 adjacent columns, the block's threads form (h / 8 column groups) x (RL row lanes); two rows per
// lane are in flight per trip.  Column sums: registers -> shared memory across the row lanes -> one atomicAdd per column and block.
template <typename T> struct Vec8;
template <> struct Vec8<float> {
    static __device__ __forceinline__ void ld(const float *p, float *v)
    {
        const float4 a = *reinterpret_cast<const float4 *>(p), b = *reinterpret_cast<const float4 *>(p + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    static __device__ __forceinline__ void st(float *p, const float *v)
    {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
};
template <> struct Vec8<__nv_bfloat16> {
    static __device__ __forceinline__ void ld(const __nv_bfloat16 *p, float *v)
    {
        const uint4 u = *reinterpret_cast<const uint4 *>(p);
        const uint32_t w[4] = { u.x, u.y, u.z, u.w };
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u); }
    }
    static __device__ __forceinline__ void st(__nv_bfloat16 *p, const float *v)
    {
        uint4 u;
        u.x = pack_bf16(v[0], v[1]); u.y = pack_bf16(v[2], v[3]); u.z = pack_bf16(v[4], v[5]); u.w = pack_bf16(v[6], v[7]);
        *reinterpret_cast<uint4 *>(p) = u;
    }
};
template <typename T>
__global__ void __launch_bounds__(256) bias_tanh_v8_kernel(const T *z, const float *b, int n, int h, int RL, T *y)
{
    const int G = h >> 3, cg = threadIdx.x % G, rl = threadIdx.x / G;
    float bb[8];
    Vec8<float>::ld(b + 8 * cg, bb);
    for (int r = blockIdx.x * RL + rl; r < n; r += gridDim.x * RL) {
        float v[8];
        Vec8<T>::ld(z + (size_t)r * h + 8 * cg, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = tanhf(v[i] + bb[i]);
        Vec8<T>::st(y + (size_t)r * h + 8 * cg, v);
    }
}
template <typename T>
__global__ void __launch_bounds__(256) bias_tanh_bwd_v8_kernel(const T *gy, const T *y, int n, int h, int RL, T *gz, float *gb)
{
    __shared__ float red[256 * 8];
    const int G = h >> 3, cg = threadIdx.x % G, rl = threadIdx.x / G;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    const int stride = gridDim.x * RL;
    int r = blockIdx.x * RL + rl;
    for (; r + stride < n; r += 2 * stride) {                           // two rows in flight
        float g0[8], t0[8], g1[8], t1[8];
        Vec8<T>::ld(gy + (size_t)r * h + 8 * cg, g0); Vec8<T>::ld(y + (size_t)r * h + 8 * cg, t0);
        Vec8<T>::ld(gy + (size_t)(r + stride) * h + 8 * cg, g1); Vec8<T>::ld(y + (size_t)(r + stride) * h + 8 * cg, t1);
#pragma unroll
        for (int i = 0; i < 8; ++i) { g0[i] *= 1.f - t0[i] * t0[i]; g1[i] *= 1.f - t1[i] * t1[i]; acc[i] += g0[i] + g1[i]; }
        Vec8<T>::st(gz + (size_t)r * h + 8 * cg, g0); Vec8<T>::st(gz + (size_t)(r + stride) * h + 8 * cg, g1);
    }
    if (r < n) {
        float g0[8], t0[8];
        Vec8<T>::ld(gy + (size_t)r * h + 8 * cg, g0); Vec8<T>::ld(y + (size_t)r * h + 8 * cg, t0);
#pragma unroll
        for (int i = 0; i < 8; ++i) { g0[i] *= 1.f - t0[i] * t0[i]; acc[i] += g0[i]; }
        Vec8<T>::st(gz + (size_t)r * h + 8 * cg, g0);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = acc[i];
    __syncthreads();
    if (rl == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float sum = 0.f;
            for (int k = 0; k < RL; ++k) sum += red[(k * G + cg) * 8 + i];
            atomicAdd(gb + 8 * cg + i, sum);
        }
    }
}

// backward of a FIRST dense tanh layer with few inputs (the deep-sets phi: 6 -> 256 over n * V rows): the input needs no gradient, so grad_z is
// never written; the pass produces grad_bias [h] and grad_weight [h, IN] = grad_z^T x directly (cuBLAS runs this 256 x 6 output, K = 393216
// reduction on an sm80 kernel without split-K: 185 us; here it rides on the one read of grad_y and y).  x is fp32 [rows, IN], IN <= 8.  Two rows per
// thread in flight; every block writes its partial sums to `part[block][(IN + 1) * h]` (no atomics), a second small kernel adds the blocks up.
template <typename T, int IN>
__global__ void __launch_bounds__(256) bias_tanh_bwd_w_kernel(const T *gy, const T *y, const float *x, int n, int h, int RL, float *part)
{
    __shared__ float red[256 * 8];
    const int G = h >> 3, cg = threadIdx.x % G, rl = threadIdx.x / G;
    float ab[8], aw[8][IN];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        ab[i] = 0.f;
#pragma unroll
        for (int k = 0; k < IN; ++k) aw[i][k] = 0.f;
    }
    const int stride = gridDim.x * RL;
    int r = blockIdx.x * RL + rl;
    for (; r + stride < n; r += 2 * stride) {
        float g0[8], t0[8], g1[8], t1[8], x0[IN], x1[IN];
        Vec8<T>::ld(gy + (size_t)r * h + 8 * cg, g0); Vec8<T>::ld(y + (size_t)r * h + 8 * cg, t0);
        Vec8<T>::ld(gy + (size_t)(r + stride) * h + 8 * cg, g1); Vec8<T>::ld(y + (size_t)(r + stride) * h + 8 * cg, t1);
#pragma unroll
        for (int k = 0; k < IN; ++k) { x0[k] = __ldg(x + (size_t)r * IN + k); x1[k] = __ldg(x + (size_t)(r + stride) * IN + k); }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float o0 = g0[i] * (1.f - t0[i] * t0[i]), o1 = g1[i] * (1.f - t1[i] * t1[i]);
            ab[i] += o0 + o1;
#pragma unroll
            for (int k = 0; k < IN; ++k) aw[i][k] = fmaf(o1, x1[k], fmaf(o0, x0[k], aw[i][k]));
        }
    }
    if (r < n) {
        float g0[8], t0[8], x0[IN];
        Vec8<T>::ld(gy + (size_t)r * h + 8 * cg, g0); Vec8<T>::ld(y + (size_t)r * h + 8 * cg, t0);
#pragma unroll
        for (int k = 0; k < IN; ++k) x0[k] = __ldg(x + (size_t)r * IN + k);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float o0 = g0[i] * (1.f - t0[i] * t0[i]);
            ab[i] += o0;
#pragma unroll
            for (int k = 0; k < IN; ++k) aw[i][k] = fmaf(o0, x0[k], aw[i][k]);
        }
    }
    float *mine = part + (size_t)blockIdx.x * (size_t)(IN + 1) * h;      // [k][column], k = IN: the bias
#pragma unroll
    for (int k = 0; k <= IN; ++k) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = (k < IN) ? aw[i][k < IN ? k : 0] : ab[i];
        __syncthreads();
        if (rl == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float sum = 0.f;
                for (int q = 0; q < RL; ++q) sum += red[(q * G + cg) * 8 + i];
                mine[(size_t)k * h + 8 * cg + i] = sum;
            }
        }
    }
}
// part [blocks][(in + 1) * h] -> gw [h, in] (nn.Linear layout), gb [h]
__global__ void bias_tanh_bwd_w_reduce_kernel(const float *part, int blocks, int h, int in_dim, float *gb, float *gw)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x, total = (in_dim + 1) * h;
    if (e >= total) return;
    float sum = 0.f;
    for (int b = 0; b < blocks; ++b) sum += part[(size_t)b * total + e];
    const int k = e / h, c = e - k * h;
    if (k < in_dim) gw[(size_t)c * in_dim + k] = sum;
    else gb[c] = sum;
}

// deep-sets tail (quad_multi_model.py:35-40): y = tanh(z + b) on [n * V, h] rows and m = mean over the V rows of each group, in one pass; the
// backward takes the gradient of m ([n, h]) and produces grad_z = gm[group] / V * (1 - y^2) and the bias gradient without ever materialising the
// expanded gradient (eager autograd: a [n * V, h] division kernel + tanh_backward + a column reduction).  Thread = (group, 8 columns).
template <typename T>
__global__ void __launch_bounds__(256) bias_tanh_mean_kernel(const T *z, const float *b, int n, int V, int h, int RL, T *y, T *m)
{
    const int G = h >> 3, cg = threadIdx.x % G, rl = threadIdx.x / G;
    float bb[8];
    Vec8<float>::ld(b + 8 * cg, bb);
    const float inv = 1.0f / (float)V;
    for (int g = blockIdx.x * RL + rl; g < n; g += gridDim.x * RL) {
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
        for (int j = 0; j < V; ++j) {
            const size_t off = ((size_t)g * V + j) * h + 8 * cg;
            float v[8];
            Vec8<T>::ld(z + off, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = tanhf(v[i] + bb[i]);
            Vec8<T>::st(y + off, v);
            Vec8<T>::ld(y + off, v);                                    // the mean is taken over the values as stored (bf16-rounded), like torch's
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += v[i];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] *= inv;
        Vec8<T>::st(m + (size_t)g * h + 8 * cg, acc);
    }
}
template <typename T>
__global__ void __launch_bounds__(256) bias_tanh_mean_bwd_kernel(const T *gm, const T *y, int n, int V, int h, int RL, T *gz, float *gb)
{
    __shared__ float red[256 * 8];
    const int G = h >> 3, cg = threadIdx.x % G, rl = threadIdx.x / G;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    const float inv = 1.0f / (float)V;
    for (int g = blockIdx.x * RL + rl; g < n; g += gridDim.x * RL) {
        float gv[8];
        Vec8<T>::ld(gm + (size_t)g * h + 8 * cg, gv);
#pragma unroll
        for (int i = 0; i < 8; ++i) gv[i] *= inv;
        for (int j = 0; j < V; ++j) {
            const size_t off = ((size_t)g * V + j) * h + 8 * cg;
            float t[8], o[8];
            Vec8<T>::ld(y + off, t);
#pragma unroll
            for (int i = 0; i < 8; ++i) { o[i] = gv[i] * (1.f - t[i] * t[i]); acc[i] += o[i]; }
            Vec8<T>::st(gz + off, o);
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = acc[i];
    __syncthreads();
    if (rl == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float sum = 0.f;
            for (int k = 0; k < RL; ++k) sum += red[(k * G + cg) * 8 + i];
            atomicAdd(gb + 8 * cg + i, sum);
        }
    }
}

}  // namespace qp

using namespace qp;

template <typename T>
static void launch_bwd_w(int in_dim, int grid, int threads, cudaStream_t s, const T *gy, const T *y, const float *x, int n, int h, int RL, float *part)
{
    switch (in_dim) {
    case 1: bias_tanh_bwd_w_kernel<T, 1><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    case 2: bias_tanh_bwd_w_kernel<T, 2><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    case 3: bias_tanh_bwd_w_kernel<T, 3><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    case 4: bias_tanh_bwd_w_kernel<T, 4><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    case 5: bias_tanh_bwd_w_kernel<T, 5><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    case 6: bias_tanh_bwd_w_kernel<T, 6><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    case 7: bias_tanh_bwd_w_kernel<T, 7><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    default: bias_tanh_bwd_w_kernel<T, 8><<<grid, threads, 0, s>>>(gy, y, x, n, h, RL, part); break;
    }
}

struct qp_policy {
    qp_config cfg;
    int device, sms;
    uint8_t *wimg[2];
    TowerParams *params[2];
    long long launches;
    long long *trace;
    int max_grid;           // tuning knob QP_MAX_GRID (0 = one block per SM)
    int stagger;            // tuning knob QP_STAGGER (clocks; default STAGGER_CLK)
    std::string err;
};

static thread_local std::string g_qp_err;
static int qp_fail(qp_policy *p, int code, const std::string &m) { if (p) p->err = m; else g_qp_err = m; return code; }
#define QP_CUDA(p, call)                                                                                          \
    do {                                                                                                          \
        cudaError_t _r = (call);                                                                                  \
        if (_r != cudaSuccess) return qp_fail(p, QP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_r)); \
    } while (0)

extern "C" {

const char *qp_last_error(const qp_policy *p) { return p ? p->err.c_str() : g_qp_err.c_str(); }
size_t qp_config_size(void) { return sizeof(qp_config); }

int qp_create(const qp_config *cfg, int device, qp_policy **out)
{
    if (!cfg || !out) return qp_fail(nullptr, QP_ERR_NULL, "qp_create: null argument");
    *out = nullptr;
    if (cfg->api_version != 1 && cfg->api_version != QP_API_VERSION) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_create: api_version mismatch");
    qp_config c;                                                         // a version-1 struct ends before obst_dim
    memset(&c, 0, sizeof(c));
    memcpy(&c, cfg, cfg->api_version == 1 ? offsetof(qp_config, obst_dim) : sizeof(qp_config));
    if (c.hidden != H) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_create: only hidden = 256 is built");
    if (c.self_dim < 1 || c.self_dim > SELF_PAD || c.nbr_dim < 0 || c.nbr_dim > NBR_PAD || c.num_nbr < 0)
        return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_create: self_dim must be in [1, 24], nbr_dim in [0, 8]");
    if (c.act_dim < 1 || c.act_dim > MAX_ACT) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_create: act_dim out of [1, 8]");
    if (c.obst_dim < 0 || c.obst_dim > MAX_OBST) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_create: obst_dim out of [0, 24]");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return qp_fail(nullptr, QP_ERR_CUDA, "qp_create: no such CUDA device");
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    qp_policy *p = new qp_policy();
    p->cfg = c; p->device = device; p->launches = 0; p->trace = nullptr; p->max_grid = 0;
    if (const char *g = getenv("QP_MAX_GRID")) p->max_grid = atoi(g);
    p->stagger = STAGGER_CLK;
    if (const char *g = getenv("QP_STAGGER")) p->stagger = atoi(g);
    p->wimg[0] = p->wimg[1] = nullptr; p->params[0] = p->params[1] = nullptr;
    cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, device);
    cudaError_t r = cudaSuccess;
    const size_t img_bytes = tower_img_bytes(c.obst_dim);
    for (int t = 0; t < 2 && r == cudaSuccess; ++t) {
        r = cudaMalloc(&p->wimg[t], img_bytes);
        if (r == cudaSuccess) r = cudaMemset(p->wimg[t], 0, img_bytes);
        if (r == cudaSuccess) r = cudaMalloc(&p->params[t], sizeof(TowerParams));
        if (r == cudaSuccess) r = cudaMemset(p->params[t], 0, sizeof(TowerParams));
    }
    if (r == cudaSuccess)
        r = c.obst_dim > 0 ? cudaFuncSetAttribute(policy_forward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem))
                           : cudaFuncSetAttribute(policy_forward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    cudaSetDevice(prev);
    if (r != cudaSuccess) {
        for (int t = 0; t < 2; ++t) { cudaFree(p->wimg[t]); cudaFree(p->params[t]); }
        delete p;
        return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_create: ") + cudaGetErrorString(r));
    }
    *out = p;
    return QP_OK;
}

int qp_destroy(qp_policy *p)
{
    if (!p) return QP_ERR_NULL;
    for (int t = 0; t < 2; ++t) { cudaFree(p->wimg[t]); cudaFree(p->params[t]); }
    delete p;
    return QP_OK;
}

int64_t qp_launch_count(const qp_policy *p) { return p ? p->launches : 0; }

/* profiling aid, not part of quadpolicy.h: `buf` = 512 int64 on the device (or null to switch off); the next forwards write clock64
 * stamps of block 0's second tile (actor tower): [0, 256) epilogue warp 0 (accumulator ready / item done), [256, 512) the MMA issuer */
int qp_debug_trace(qp_policy *p, long long *buf) { if (!p) return QP_ERR_NULL; p->trace = buf; return QP_OK; }

int qp_set_weights(qp_policy *p, int tower, const qp_tower_weights *w, void *stream)
{
    if (!p || !w) return qp_fail(p, QP_ERR_NULL, "qp_set_weights: null argument");
    if (tower < 0 || tower > 1) return qp_fail(p, QP_ERR_BAD_CONFIG, "qp_set_weights: tower must be 0 (actor) or 1 (critic)");
    const int S = p->cfg.self_dim, O = p->cfg.obst_dim;
    if (O > 0 && (!w->obst_w1 || !w->obst_b1 || !w->obst_w2 || !w->obst_b2))       // a handle without obstacles never reads these fields
        return qp_fail(p, QP_ERR_NULL, "qp_set_weights: null obstacle-encoder pointer (obst_dim > 0)");
    cudaStream_t s = (cudaStream_t)stream;
    const int n_out = tower == 0 ? p->cfg.act_dim : 1;
    uint8_t *img = p->wimg[tower];
    // one (N = 128) x kc image
    auto pack = [&](const float *src, int out_dim, int in_dim, int n0, int k0, int kc, int split, int len1, uint8_t *dst) {
        pack_chunk_kernel<<<(NH * kc + 255) / 256, 256, 0, s>>>(src, out_dim, in_dim, n0, k0, kc, split, len1, dst);
    };
    // resident block: neighbour L1 halves, neighbour L2 (half, K chunk)
    if (p->cfg.num_nbr > 0) {
        // phi reads the neighbour row alone: its W inputs sit in K slots 24..31 (the x tile's neighbour chunk), the self slots meet zeros
        for (int h = 0; h < 2; ++h) pack(w->nbr_w1, H, p->cfg.nbr_dim, NH * h, 0, 32, SELF_PAD, 0, img + (size_t)h * CHUNK1);
        for (int h = 0; h < 2; ++h)
            for (int c = 0; c < 4; ++c) pack(w->nbr_w2, H, H, NH * h, 64 * c, 64, 0, 0, img + 2 * CHUNK1 + (size_t)(h * 4 + c) * CHUNK);
    }
    // streamed block, in consumption order: self L1 halves, self L2 (half, chunk), [obstacle L1 halves, obstacle L2 (half, chunk),]
    // feed-forward (quarter, chunk)
    uint8_t *st = img + RES_BYTES;
    auto pack_encoder = [&](const float *w1, int in_dim, const float *w2) {
        // layer 1 reads K slots 0 .. in_dim - 1 of its x tile; the neighbour slots (24..31) meet zeros
        for (int h = 0; h < 2; ++h) pack(w1, H, in_dim, NH * h, 0, 32, SELF_PAD, in_dim, st + (size_t)h * CHUNK1);
        st += 2 * CHUNK1;
        for (int h = 0; h < 2; ++h)
            for (int c = 0; c < 4; ++c) pack(w2, H, H, NH * h, 64 * c, 64, 0, 0, st + (size_t)(h * 4 + c) * CHUNK);
        st += 8 * CHUNK;
    };
    pack_encoder(w->self_w1, S, w->self_w2);
    if (O > 0) pack_encoder(w->obst_w1, O, w->obst_w2);
    const int ff_chunks = O > 0 ? 12 : 8, ff_in = 64 * ff_chunks;         // K = [self | neighbour (| obstacle)]
    for (int qtr = 0; qtr < 4; ++qtr)
        for (int c = 0; c < ff_chunks; ++c) pack(w->ff_w, FF, ff_in, NH * qtr, 64 * c, 64, 0, 0, st + (size_t)(qtr * ff_chunks + c) * CHUNK);
    TowerParams *P = p->params[tower];
    const cudaMemcpyKind dd = cudaMemcpyDeviceToDevice;
    QP_CUDA(p, cudaMemcpyAsync(P->bias + B_SELF1, w->self_b1, H * sizeof(float), dd, s));
    QP_CUDA(p, cudaMemcpyAsync(P->bias + B_SELF2, w->self_b2, H * sizeof(float), dd, s));
    if (p->cfg.num_nbr > 0) {
        QP_CUDA(p, cudaMemcpyAsync(P->bias + B_NBR1, w->nbr_b1, H * sizeof(float), dd, s));
        QP_CUDA(p, cudaMemcpyAsync(P->bias + B_NBR2, w->nbr_b2, H * sizeof(float), dd, s));
    }
    QP_CUDA(p, cudaMemcpyAsync(P->bias + B_FF, w->ff_b, FF * sizeof(float), dd, s));
    if (O > 0) {
        QP_CUDA(p, cudaMemcpyAsync(P->obst_bias, w->obst_b1, H * sizeof(float), dd, s));
        QP_CUDA(p, cudaMemcpyAsync(P->obst_bias + H, w->obst_b2, H * sizeof(float), dd, s));
    }
    pack_head_kernel<<<(FF * MAX_ACT + 255) / 256, 256, 0, s>>>(w->head_w, n_out, P->head_wt);
    QP_CUDA(p, cudaMemsetAsync(P->head_b, 0, sizeof(P->head_b), s));
    QP_CUDA(p, cudaMemcpyAsync(P->head_b, w->head_b, (size_t)n_out * sizeof(float), dd, s));
    QP_CUDA(p, cudaGetLastError());
    return QP_OK;
}

int qp_gae(const float *rewards, const float *values, const uint8_t *dones, const float *last_values, int T, int n, float gamma, float lam,
           float *advantages, float *returns, void *stream)
{
    if (!rewards || !values || !dones || !last_values || !advantages || !returns) return qp_fail(nullptr, QP_ERR_NULL, "qp_gae: null argument");
    if (T < 1 || n < 1) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_gae: bad T / n");
    gae_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, T, n, gamma, lam, advantages, returns);
    cudaError_t r = cudaGetLastError();
    if (r != cudaSuccess) return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_gae: ") + cudaGetErrorString(r));
    return QP_OK;
}

// the pair kernels (bias_tanh_kernel, bias_tanh_bwd_kernel) load and store float2 / __nv_bfloat162: every [n, h] operand must be aligned
// to one element pair, which "h even" alone does not give (a contiguous view at an odd element offset)
static bool pair_aligned(int is_bf16, size_t addr_bits) { return (addr_bits & (is_bf16 ? 3 : 7)) == 0; }

static int bias_tanh_grid(int n)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int g = sms * 8;
    return n < g ? n : g;
}

int qp_bias_tanh(const void *z, const float *bias, int n, int h, int is_bf16, void *y, void *stream)
{
    if (!z || !bias || !y) return qp_fail(nullptr, QP_ERR_NULL, "qp_bias_tanh: null argument");
    if (n < 1 || h < 2 || (h & 1) || h > 2048) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh: h must be even and <= 2048, n >= 1");
    if (!pair_aligned(is_bf16, (size_t)z | (size_t)y))
        return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh: pointers must be aligned to one element pair (8 bytes fp32, 4 bytes bf16)");
    cudaStream_t s = (cudaStream_t)stream;
    if ((h & 7) == 0 && (((size_t)z | (size_t)y | (size_t)bias) & 15) == 0) {
        const int G = h / 8, RL = G >= 256 ? 1 : 256 / G, rows = (n + RL - 1) / RL, grid = bias_tanh_grid(rows);
        if (is_bf16) bias_tanh_v8_kernel<<<grid, G * RL, 0, s>>>((const __nv_bfloat16 *)z, bias, n, h, RL, (__nv_bfloat16 *)y);
        else bias_tanh_v8_kernel<<<grid, G * RL, 0, s>>>((const float *)z, bias, n, h, RL, (float *)y);
    } else if (is_bf16) bias_tanh_kernel<<<bias_tanh_grid(n), h / 2, 0, s>>>((const __nv_bfloat16 *)z, bias, n, h, (__nv_bfloat16 *)y);
    else bias_tanh_kernel<<<bias_tanh_grid(n), h / 2, 0, s>>>((const float *)z, bias, n, h, (float *)y);
    cudaError_t r = cudaGetLastError();
    if (r != cudaSuccess) return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_bias_tanh: ") + cudaGetErrorString(r));
    return QP_OK;
}

int qp_bias_tanh_backward(const void *grad_y, const void *y, int n, int h, int is_bf16, void *grad_z, float *grad_bias, void *stream)
{
    if (!grad_y || !y || !grad_z || !grad_bias) return qp_fail(nullptr, QP_ERR_NULL, "qp_bias_tanh_backward: null argument");
    if (n < 1 || h < 2 || (h & 1) || h > 2048) return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh_backward: h must be even and <= 2048, n >= 1");
    if (!pair_aligned(is_bf16, (size_t)grad_y | (size_t)y | (size_t)grad_z))
        return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh_backward: pointers must be aligned to one element pair (8 bytes fp32, 4 bytes bf16)");
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t r = cudaMemsetAsync(grad_bias, 0, (size_t)h * sizeof(float), s);
    if (r == cudaSuccess) {
        if ((h & 7) == 0 && (((size_t)grad_y | (size_t)y | (size_t)grad_z) & 15) == 0) {
            const int G = h / 8, RL = G >= 256 ? 1 : 256 / G, rows = (n + RL - 1) / RL;
            int grid = bias_tanh_grid(rows);
            if (grid > 592) grid = 592;                                 // 4 blocks per SM: fewer, longer blocks = fewer atomics per column
            if (is_bf16) bias_tanh_bwd_v8_kernel<<<grid, G * RL, 0, s>>>((const __nv_bfloat16 *)grad_y, (const __nv_bfloat16 *)y, n, h, RL, (__nv_bfloat16 *)grad_z, grad_bias);
            else bias_tanh_bwd_v8_kernel<<<grid, G * RL, 0, s>>>((const float *)grad_y, (const float *)y, n, h, RL, (float *)grad_z, grad_bias);
        } else if (is_bf16) bias_tanh_bwd_kernel<<<bias_tanh_grid(n), h / 2, 0, s>>>((const __nv_bfloat16 *)grad_y, (const __nv_bfloat16 *)y, n, h, (__nv_bfloat16 *)grad_z, grad_bias);
        else bias_tanh_bwd_kernel<<<bias_tanh_grid(n), h / 2, 0, s>>>((const float *)grad_y, (const float *)y, n, h, (float *)grad_z, grad_bias);
        r = cudaGetLastError();
    }
    if (r != cudaSuccess) return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_bias_tanh_backward: ") + cudaGetErrorString(r));
    return QP_OK;
}

size_t qp_bias_tanh_backward_first_workspace(int h, int in_dim) { return (size_t)592 * (size_t)(in_dim + 1) * (size_t)h * sizeof(float); }

int qp_bias_tanh_backward_first(const void *grad_y, const void *y, const float *x, int n, int h, int in_dim, int is_bf16, void *workspace,
                                float *grad_bias, float *grad_weight, void *stream)
{
    if (!grad_y || !y || !x || !workspace || !grad_bias || !grad_weight) return qp_fail(nullptr, QP_ERR_NULL, "qp_bias_tanh_backward_first: null argument");
    if (n < 1 || h < 8 || (h & 7) || h > 2048 || in_dim < 1 || in_dim > 8 || ((((size_t)grad_y | (size_t)y) & 15) != 0))
        return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh_backward_first: h a multiple of 8 (<= 2048), 1 <= in_dim <= 8, pointers 16-byte aligned");
    const int G = h / 8, RL = G >= 256 ? 1 : 256 / G;
    int grid = bias_tanh_grid((n + RL - 1) / RL);
    if (grid > 592) grid = 592;
    cudaStream_t s = (cudaStream_t)stream;
    float *part = (float *)workspace;
    if (is_bf16) launch_bwd_w<__nv_bfloat16>(in_dim, grid, G * RL, s, (const __nv_bfloat16 *)grad_y, (const __nv_bfloat16 *)y, x, n, h, RL, part);
    else launch_bwd_w<float>(in_dim, grid, G * RL, s, (const float *)grad_y, (const float *)y, x, n, h, RL, part);
    const int total = (in_dim + 1) * h;
    bias_tanh_bwd_w_reduce_kernel<<<(total + 127) / 128, 128, 0, s>>>(part, grid, h, in_dim, grad_bias, grad_weight);
    cudaError_t r = cudaGetLastError();
    if (r != cudaSuccess) return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_bias_tanh_backward_first: ") + cudaGetErrorString(r));
    return QP_OK;
}

int qp_bias_tanh_mean(const void *z, const float *bias, int n, int V, int h, int is_bf16, void *y, void *mean, void *stream)
{
    if (!z || !bias || !y || !mean) return qp_fail(nullptr, QP_ERR_NULL, "qp_bias_tanh_mean: null argument");
    if (n < 1 || V < 1 || h < 8 || (h & 7) || h > 2048 || ((((size_t)z | (size_t)y | (size_t)mean | (size_t)bias) & 15) != 0))
        return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh_mean: n >= 1, V >= 1, h a multiple of 8 (<= 2048), pointers 16-byte aligned");
    const int G = h / 8, RL = G >= 256 ? 1 : 256 / G, grid = bias_tanh_grid((n + RL - 1) / RL);
    cudaStream_t s = (cudaStream_t)stream;
    if (is_bf16) bias_tanh_mean_kernel<<<grid, G * RL, 0, s>>>((const __nv_bfloat16 *)z, bias, n, V, h, RL, (__nv_bfloat16 *)y, (__nv_bfloat16 *)mean);
    else bias_tanh_mean_kernel<<<grid, G * RL, 0, s>>>((const float *)z, bias, n, V, h, RL, (float *)y, (float *)mean);
    cudaError_t r = cudaGetLastError();
    if (r != cudaSuccess) return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_bias_tanh_mean: ") + cudaGetErrorString(r));
    return QP_OK;
}

int qp_bias_tanh_mean_backward(const void *grad_mean, const void *y, int n, int V, int h, int is_bf16, void *grad_z, float *grad_bias, void *stream)
{
    if (!grad_mean || !y || !grad_z || !grad_bias) return qp_fail(nullptr, QP_ERR_NULL, "qp_bias_tanh_mean_backward: null argument");
    if (n < 1 || V < 1 || h < 8 || (h & 7) || h > 2048 || ((((size_t)grad_mean | (size_t)y | (size_t)grad_z) & 15) != 0))
        return qp_fail(nullptr, QP_ERR_BAD_CONFIG, "qp_bias_tanh_mean_backward: n >= 1, V >= 1, h a multiple of 8 (<= 2048), pointers 16-byte aligned");
    const int G = h / 8, RL = G >= 256 ? 1 : 256 / G;
    int grid = bias_tanh_grid((n + RL - 1) / RL);
    if (grid > 592) grid = 592;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t r = cudaMemsetAsync(grad_bias, 0, (size_t)h * sizeof(float), s);
    if (r == cudaSuccess) {
        if (is_bf16) bias_tanh_mean_bwd_kernel<<<grid, G * RL, 0, s>>>((const __nv_bfloat16 *)grad_mean, (const __nv_bfloat16 *)y, n, V, h, RL, (__nv_bfloat16 *)grad_z, grad_bias);
        else bias_tanh_mean_bwd_kernel<<<grid, G * RL, 0, s>>>((const float *)grad_mean, (const float *)y, n, V, h, RL, (float *)grad_z, grad_bias);
        r = cudaGetLastError();
    }
    if (r != cudaSuccess) return qp_fail(nullptr, QP_ERR_CUDA, std::string("qp_bias_tanh_mean_backward: ") + cudaGetErrorString(r));
    return QP_OK;
}

int qp_forward(qp_policy *p, const float *obs, int n, int obs_stride, float *mean, float *value, void *stream)
{
    if (!p || !obs || !mean || !value) return qp_fail(p, QP_ERR_NULL, "qp_forward: null argument");
    if (n < 1 || obs_stride < p->cfg.self_dim + p->cfg.nbr_dim * p->cfg.num_nbr + p->cfg.obst_dim)
        return qp_fail(p, QP_ERR_BAD_CONFIG, "qp_forward: bad n / obs_stride (obs_stride must be >= S + V * W + O)");
    ArgsOb a;
    a.obs = obs; a.n = n; a.stride = obs_stride; a.S = p->cfg.self_dim; a.W = p->cfg.nbr_dim; a.V = p->cfg.num_nbr; a.A = p->cfg.act_dim;
    for (int t = 0; t < 2; ++t) { a.wimg[t] = p->wimg[t]; a.params[t] = p->params[t]; }
    a.mean = mean; a.value = value; a.trace = p->trace; a.O = p->cfg.obst_dim;
    a.stagger = (n >= 8 * p->sms * TILE_M) ? p->stagger : 0;            // only worth it when every block has several tiles
    const int tiles = (n + TILE_M - 1) / TILE_M;
    int grid = tiles < p->sms ? tiles : p->sms;
    if (p->max_grid > 0 && grid > p->max_grid) grid = p->max_grid;
    if (a.O > 0) policy_forward_kernel<true><<<grid, THREADS, sizeof(Smem), (cudaStream_t)stream>>>(a);
    else policy_forward_kernel<false><<<grid, THREADS, sizeof(Smem), (cudaStream_t)stream>>>(static_cast<const Args &>(a));
    p->launches += 1;
    QP_CUDA(p, cudaGetLastError());
    return QP_OK;
}

}  // extern "C"
