// hlynr_policy.cu -- fused actor-critic forward on the tcgen05 tensor cores (C ABI: include/hlynr_policy.h).
//
// Network = the reference's policy (rl_system/scripts/train_flat_ppo.py:37-85 CustomMLP as SB3 features extractor, :419-429
// net_arch=[] so action_net / value_net sit directly on the 256 features):
//     x[in_dim] -> Linear 512 -> LayerNorm -> ReLU -> Linear 512 -> LayerNorm -> ReLU -> Linear 256 -> LayerNorm -> ReLU -> f[256]
//     (in_dim = 104 = 4 stacked 26-D frames by default; any width 1-256, e.g. 68 = 4 stacked 17-D frames)
//     mean = action_net(f) [6], V = value_net(f) [1], a = mean + exp(log_std) * eps, log pi(a)
//
// One persistent CTA per SM walks over 128-row tiles.  Per tile the activations never leave the SM:
//
//   warps 0-15 (512 threads)  load x (fp32 -> bf16) into the A-operand region of shared memory; after every GEMM read the fp32
//                             accumulators from TMEM (tcgen05.ld, thread = row), add the bias, LayerNorm + ReLU in fp32, and
//                             write the bf16 result back into the A region in the canonical 128B-swizzled K-major layout the
//                             next GEMM reads; after the head GEMM they add the head biases, sample the action and store
//   warp  16   (1 thread)     TMA producer: streams the weight tiles [256 rows x 64 K] bf16 (32 KiB, SWIZZLE_128B) of all four
//                             GEMMs through a 3-stage shared-memory ring (cp.async.bulk.tensor.2d, mbarrier complete_tx)
//   warp  17   (1 thread)     MMA issuer: tcgen05.mma.cta_group::1.kind::f16, M = 128, N = 256 (16 for the heads), K = 16 per
//                             instruction, fp32 accumulators in TMEM (512 columns); tcgen05.commit frees ring stages and
//                             signals "accumulators ready"
//
// Layers are serialised inside a tile by two mbarriers (a_ready: operand written + TMEM drained; acc_ready: GEMM complete);
// the weight ring runs ahead across layers and tiles, because weights do not depend on the activations.
#include <cstring>
#include <new>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/hlynr_policy.h"
#include "../../include/hlynr_rng.h"
#include "hlynr_host.cuh"

namespace {

constexpr int IN = HLYNR_POLICY_IN, H1 = HLYNR_POLICY_H1, H2 = HLYNR_POLICY_H2, H3 = HLYNR_POLICY_H3, ACT = HLYNR_POLICY_ACT;
constexpr int IN_PAD = 128;      // K of the first GEMM at in_dim = 104, padded to two 64-wide K blocks (zeros)
constexpr int HEAD_N = 16;       // action_net (6 rows) + value_net (1 row) + zero rows: the smallest UMMA N for M = 128
constexpr int BM = 128;          // rows per tile = UMMA M = TMEM lanes
constexpr int BK = 64;           // bf16 elements per K block: 128 bytes = one swizzle span
constexpr int BN = 256;          // weight rows per ring stage = UMMA N
constexpr int STAGES = 3;
constexpr int KBLOCK_BYTES = BM * BK * 2;            // 16 KiB: one K block of the A operand
constexpr int A_BYTES = BM * 512 * 2;                // 128 KiB: x (ceil(in_dim / 64) <= 4 K blocks), then H1 / H2 (8), then H3 (4)
constexpr int STAGE_BYTES = BN * BK * 2;             // 32 KiB
#ifndef HLYNR_POLICY_EPI_WARPS
#define HLYNR_POLICY_EPI_WARPS 16   /* measured on B200 at 131072 rows: 8 warps 219 us, 16 warps 203 us (profiles/r02_h_policy_epilogue_warps.log) */
#endif
constexpr int EPI_WARPS = HLYNR_POLICY_EPI_WARPS, EPI_THREADS = EPI_WARPS * 32;   // 8 or 16: PARTS warps share a TMEM lane quarter
constexpr int PARTS = EPI_WARPS / 4;                                              // ... and split the columns of a layer PARTS ways
static_assert(EPI_WARPS == 8 || EPI_WARPS == 16, "two or four column parts per lane quarter");
constexpr int THREADS = EPI_THREADS + 64;
constexpr int OFF_RING = A_BYTES;
constexpr int OFF_STATS = OFF_RING + STAGES * STAGE_BYTES;      // float2[2][128]
constexpr int OFF_BARS = OFF_STATS + 2 * BM * 8;                 // full[S], empty[S], a_ready, acc_ready
constexpr int OFF_TMEM = OFF_BARS + (2 * STAGES + 2) * 8;
constexpr int OFF_CTR = OFF_TMEM + 8;                            // this launch's call counter, read from the device (u64)
constexpr int SMEM_BYTES = OFF_TMEM + 16;
static_assert(SMEM_BYTES <= 232448, "shared memory budget of one CTA (227 KiB)");
constexpr uint32_t TMEM_COLS = 512;
constexpr int N_LAYERS = 4;      // three hidden GEMMs + the head GEMM

// kb0 = K blocks of the first GEMM, ceil(in_dim / 64)
__host__ __device__ constexpr int layer_kblocks(int l, int kb0) { return l == 0 ? kb0 : (l == 3 ? H3 / BK : 512 / BK); }
__host__ __device__ constexpr int layer_nchunks(int l) { return l < 2 ? 2 : 1; }
__host__ __device__ constexpr int layer_n(int l) { return l == 3 ? HEAD_N : BN; }
__host__ __device__ constexpr uint32_t layer_col(int l, int nc) { return l == 3 ? 256u : (uint32_t)(nc * BN); }   // TMEM column of the accumulator

// UMMA instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A / B bf16, both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t instr_desc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// Per-column vectors of the epilogues (biases, LayerNorm gamma / beta, head biases, log_std) live in one global array read with
// warp-uniform 128-bit loads (L1 hits).  Passing them by value as a 15 KiB kernel parameter (constant bank, indexed LDC.64) was
// measured SLOWER: 9.5 instead of 6.8 us per 512-wide epilogue.
constexpr int VEC_B1 = 0, VEC_G1 = 512, VEC_BE1 = 1024, VEC_B2 = 1536, VEC_G2 = 2048, VEC_BE2 = 2560, VEC_B3 = 3072, VEC_G3 = 3328,
              VEC_BE3 = 3584, VEC_BH = 3840, VEC_LS = 3856, VEC_TOTAL = 3864;

struct Params {
    const float* obs;       // [n_rows, in_dim]
    int in_dim, kb0;        // row width, K blocks of the first GEMM (ceil(in_dim / 64))
    int64_t n_rows;
    const int32_t* n_rows_dev;
    const float* vec;   // the per-column vectors, VEC_* offsets
    float* actions; float* values; float* logp; float* mean; float* actions_clipped;
    float ln_eps;
    uint32_t k0, k1;        // Philox key (seed)
    uint32_t ctr_lo, ctr_hi; // call counter
    int deterministic;
    int* error_flag;
    long long* timing;   // debug: SM-clock timestamps of the phases of CTA 0's tiles (NULL = off), [tile][16]
    int timing_tiles;
};

// ---- PTX wrappers -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// never hang the GPU: a lost arrival becomes a launch failure with a flag the host reports
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* error_flag, int code) {
    for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins)
        if (spins > (1u << 27)) { if (error_flag) atomicExch(error_flag, code); __trap(); }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// multicast variants (thread-block clusters): one L2 read of a weight slice lands in the shared memory of every CTA of the
// cluster (same offset), completing bytes on each CTA's own mbarrier; the commit arrives on the empty barrier of every CTA
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): K-major, SWIZZLE_128B (layout type 2), 8-row groups 1024 B
// apart (SBO), version 1 (Blackwell); the start address may be advanced by 32 B per UMMA_K = 16 slice inside the swizzle span
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void tmem_ld32(uint32_t addr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(addr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(addr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// wait + a data dependency on the loaded registers, so that no use of them can be scheduled above the wait
__device__ __forceinline__ void tmem_wait_ld32(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]),
                   "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]),
                   "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :: "memory");
}
__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :: "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
}
// byte offset of the 16-byte chunk holding columns [8*c, 8*c + 8) of row r in the K-major SWIZZLE_128B operand layout
__device__ __forceinline__ uint32_t a_chunk_offset(int r, int c) {
    return (uint32_t)((c >> 3) * KBLOCK_BYTES + (r >> 3) * 1024 + (r & 7) * 128 + (((c & 7) ^ (r & 7)) << 4));
}

__device__ __forceinline__ uint4 philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)HLYNR_PHILOX_M0 * c0, p1 = (uint64_t)HLYNR_PHILOX_M1 * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
        k0 += HLYNR_PHILOX_W0; k1 += HLYNR_PHILOX_W1;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ void box_muller(uint32_t xa, uint32_t xb, float* z0, float* z1) {
    const float r = sqrtf(-2.0f * logf((float)((xa >> 8) + 1u) * 5.9604644775390625e-8f));
    float s, c;
    sincospif(2.0f * ((float)(xb >> 8) * 5.9604644775390625e-8f), &s, &c);
    *z0 = r * c; *z1 = r * s;
}

// packed fp32 pairs (sm_100 FADD2 / FFMA2: two lanes of fp32 per instruction) and the fused ReLU + bf16x2 conversion
__device__ __forceinline__ uint64_t pk2(float lo, float hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ uint64_t pk2u(uint32_t lo, uint32_t hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ uint32_t relu_bf16x2(uint64_t v) {   // {lo, hi} fp32 -> max(., 0) -> bf16x2 (lo in the low half)
    float lo, hi;
    upk2(v, lo, hi);
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// bias + LayerNorm + ReLU epilogue of one hidden layer: TMEM accumulators -> bf16 A operand of the next GEMM.
// Two warps share a row quarter: warp w and w + 4 read TMEM lanes 32 * (w % 4) ..., each over half of the N columns.
// The arithmetic runs on packed fp32 pairs (4 instead of 9.5 floating-point instructions per element over the two passes).
// one 32-column chunk of pass 1: x = v + b - k with k the part's shift {-k, -k} = nk2, accumulate the sum and the sum of squares
// (packed fp32 pairs).  The shift keeps the sums small when a row has a large common mean: E[x^2] - mean^2 in fp32 loses
// (mean / std)^2 * 2^-24 of the variance, 20 % at mean / std = 1000.
__device__ __forceinline__ void stats_chunk(const uint32_t (&v)[32], const float4 (&b)[8], uint64_t nk2, uint64_t& s2, uint64_t& ss2) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint64_t x0 = add2(add2(pk2u(v[4 * j], v[4 * j + 1]), pk2(b[j].x, b[j].y)), nk2);
        const uint64_t x1 = add2(add2(pk2u(v[4 * j + 2], v[4 * j + 3]), pk2(b[j].z, b[j].w)), nk2);
        s2 = add2(s2, add2(x0, x1));
        ss2 = fma2(x0, x0, fma2(x1, x1, ss2));
    }
}
__device__ __forceinline__ void stats_chunk16(const uint32_t (&v)[16], const float4 (&b)[4], uint64_t nk2, uint64_t& s2, uint64_t& ss2) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint64_t x0 = add2(add2(pk2u(v[4 * j], v[4 * j + 1]), pk2(b[j].x, b[j].y)), nk2);
        const uint64_t x1 = add2(add2(pk2u(v[4 * j + 2], v[4 * j + 3]), pk2(b[j].z, b[j].w)), nk2);
        s2 = add2(s2, add2(x0, x1));
        ss2 = fma2(x0, x0, fma2(x1, x1, ss2));
    }
}
// Chan's merge of two column parts of n columns each: (mean, M2 = sum of squared deviations from the mean).  Symmetric in a and b
// up to exact operations, so every thread that merges the same two parts gets the same bits.
__device__ __forceinline__ float2 chan_merge(float2 a, float2 b, float n) {
    const float d = a.x - b.x;
    return make_float2((a.x + b.x) * 0.5f, (a.y + b.y) + d * d * (0.5f * n));
}
// one 16-column chunk of pass 2: y = ((v + b) * rstd - mean * rstd) * gamma + beta, ReLU fused into the bf16 conversion, two
// 16-byte chunks of the swizzled K-major A operand
__device__ __forceinline__ void norm_chunk(const uint32_t (&v)[16], const float4 (&b)[4], const float4 (&g)[4], const float4 (&be)[4],
                                           uint64_t rstd2, uint64_t shift2, uint32_t a_base, int row, int c0) {
    uint32_t out[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint64_t t0 = fma2(add2(pk2u(v[4 * j], v[4 * j + 1]), pk2(b[j].x, b[j].y)), rstd2, shift2);
        const uint64_t t1 = fma2(add2(pk2u(v[4 * j + 2], v[4 * j + 3]), pk2(b[j].z, b[j].w)), rstd2, shift2);
        out[2 * j] = relu_bf16x2(fma2(t0, pk2(g[j].x, g[j].y), pk2(be[j].x, be[j].y)));
        out[2 * j + 1] = relu_bf16x2(fma2(t1, pk2(g[j].z, g[j].w), pk2(be[j].z, be[j].w)));
    }
    st_shared_v4(a_base + a_chunk_offset(row, c0 >> 3), make_uint4(out[0], out[1], out[2], out[3]));
    st_shared_v4(a_base + a_chunk_offset(row, (c0 >> 3) + 1), make_uint4(out[4], out[5], out[6], out[7]));
}

// bias + LayerNorm + ReLU epilogue of one hidden layer: TMEM accumulators -> bf16 A operand of the next GEMM.
// Two warps share a row quarter: warp w and w + 4 read TMEM lanes 32 * (w % 4) ..., each over half of the N columns.
// The arithmetic runs on packed fp32 pairs (4 instead of 9.5 floating-point instructions per element over the two passes), and
// the TMEM loads are double-buffered in registers: the load of chunk i + 1 is in flight while chunk i is processed (a TMEM round
// trip per chunk, exposed at 2 warps per scheduler, was most of the epilogue's time: profiles/r02_c_policy_phases.log).
template <int N>
__device__ __forceinline__ void layer_epilogue(uint32_t lane_addr, uint32_t a_base, float2 (*stats)[BM], int row, int half,
                                               const float* __restrict__ bias, const float* __restrict__ gamma,
                                               const float* __restrict__ beta, float eps) {
    constexpr int HALF = N / PARTS;   // columns of this warp
    static_assert(HALF % 64 == 0, "two 32-column chunks per iteration");
    const int cbeg = half * HALF;
    uint64_t s2 = pk2(0.f, 0.f), ss2 = pk2(0.f, 0.f);
    float k = 0.f;                    // the part's shift: its first column's v + b
    uint64_t nk2 = pk2(0.f, 0.f);
    if constexpr (PARTS == 2) {
        uint32_t va[32], vb[32];
        tmem_ld32(lane_addr + (uint32_t)cbeg, va);
#pragma unroll 1
        for (int c0 = cbeg; c0 < cbeg + HALF; c0 += 64) {
            float4 b[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = __ldg(reinterpret_cast<const float4*>(bias + c0) + j);
            tmem_wait_ld32(va);
            if (c0 == cbeg) { k = __uint_as_float(va[0]) + b[0].x; nk2 = pk2(-k, -k); }
            tmem_ld32(lane_addr + (uint32_t)(c0 + 32), vb);           // in flight while chunk A is summed
            stats_chunk(va, b, nk2, s2, ss2);
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = __ldg(reinterpret_cast<const float4*>(bias + c0 + 32) + j);
            tmem_wait_ld32(vb);
            if (c0 + 64 < cbeg + HALF) tmem_ld32(lane_addr + (uint32_t)(c0 + 64), va);
            stats_chunk(vb, b, nk2, s2, ss2);
        }
    } else {   // 18 warps share the register file (96 per thread): 16-column chunks
        uint32_t va[16], vb[16];
        tmem_ld16(lane_addr + (uint32_t)cbeg, va);
#pragma unroll 1
        for (int c0 = cbeg; c0 < cbeg + HALF; c0 += 32) {
            float4 b[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = __ldg(reinterpret_cast<const float4*>(bias + c0) + j);
            tmem_wait_ld16(va);
            if (c0 == cbeg) { k = __uint_as_float(va[0]) + b[0].x; nk2 = pk2(-k, -k); }
            tmem_ld16(lane_addr + (uint32_t)(c0 + 16), vb);
            stats_chunk16(va, b, nk2, s2, ss2);
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = __ldg(reinterpret_cast<const float4*>(bias + c0 + 16) + j);
            tmem_wait_ld16(vb);
            if (c0 + 32 < cbeg + HALF) tmem_ld16(lane_addr + (uint32_t)(c0 + 32), va);
            stats_chunk16(vb, b, nk2, s2, ss2);
        }
    }
    float s_lo, s_hi, q_lo, q_hi;
    upk2(s2, s_lo, s_hi); upk2(ss2, q_lo, q_hi);
    const float s = s_lo + s_hi, ss = q_lo + q_hi, ms = s * (1.0f / HALF);
    const float2 part = make_float2(k + ms, fmaxf(fmaf(-s, ms, ss), 0.f));   // the part's (mean, M2)
    float2 all;
    if (PARTS == 2) {
        stats[half][row] = part;
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");   // the two halves of every row have published their statistics
        all = chan_merge(stats[0][row], stats[1][row], (float)HALF);
    } else {
        // four parts through the same 2 KiB (224 of the 227 KiB are operands and weight ring): parts 2, 3 hand their statistics to
        // parts 0, 1, which publish the merged pairs; everybody merges the two pairs in the same order
        if (half >= 2) stats[half - 2][row] = part;
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
        if (half < 2) stats[half][row] = chan_merge(part, stats[half][row], (float)HALF);
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
        all = chan_merge(stats[0][row], stats[1][row], (float)(2 * HALF));
    }   // (the next layer's writes come after a_ready / acc_ready, which every epilogue thread passes first)
    const float mean = all.x, var = all.y * (1.0f / N);   // biased variance, as nn.LayerNorm
    const float rstd = rsqrtf(var + eps);
    const uint64_t rstd2 = pk2(rstd, rstd), shift2 = pk2(-mean * rstd, -mean * rstd);
    {
        uint32_t va[16], vb[16];
        tmem_ld16(lane_addr + (uint32_t)cbeg, va);
#pragma unroll 1
        for (int c0 = cbeg; c0 < cbeg + HALF; c0 += 32) {
            float4 b[4], g[4], be[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                b[j] = __ldg(reinterpret_cast<const float4*>(bias + c0) + j);
                g[j] = __ldg(reinterpret_cast<const float4*>(gamma + c0) + j);
                be[j] = __ldg(reinterpret_cast<const float4*>(beta + c0) + j);
            }
            tmem_wait_ld16(va);
            tmem_ld16(lane_addr + (uint32_t)(c0 + 16), vb);
            norm_chunk(va, b, g, be, rstd2, shift2, a_base, row, c0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                b[j] = __ldg(reinterpret_cast<const float4*>(bias + c0 + 16) + j);
                g[j] = __ldg(reinterpret_cast<const float4*>(gamma + c0 + 16) + j);
                be[j] = __ldg(reinterpret_cast<const float4*>(beta + c0 + 16) + j);
            }
            tmem_wait_ld16(vb);
            if (c0 + 32 < cbeg + HALF) tmem_ld16(lane_addr + (uint32_t)(c0 + 32), va);
            norm_chunk(vb, b, g, be, rstd2, shift2, a_base, row, c0 + 16);
        }
    }
}

// Device-resident call counter: every launch advances it by exactly one, a launch that computes no row included.  Each CTA
// reads it into shared memory (OFF_CTR, for its head epilogue), then arrives on the ticket; only the last arrival, after every
// CTA has read the old value, stores the new one and re-arms the ticket.  A CTA with tiles does it in the shadow of its second
// GEMM (4.7 us), where it costs nothing measurable: 206.1 against 206.3 us per forward at 131 072 rows (B200, 1000 W).  Placements
// measured and dropped: at the start of the kernel, before the CTA-wide barrier, 1.8 us; in the shadow of the first GEMM, 0.7 us.
__device__ __forceinline__ void counter_arrive(unsigned long long* ctr_dev, unsigned char* smem) {
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ctr_dev + 1);
    const unsigned long long c = *reinterpret_cast<volatile unsigned long long*>(ctr_dev) + 1ull;
    *reinterpret_cast<unsigned long long*>(smem + OFF_CTR) = c;
    __threadfence();   // this CTA's read is ordered before its arrival
    if (atomicAdd(ticket, 1u) == gridDim.x - 1u) { *ctr_dev = c; *ticket = 0u; }
}

// CL = CTAs per thread-block cluster (1, 2 or 4).  The CTAs of a cluster work on different row tiles in lock step and share
// every weight tile: CTA r loads rows [r * N / CL, (r + 1) * N / CL) of a stage and multicasts them to all, so the L2 -> SM weight
// traffic (904 KiB per 128-row tile, the kernel's bottleneck at CL = 1) is divided by CL.  A stage may be refilled only after the
// MMAs of ALL CTAs have read it: the empty barriers count CL arrivals, delivered by multicast tcgen05.commit.
// XW = IN: rows of exactly 104 floats, 16-byte aligned (the default network); XW = 0: any in_dim in [1, 256], rows 4-byte aligned.
// ctr_dev: NULL (the counter is P.ctr_lo / P.ctr_hi), or the handle's {u64 counter, u32 ticket} block.  It is a kernel argument
// of its own because two more fields in Params, even unused ones, made ptxas spill 80-96 B in the XW = 104 instantiations.
template <int CL, int XW>
__global__ void __launch_bounds__(THREADS, 1)   // (ptxas caps the registers per SM sub-partition: 3 of 10 warps x 168, 5 of 18 warps x 96)
policy_forward_kernel(const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1,
                      const __grid_constant__ CUtensorMap tm2, const __grid_constant__ CUtensorMap tm3, const Params P, unsigned long long* ctr_dev) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const uint32_t a_base = sbase, ring = sbase + OFF_RING, bars = sbase + OFF_BARS;
    float2 (*stats)[BM] = reinterpret_cast<float2 (*)[BM]>(smem + OFF_STATS);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM);
    const uint32_t bar_full = bars, bar_empty = bars + STAGES * 8, bar_a = bars + 2 * STAGES * 8, bar_acc = bar_a + 8;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kb0 = XW == IN ? IN_PAD / BK : P.kb0;

    int64_t n_rows = P.n_rows;
    if (P.n_rows_dev) { const int64_t lim = (int64_t)*P.n_rows_dev; n_rows = lim < n_rows ? (lim < 0 ? 0 : lim) : n_rows; }
    const int64_t n_tiles = (n_rows + BM - 1) / BM;
    if ((int64_t)(blockIdx.x / CL) * CL >= n_tiles) {   // uniform for the whole cluster: nothing was allocated yet
        if (ctr_dev && threadIdx.x == 0) counter_arrive(ctr_dev, smem);   // a launch without rows advances the counter too
        return;
    }
    // every CTA that stays runs the same number of iterations (the ring protocol is cluster-wide); a tile index beyond n_tiles is
    // an all-padding tile: zero rows in, no rows out
    const int64_t n_iter = (n_tiles + gridDim.x - 1) / gridDim.x;
    uint32_t cta_rank = 0;
    if (CL > 1) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta_rank));
    constexpr uint16_t MC_MASK = (uint16_t)((1u << CL) - 1u);
    if ((sbase & 1023u) != 0) { if (threadIdx.x == 0 && P.error_flag) atomicExch(P.error_flag, 100); __trap(); }

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, CL); }
        mbar_init(bar_a, EPI_THREADS);
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == EPI_WARPS + 1) {   // TMEM: all 512 columns (one CTA per SM by its shared-memory footprint)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + OFF_TMEM), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    if (CL > 1) cluster_sync_all();   // the peers' barriers are initialised before anything arrives on them remotely
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == EPI_WARPS) {
        // ===== TMA producer =====
        if (lane == 0) {
            const CUtensorMap* maps[N_LAYERS] = {&tm0, &tm1, &tm2, &tm3};
            int stage = 0; uint32_t phase = 0;
            for (int64_t it = 0; it < n_iter; ++it) {
#pragma unroll 1
                for (int l = 0; l < N_LAYERS; ++l) {
                    const uint32_t bytes = (uint32_t)(layer_n(l) * BK * 2);        // of the whole stage, all slices
                    const int slice_rows = layer_n(l) / CL;
                    for (int nc = 0; nc < layer_nchunks(l); ++nc)
                        for (int kb = 0; kb < layer_kblocks(l, kb0); ++kb) {
                            mbar_wait(bar_empty + stage * 8, phase ^ 1u, P.error_flag, 1);   // released by the MMAs of all CL CTAs
                            mbar_expect_tx(bar_full + stage * 8, bytes);
                            const uint32_t dst = ring + stage * STAGE_BYTES + cta_rank * (uint32_t)(slice_rows * BK * 2);
                            if (CL == 1) tma_load_2d(dst, maps[l], bar_full + stage * 8, kb * BK, nc * BN);
                            else tma_load_2d_mc(dst, maps[l], bar_full + stage * 8, kb * BK, nc * BN + (int)cta_rank * slice_rows, MC_MASK);
                            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                        }
                }
            }
        }
        __syncwarp();
    } else if (warp == EPI_WARPS + 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0, pa = 0;
            for (int64_t it = 0; it < n_iter; ++it) {
#pragma unroll 1
                for (int l = 0; l < N_LAYERS; ++l) {
                    mbar_wait(bar_a, pa, P.error_flag, 2);   // A operand of this layer is in shared memory, TMEM is drained
                    pa ^= 1u;
                    tc_fence_after();
                    const uint32_t idesc = instr_desc(layer_n(l));
                    for (int nc = 0; nc < layer_nchunks(l); ++nc) {
                        const uint32_t d = tmem_base + layer_col(l, nc);
                        for (int kb = 0; kb < layer_kblocks(l, kb0); ++kb) {
                            mbar_wait(bar_full + stage * 8, phase, P.error_flag, 3);
                            tc_fence_after();
                            const uint64_t adesc = smem_desc(a_base + kb * KBLOCK_BYTES), bdesc = smem_desc(ring + stage * STAGE_BYTES);
#pragma unroll
                            for (int s = 0; s < BK / 16; ++s)   // UMMA_K = 16 bf16 = 32 bytes inside the swizzle span
                                umma_f16(d, adesc + (uint64_t)(2 * s), bdesc + (uint64_t)(2 * s), idesc, (kb | s) ? 1u : 0u);
                            if (CL == 1) umma_commit(bar_empty + stage * 8);   // the stage is free once these MMAs have read it
                            else umma_commit_mc(bar_empty + stage * 8, MC_MASK);   // ... in every CTA of the cluster
                            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                        }
                    }
                    umma_commit(bar_acc);   // accumulators of this layer complete
                }
            }
        }
        __syncwarp();
    } else {
        // ===== operand loader + epilogue (warps 0-7) =====
        const int q = warp & 3, half = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t pacc = 0;
        long long* tstamp = nullptr;
        for (int64_t it = 0; it < n_iter; ++it) {
            const int64_t tile = (int64_t)blockIdx.x + it * gridDim.x;
            tstamp = (P.timing && blockIdx.x == 0 && threadIdx.x == 0 && it < P.timing_tiles) ? P.timing + it * 16 : nullptr;
            if (tstamp) tstamp[0] = clock64();
            if constexpr (XW == IN) {
                // x tile: fp32 [128, 104] -> bf16, K padded to 128 with zeros, swizzled K-major
#pragma unroll
                for (int i = 0; i < (BM * IN_PAD / 8) / EPI_THREADS; ++i) {
                    const int task = (int)threadIdx.x + i * EPI_THREADS;
                    const int r = task >> 4, c = task & 15;
                    uint4 packed = make_uint4(0u, 0u, 0u, 0u);
                    const int64_t grow = tile * BM + r;
                    if (c < IN / 8 && grow < n_rows) {
                        const float4* src = reinterpret_cast<const float4*>(P.obs + grow * IN + c * 8);
                        const float4 a = __ldg(src), b = __ldg(src + 1);
                        packed = make_uint4(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w), pack_bf16(b.x, b.y), pack_bf16(b.z, b.w));
                    }
                    st_shared_v4(a_base + a_chunk_offset(r, c), packed);
                }
            } else {
                // x tile: fp32 [128, in_dim] -> bf16, K padded to 64 * kb0 with zeros, swizzled K-major.  A row of a rollout buffer
                // [T + 1, N, in_dim] is only 4-byte aligned when in_dim * N is odd: one float per load, the 8 loads of a chunk
                // in flight together; the lanes of a warp cover consecutive chunks of a row
                const int chunks = kb0 * 8, in_dim = P.in_dim;
#pragma unroll 1
                for (int task = (int)threadIdx.x; task < BM * chunks; task += EPI_THREADS) {
                    const int r = task / chunks, c = task - r * chunks, c0 = c * 8;
                    const int64_t grow = tile * BM + r;
                    float x[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] = 0.f;
                    if (c0 < in_dim && grow < n_rows) {
                        const float* src = P.obs + grow * in_dim + c0;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (c0 + j < in_dim) x[j] = __ldg(src + j);
                    }
                    st_shared_v4(a_base + a_chunk_offset(r, c),
                                 make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7])));
                }
            }
            fence_async_smem();    // generic-proxy writes -> visible to the tensor core's async-proxy reads
            tc_fence_before();
            mbar_arrive(bar_a);
            if (tstamp) tstamp[1] = clock64();
            // hidden layers
#pragma unroll 1
            for (int l = 0; l < 3; ++l) {
                mbar_wait(bar_acc, pacc, P.error_flag, 4);
                pacc ^= 1u;
                tc_fence_after();
                if (tstamp) tstamp[2 + 2 * l] = clock64();
                if (l == 0) layer_epilogue<H1>(lane_addr, a_base, stats, row, half, P.vec + VEC_B1, P.vec + VEC_G1, P.vec + VEC_BE1, P.ln_eps);
                else if (l == 1) layer_epilogue<H2>(lane_addr, a_base, stats, row, half, P.vec + VEC_B2, P.vec + VEC_G2, P.vec + VEC_BE2, P.ln_eps);
                else layer_epilogue<H3>(lane_addr, a_base, stats, row, half, P.vec + VEC_B3, P.vec + VEC_G3, P.vec + VEC_BE3, P.ln_eps);
                fence_async_smem();
                tc_fence_before();
                mbar_arrive(bar_a);
                // while the second GEMM runs; the head epilogue reads the counter after the next layers' bar.sync 1
                if (it == 0 && l == 0 && ctr_dev && threadIdx.x == 0) counter_arrive(ctr_dev, smem);
                if (tstamp) tstamp[3 + 2 * l] = clock64();
            }
            // heads
            mbar_wait(bar_acc, pacc, P.error_flag, 5);
            pacc ^= 1u;
            tc_fence_after();
            if (tstamp) tstamp[8] = clock64();
            if (half == 0) {
                uint32_t v[16];
                tmem_ld16(lane_addr + 256u, v);
                tmem_wait_ld();
                const int64_t grow = tile * BM + row;
                if (grow < n_rows) {
                    float mean[ACT], eps[ACT + 2];
                    const float* vf = P.vec;
#pragma unroll
                    for (int k = 0; k < ACT; ++k) { mean[k] = __uint_as_float(v[k]) + vf[VEC_BH + k]; eps[k] = 0.f; }
                    const float value = __uint_as_float(v[ACT]) + vf[VEC_BH + ACT];
                    if (!P.deterministic && (P.actions || P.logp || P.actions_clipped)) {
                        uint32_t clo = P.ctr_lo, chi = P.ctr_hi;
                        if (ctr_dev) {
                            const unsigned long long c = *reinterpret_cast<const unsigned long long*>(smem + OFF_CTR);
                            clo = (uint32_t)c; chi = (uint32_t)(c >> 32);
                        }
                        const uint4 r0 = philox((uint32_t)grow, (uint32_t)((uint64_t)grow >> 32), clo, chi, P.k0, P.k1);
                        const uint4 r1 = philox((uint32_t)grow, (uint32_t)((uint64_t)grow >> 32) | 0x80000000u, clo, chi, P.k0, P.k1);
                        box_muller(r0.x, r0.y, &eps[0], &eps[1]);
                        box_muller(r0.z, r0.w, &eps[2], &eps[3]);
                        box_muller(r1.x, r1.y, &eps[4], &eps[5]);
                    }
                    float lp = -0.5f * ACT * 1.8378770664093453f;   // -(k/2) log(2 pi)
#pragma unroll
                    for (int k = 0; k < ACT; ++k) {
                        const float ls = vf[VEC_LS + k];
                        lp += -0.5f * eps[k] * eps[k] - ls;
                        const float a = fmaf(__expf(ls), eps[k], mean[k]);
                        if (P.actions) P.actions[grow * ACT + k] = a;
                        if (P.actions_clipped) P.actions_clipped[grow * ACT + k] = fminf(fmaxf(a, -1.f), 1.f);   // np.clip to the action space
                        if (P.mean) P.mean[grow * ACT + k] = mean[k];
                    }
                    if (P.values) P.values[grow] = value;
                    if (P.logp) P.logp[grow] = lp;
                }
            }
            tc_fence_before();   // the next tile's first GEMM overwrites the head accumulators: order the loads before its a_ready
            if (tstamp) tstamp[9] = clock64();
        }
    }
    tc_fence_before();
    if (CL > 1) cluster_sync_all();   // no CTA leaves while a peer may still multicast into its shared memory or arrive on its barriers
    else __syncthreads();
    if (warp == EPI_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// fp32 [rows, k_src] -> bf16 [rows_dst, k_dst], zero padded
__global__ void pack_bf16_kernel(const float* __restrict__ src, int rows, int k_src, __nv_bfloat16* __restrict__ dst, int rows_dst, int k_dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows_dst * k_dst) return;
    const int r = i / k_dst, c = i - r * k_dst;
    dst[i] = __float2bfloat16_rn((r < rows && c < k_src) ? src[(size_t)r * k_src + c] : 0.f);
}
// dst = src - mean(src), one block of 256 threads.  LayerNorm is shift invariant, so this changes nothing but the rounding: a
// common offset of a layer's bias is taken out once here instead of riding through every row's fp32 epilogue, where it would cost
// (offset / std) * 2^-24 of each normalised value (b_i - mean(b) is exact whenever b_i and the mean are within a factor 2).
__global__ void copy_centred_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int n) {
    __shared__ double part[256];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += src[i];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) part[threadIdx.x] += part[threadIdx.x + w];
        __syncthreads();
    }
    const float m = (float)(part[0] / n);
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i] - m;
}
// the handle's {counter, ticket} block: a new counter value, and a ticket re-armed for the next forward
__global__ void set_counter_kernel(unsigned long long* ctr, unsigned long long value) {
    ctr[0] = value;
    *reinterpret_cast<unsigned int*>(ctr + 1) = 0u;
}
__global__ void copy_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int n, int n_dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_dst) dst[i] = i < n ? src[i] : 0.f;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct hlynr_policy {
    int device = 0, sm_count = 148;
    int in_dim = IN, kb0 = IN_PAD / BK;   // input width, K blocks of the first GEMM
    DevPtr<__nv_bfloat16> w1, w2, w3, wh;   // [512,64*kb0], [512,512], [256,512], [16,256]
    DevPtr<float> vec;   // b1 g1 be1 (512 x3) | b2 g2 be2 (512 x3) | b3 g3 be3 (256 x3) | bh (16) | log_std (8)
    DevPtr<int> error_flag;
    DevPtr<unsigned long long> ctr;   // 16 bytes: the device-resident call counter (u64), then the forward's ticket (u32)
    DevPtr<long long> timing;   // debug timestamps (option "timing")
    int timing_on = 0;
    CUtensorMap tm[3][4];   // [log2(cluster size)][layer]: box rows = N / cluster size
    int cluster = 1;        // CTAs per cluster (option "cluster": 1, 2 or 4)
    int grid_for_cluster[3] = {0, 0, 0};
    float ln_eps = 1e-5f;
    bool ready = false, smem_configured = false;
    int64_t launches = 0;
};

namespace {
int make_map(EncodeTiledFn enc, CUtensorMap* m, void* base, int rows, int k, int box_rows) {
    const cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)k * 2};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : fail("cuTensorMapEncodeTiled failed with CUresult %d (rows %d, k %d)", (int)r, rows, k);
}

// The instantiation for log2 of the cluster size (ci: 0, 1, 2) and the input rows (fixed: the 104-wide loader, else the generic one).
using ForwardKernel = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, Params, unsigned long long*);
ForwardKernel forward_kernel(int ci, bool fixed) {
    static const ForwardKernel k[2][3] = {{policy_forward_kernel<1, IN>, policy_forward_kernel<2, IN>, policy_forward_kernel<4, IN>},
                                          {policy_forward_kernel<1, 0>, policy_forward_kernel<2, 0>, policy_forward_kernel<4, 0>}};
    return k[fixed ? 0 : 1][ci];
}
}  // namespace

extern "C" {

void hlynr_policy_destroy(hlynr_policy_t* p) {
    if (!p) return;
    DeviceGuard g(p->device);
    delete p;
}

int hlynr_policy_create(int device, hlynr_policy_t** out) { return hlynr_policy_create_dim(device, IN, out); }

int hlynr_policy_create_dim(int device, int in_dim, hlynr_policy_t** out) {
    if (!out) return fail("hlynr_policy_create: null argument");
    if (in_dim < 1 || in_dim > HLYNR_POLICY_MAX_IN) return fail("hlynr_policy_create: in_dim must be in [1, %d], got %d", HLYNR_POLICY_MAX_IN, in_dim);
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail("hlynr_policy_create: device %d not available (%d devices)", device, ndev);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("hlynr_policy_create: the fused policy kernel is sm_100a code (tcgen05 / TMEM); device %d is sm_%d%d", device, prop.major, prop.minor);
    std::unique_ptr<hlynr_policy> p(new (std::nothrow) hlynr_policy());
    if (!p) return fail("hlynr_policy_create: out of host memory");
    p->device = device; p->sm_count = prop.multiProcessorCount;
    p->in_dim = in_dim; p->kb0 = (in_dim + BK - 1) / BK;
    // the TMA map needs 16-byte row strides: w1 lives in a [512, 64 * kb0] buffer whose columns past in_dim are zero
    CK(alloc(p->w1, H1 * BK * p->kb0));
    CK(alloc(p->w2, H2 * H1));
    CK(alloc(p->w3, H3 * H2));
    CK(alloc(p->wh, HEAD_N * H3));
    CK(alloc(p->vec, VEC_TOTAL));
    CK(alloc(p->error_flag, 1));
    CK(cudaMemset(p->error_flag.get(), 0, sizeof(int)));
    CK(alloc(p->ctr, 2));
    CK(cudaMemset(p->ctr.get(), 0, 16));
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    const cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
        return fail("hlynr_policy_create: cuTensorMapEncodeTiled is not available from the driver");
    EncodeTiledFn enc = reinterpret_cast<EncodeTiledFn>(fn);
    for (int c = 0; c < 3; ++c) {
        const int cl = 1 << c;
        if (make_map(enc, &p->tm[c][0], p->w1.get(), H1, BK * p->kb0, BN / cl) || make_map(enc, &p->tm[c][1], p->w2.get(), H2, H1, BN / cl) ||
            make_map(enc, &p->tm[c][2], p->w3.get(), H3, H2, BN / cl) || make_map(enc, &p->tm[c][3], p->wh.get(), HEAD_N, H3, HEAD_N / cl))
            return 1;
    }
    *out = p.release();
    return 0;
}

int hlynr_policy_set_weights(hlynr_policy_t* p, const HlynrPolicyWeights* w, void* stream) {
    if (!p || !w) return fail("hlynr_policy_set_weights: null argument");
    const float* all[] = {w->w1, w->b1, w->ln1_g, w->ln1_b, w->w2, w->b2, w->ln2_g, w->ln2_b, w->w3, w->b3, w->ln3_g, w->ln3_b,
                          w->wa, w->ba, w->wv, w->bv, w->log_std};
    for (const float* q : all) if (!q) return fail("hlynr_policy_set_weights: null weight pointer");
    DeviceGuard g(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    auto pack = [&](const float* src, int rows, int k, __nv_bfloat16* dst, int rows_dst, int k_dst) {
        const int n = rows_dst * k_dst;
        pack_bf16_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, rows, k, dst, rows_dst, k_dst);
    };
    auto vec = [&](const float* src, int n, int off, int n_dst) { copy_f32_kernel<<<(n_dst + 255) / 256, 256, 0, st>>>(src, p->vec.get() + off, n, n_dst); };
    pack(w->w1, H1, p->in_dim, p->w1.get(), H1, BK * p->kb0);
    pack(w->w2, H2, H1, p->w2.get(), H2, H1);
    pack(w->w3, H3, H2, p->w3.get(), H3, H2);
    CK(cudaMemsetAsync(p->wh.get(), 0, sizeof(__nv_bfloat16) * HEAD_N * H3, st));
    pack(w->wa, ACT, H3, p->wh.get(), ACT, H3);                 // rows 0-5: action_net
    pack(w->wv, 1, H3, p->wh.get() + (size_t)ACT * H3, 1, H3);  // row 6: value_net
    auto centred = [&](const float* src, int n, int off) { copy_centred_f32_kernel<<<1, 256, 0, st>>>(src, p->vec.get() + off, n); };
    centred(w->b1, H1, VEC_B1); vec(w->ln1_g, H1, VEC_G1, H1); vec(w->ln1_b, H1, VEC_BE1, H1);
    centred(w->b2, H2, VEC_B2); vec(w->ln2_g, H2, VEC_G2, H2); vec(w->ln2_b, H2, VEC_BE2, H2);
    centred(w->b3, H3, VEC_B3); vec(w->ln3_g, H3, VEC_G3, H3); vec(w->ln3_b, H3, VEC_BE3, H3);
    CK(cudaMemsetAsync(p->vec.get() + VEC_BH, 0, sizeof(float) * 16, st));
    vec(w->ba, ACT, VEC_BH, ACT); vec(w->bv, 1, VEC_BH + ACT, 1);
    vec(w->log_std, ACT, VEC_LS, 8);
    CK(cudaGetLastError());
    p->ln_eps = w->ln_eps > 0.f ? w->ln_eps : 1e-5f;
    p->ready = true;
    p->launches += 17;
    return 0;
}

}  // extern "C"

namespace {
// hlynr_policy_forward (counter by value) and hlynr_policy_forward_dev (dev_counter: the handle's device-resident counter)
int launch_forward(const char* fn, hlynr_policy_t* p, const float* obs_dev, int64_t n_rows, const int32_t* n_rows_dev,
                   float* actions_dev, float* values_dev, float* logp_dev, float* mean_dev, float* actions_clipped_dev,
                   uint64_t seed, uint64_t counter, bool dev_counter, int deterministic, void* stream) {
    if (!p || !obs_dev) return fail("%s: null argument", fn);
    if (!p->ready) return fail("%s: hlynr_policy_set_weights has not been called", fn);
    if (n_rows <= 0) return fail("%s: n_rows must be positive", fn);
    const bool fixed = p->in_dim == IN;   // the 104-wide instantiation: float4 loads of 16-byte aligned rows
    if (fixed && ((uintptr_t)obs_dev & 15u) != 0) return fail("%s: obs_dev must be 16-byte aligned", fn);
    if (((uintptr_t)obs_dev & 3u) != 0) return fail("%s: obs_dev must be 4-byte aligned", fn);
    DeviceGuard g(p->device);
    if (!p->smem_configured) {
        for (int c = 0; c < 3; ++c) CK(cudaFuncSetAttribute(forward_kernel(c, fixed), cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        p->smem_configured = true;
    }
    Params P;
    memset(&P, 0, sizeof(P));
    P.obs = obs_dev; P.in_dim = p->in_dim; P.kb0 = p->kb0; P.n_rows = n_rows; P.n_rows_dev = n_rows_dev;
    P.vec = p->vec.get();
    P.actions = actions_dev; P.values = values_dev; P.logp = logp_dev; P.mean = mean_dev; P.actions_clipped = actions_clipped_dev;
    P.ln_eps = p->ln_eps;
    P.k0 = (uint32_t)seed; P.k1 = (uint32_t)(seed >> 32); P.ctr_lo = (uint32_t)counter; P.ctr_hi = (uint32_t)(counter >> 32);
    unsigned long long* ctr_dev = dev_counter ? p->ctr.get() : nullptr;
    P.deterministic = deterministic; P.error_flag = p->error_flag.get();
    P.timing = p->timing_on ? p->timing.get() : nullptr; P.timing_tiles = 8;
    const int64_t n_tiles = (n_rows + BM - 1) / BM;
    const int cl = p->cluster, ci = cl == 4 ? 2 : (cl == 2 ? 1 : 0);
    const ForwardKernel kernel = forward_kernel(ci, fixed);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = cl > 1 ? 1u : 0u;
    if (p->grid_for_cluster[ci] == 0) {   // one resident wave: as many clusters as fit the device (GPC boundaries limit cl = 4)
        int clusters = p->sm_count / cl;
        if (cl > 1) {
            cfg.gridDim = dim3((unsigned)(clusters * cl));
            int fit = 0;
            const cudaError_t oe = cudaOccupancyMaxActiveClusters(&fit, kernel, &cfg);
            if (oe == cudaSuccess && fit > 0 && fit < clusters) clusters = fit;
            else if (oe != cudaSuccess) cudaGetLastError();
        }
        p->grid_for_cluster[ci] = clusters * cl;
    }
    int64_t grid = ((n_tiles + cl - 1) / cl) * cl;
    if (grid > p->grid_for_cluster[ci]) grid = p->grid_for_cluster[ci];
    cfg.gridDim = dim3((unsigned)grid);
    const CUtensorMap* tm = p->tm[ci];
    const cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, tm[0], tm[1], tm[2], tm[3], P, ctr_dev);
    if (le != cudaSuccess) return fail("%s: launch failed: %s", fn, cudaGetErrorString(le));
    CK(cudaGetLastError());
    p->launches += 1;
    return 0;
}
}  // namespace

extern "C" {

int hlynr_policy_forward(hlynr_policy_t* p, const float* obs_dev, int64_t n_rows, const int32_t* n_rows_dev, float* actions_dev,
                         float* values_dev, float* logp_dev, float* mean_dev, float* actions_clipped_dev, uint64_t seed,
                         uint64_t counter, int deterministic, void* stream) {
    return launch_forward("hlynr_policy_forward", p, obs_dev, n_rows, n_rows_dev, actions_dev, values_dev, logp_dev, mean_dev,
                          actions_clipped_dev, seed, counter, false, deterministic, stream);
}

int hlynr_policy_forward_dev(hlynr_policy_t* p, const float* obs_dev, int64_t n_rows, const int32_t* n_rows_dev, float* actions_dev,
                             float* values_dev, float* logp_dev, float* mean_dev, float* actions_clipped_dev, uint64_t seed,
                             int deterministic, void* stream) {
    return launch_forward("hlynr_policy_forward_dev", p, obs_dev, n_rows, n_rows_dev, actions_dev, values_dev, logp_dev, mean_dev,
                          actions_clipped_dev, seed, 0, true, deterministic, stream);
}

int hlynr_policy_set_counter(hlynr_policy_t* p, uint64_t value, void* stream) {
    if (!p) return fail("hlynr_policy_set_counter: null argument");
    DeviceGuard g(p->device);
    set_counter_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(p->ctr.get(), (unsigned long long)value);
    CK(cudaGetLastError());
    p->launches += 1;
    return 0;
}

int hlynr_policy_get_counter(hlynr_policy_t* p, uint64_t* out, void* stream) {
    if (!p || !out) return fail("hlynr_policy_get_counter: null argument");
    DeviceGuard g(p->device);
    const cudaStream_t st = (cudaStream_t)stream;
    CK(cudaStreamSynchronize(st));
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, p->ctr.get(), sizeof(v), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *out = (uint64_t)v;
    return 0;
}

int hlynr_policy_set_option(hlynr_policy_t* p, const char* name, int64_t value) {
    if (!p || !name) return fail("null argument");
    if (strcmp(name, "timing") == 0) {   // debug: record SM-clock timestamps of the phases of CTA 0's first 8 tiles
        DeviceGuard g(p->device);
        if (value && !p->timing) {
            DevPtr<long long> t;   // kept only once it is zeroed
            CK(alloc(t, 8 * 16));
            CK(cudaMemset(t.get(), 0, sizeof(long long) * 8 * 16));
            p->timing = std::move(t);
        }
        p->timing_on = value != 0;
        return 0;
    }
    if (strcmp(name, "cluster") == 0) {
        if (value != 1 && value != 2 && value != 4) return fail("hlynr_policy_set_option: cluster must be 1, 2 or 4");
        p->cluster = (int)value;
        return 0;
    }
    return fail("hlynr_policy_set_option: unknown option '%s'", name);
}

/* Debug: the timestamps recorded by the last forward with option "timing" = 1: out[tile][16] (SM clock cycles): 0 tile start,
 * 1 x loaded, 2/4/6 accumulators of layer 1/2/3 ready, 3/5/7 epilogue of layer 1/2/3 done, 8 head accumulators ready, 9 tile done. */
int hlynr_policy_get_timing(hlynr_policy_t* p, long long* host_out) {
    if (!p || !host_out || !p->timing) return fail("hlynr_policy_get_timing: option \"timing\" was never enabled");
    DeviceGuard g(p->device);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(host_out, p->timing.get(), sizeof(long long) * 8 * 16, cudaMemcpyDeviceToHost));
    return 0;
}

int hlynr_policy_launch_count(const hlynr_policy_t* p, int64_t* out) {
    if (!p || !out) return fail("null argument");
    *out = p->launches;
    return 0;
}

}  // extern "C"
