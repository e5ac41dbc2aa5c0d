// kernels_tc.cu — prefill MulMat on the 5th-generation tensor cores (sm_100a only):
//   Y[n][m] = sum_k W[m][k] * X[n][k]   (ComputeForwardMulMatFP32, pkg/ml/ml.go:1976-2098, N > 8)
//
// tcgen05.mma.cta_group::1.kind::tf32 tiles (128 x 128 x 8), operands staged in shared memory by
// TMA (cp.async.bulk.tensor, 128-byte swizzle, K-major), FP32 accumulators in TMEM, epilogue through
// tcgen05.ld.  The reference computes in true FP32, and a single TF32 pass (10-bit mantissa) would
// cost ~5e-4 relative per GEMM; so the FP32 operands are split in the shared-memory stage
// ("3xTF32"): the tensor core truncates the raw FP32 tile to its TF32 high part a_hi by itself,
// a transform warp-group writes the residual a_lo = a - trunc_tf32(a) into a second buffer with the
// identical swizzled layout, and three MMAs accumulate  a_hi*b_hi + a_hi*b_lo + a_lo*b_hi  into the
// same TMEM tile: products accurate to ~2^-20, i.e. FP32-class results.
//
// The tensor core adds into its FP32 accumulator with truncation (measured: relative error grows
// linearly with the number of dependent accumulations, 3e-5 at K = 4096 with one accumulator), so the
// accumulation is two-level, like FP8 "promotion": TMEM holds the sum of only TC_CHUNK_KB k-blocks
// (K = 256), then an accumulate warp-group adds that partial tile into FP32 registers (round to
// nearest) while the MMA warp fills the other TMEM buffer.
//
// Q8_0 weights (WK_Q8): the weight operand arrives as the int8 tile (4 KB) + its block
// scales (512 B) by TMA from the 4-row-interleaved planes of kernels_q8.cu, and the transform warp-group
// DEQUANTISES IN THE SHARED-MEMORY STAGE: v = f32(d*q) is written as the hi operand and v - trunc(v)
// as the lo operand, both at the 128-byte-swizzled K-major positions the MMA descriptors expect.
//
// F16 weights (WK_F16): the weight operand arrives as the row-major binary16 tile (128 rows x 64 B, 8 KB) by TMA into
// the stage's a_lo buffer, and the transform warp-group widens it to FP32 into a_raw at the swizzled K-major positions.
// Every binary16 value (subnormals included) is exact in TF32, so the weight's lo part is zero: each K step issues
// two MMAs, a*b_lo + a*b_hi, with the same two-level accumulation.
//
// Warp roles (320 threads, 1 CTA per SM, one 128x128 output tile per CTA):
//   warp 0      : TMA producer (one elected lane)
//   warp 1      : TMEM allocator + MMA issuer (one elected lane)
//   warps 2..5  : transform (hi/lo split of every stage)
//   warps 6..9  : accumulate (TMEM chunk -> registers, FP32 RN) and epilogue (registers -> HBM)
// Pipelines: full_raw[s] (TMA -> transform, MMA), full_lo[s] (transform -> MMA),
//            empty[s] (tcgen05.commit -> TMA), tmem_full[b] (chunk commit -> accumulate),
//            tmem_empty[b] (accumulate -> MMA).
// Every wait has a clock-based timeout that traps instead of hanging the GPU.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "kernels.cuh"

namespace lb {
namespace k {

constexpr int TC_BM = 128;      // weight rows per tile  (UMMA M)
constexpr int TC_BN = 128;      // tokens per tile       (UMMA N)
constexpr int TC_BK = 32;       // floats per stage along K = one 128-byte swizzle row
constexpr int TC_UK = 8;        // K per tcgen05.mma for kind::tf32 (32 bytes)
constexpr int TC_STAGES = 3;
constexpr int TC_THREADS = 320;
constexpr int TC_CHUNK_KB = 8;  // k-blocks (of 32) summed inside TMEM before promotion to registers
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 4;  // 16 KB
constexpr uint32_t TC_B_BYTES = TC_BN * TC_BK * 4;  // 16 KB
constexpr uint32_t TC_Q_BYTES = TC_BM * TC_BK;              // int8 weight tile (Q8 mode): 32 row groups x 128 B
constexpr uint32_t TC_D_BYTES = (TC_BM / 4) * 16;           // its scales: one float4 per row group
constexpr uint32_t TC_H_BYTES = TC_BM * TC_BK * 2;          // binary16 weight tile (F16 mode), staged in the a_lo buffer
enum WeightKind { WK_F32 = 0, WK_Q8 = 1, WK_F16 = 2 };
constexpr uint32_t TC_STAGE_BYTES = 2 * TC_A_BYTES + 2 * TC_B_BYTES + TC_Q_BYTES + 1024;  // raw + lo for A and B, q tile, scales (padded)
constexpr uint32_t TC_SMEM_BYTES = TC_STAGES * TC_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    const long long t0 = clock64();
    while (true) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
        if (clock64() - t0 > 4000000000LL) __trap();  // ~2 s: a pipeline bug must not hang the box
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 32 columns of 32-bit accumulators -> 32 registers per thread
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float v[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}

// K-major, SWIZZLE_128B shared-memory operand descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1)
//   [32,46) stride byte offset >> 4 = 1024 B between 8-row groups | [46,48) version = 1 | [61,64) layout = 2
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major
__host__ __device__ constexpr uint32_t make_idesc_tf32(uint32_t M, uint32_t N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// unpack 4 int8 (see kernels_q8.cu): exact, avoids the I2F pipe
__device__ __forceinline__ void tc_unpack4(uint32_t w, float f[4]) {
    const uint32_t u = w ^ 0x80808080u;
    f[0] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7650)) - 8388736.0f;
    f[1] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7651)) - 8388736.0f;
    f[2] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7652)) - 8388736.0f;
    f[3] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7653)) - 8388736.0f;
}

template <int WK>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmD,
                   const __grid_constant__ CUtensorMap tmX, float *__restrict__ Y,
                   uint32_t ldy, const float *__restrict__ res, uint32_t M, uint32_t N, uint32_t K) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // swizzle-128B atoms need 1024-byte alignment
    uint8_t *base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bars = base + TC_STAGES * TC_STAGE_BYTES;
    auto full_raw = [&](int s) { return bars + 8u * s; };
    auto full_lo = [&](int s) { return bars + 8u * (TC_STAGES + s); };
    auto empty = [&](int s) { return bars + 8u * (2 * TC_STAGES + s); };
    auto tmem_full = [&](int b) { return bars + 8u * (3 * TC_STAGES + b); };
    auto tmem_empty = [&](int b) { return bars + 8u * (3 * TC_STAGES + 2 + b); };
    const uint32_t tmem_slot = bars + 8u * (3 * TC_STAGES + 4);
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(base_ptr + TC_STAGES * TC_STAGE_BYTES + 8u * (3 * TC_STAGES + 4));
    auto a_raw = [&](int s) { return base + s * TC_STAGE_BYTES; };
    auto a_lo = [&](int s) { return base + s * TC_STAGE_BYTES + TC_A_BYTES; };
    auto b_raw = [&](int s) { return base + s * TC_STAGE_BYTES + 2 * TC_A_BYTES; };
    auto b_lo = [&](int s) { return base + s * TC_STAGE_BYTES + 2 * TC_A_BYTES + TC_B_BYTES; };
    auto q_tile = [&](int s) { return base + s * TC_STAGE_BYTES + 2 * TC_A_BYTES + 2 * TC_B_BYTES; };
    auto d_tile = [&](int s) { return base + s * TC_STAGE_BYTES + 2 * TC_A_BYTES + 2 * TC_B_BYTES + TC_Q_BYTES; };

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t m0 = blockIdx.x * TC_BM, n0 = blockIdx.y * TC_BN;
    const uint32_t num_kb = K / TC_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; s++) {
            mbar_init(full_raw(s), 1);
            mbar_init(full_lo(s), 128);
            mbar_init(empty(s), 1);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(tmem_full(b), 1);
            mbar_init(tmem_empty(b), 128);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 2 * TC_BN);  // two 128-column FP32 accumulator buffers
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            for (uint32_t kb = 0; kb < num_kb; kb++) {
                const int s = kb % TC_STAGES;
                const uint32_t ph = (kb / TC_STAGES) & 1;
                mbar_wait(empty(s), ph ^ 1);
                if (WK == WK_Q8) {
                    mbar_expect_tx(full_raw(s), TC_Q_BYTES + TC_D_BYTES + TC_B_BYTES);
                    tma_load_2d(q_tile(s), &tmW, full_raw(s), (int)(kb * TC_BK * 4), (int)(m0 / 4));  // 128 B per row group
                    tma_load_2d(d_tile(s), &tmD, full_raw(s), (int)(kb * 4), (int)(m0 / 4));           // one float4 per row group
                } else if (WK == WK_F16) {
                    mbar_expect_tx(full_raw(s), TC_H_BYTES + TC_B_BYTES);
                    tma_load_2d(a_lo(s), &tmW, full_raw(s), (int)(kb * TC_BK), (int)m0);             // 64 B per row, unswizzled
                } else {
                    mbar_expect_tx(full_raw(s), TC_A_BYTES + TC_B_BYTES);
                    tma_load_2d(a_raw(s), &tmW, full_raw(s), (int)(kb * TC_BK), (int)m0);
                }
                tma_load_2d(b_raw(s), &tmX, full_raw(s), (int)(kb * TC_BK), (int)n0);
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_tf32(TC_BM, TC_BN);
            for (uint32_t kb = 0; kb < num_kb; kb++) {
                const int s = kb % TC_STAGES;
                const uint32_t ph = (kb / TC_STAGES) & 1;
                const uint32_t chunk = kb / TC_CHUNK_KB, buf = chunk & 1;
                const uint32_t tmem_d = tmem_base + buf * TC_BN;
                const bool first_of_chunk = (kb % TC_CHUNK_KB) == 0;
                if (first_of_chunk) {
                    mbar_wait(tmem_empty(buf), ((chunk >> 1) & 1) ^ 1);  // accumulate warps drained this buffer
                    tc_fence_after();
                }
                mbar_wait(full_raw(s), ph);
                mbar_wait(full_lo(s), ph);
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < TC_BK / TC_UK; kk++) {
                    const uint32_t koff = kk * TC_UK * 4;  // 32 bytes per K step inside the swizzled row
                    const uint64_t dA = make_smem_desc(a_raw(s) + koff), dAl = make_smem_desc(a_lo(s) + koff);
                    const uint64_t dB = make_smem_desc(b_raw(s) + koff), dBl = make_smem_desc(b_lo(s) + koff);
                    if (WK == WK_F16) {   // a is exact in TF32: no a_lo term
                        tc_mma_tf32(tmem_d, dA, dBl, idesc, (first_of_chunk && kk == 0) ? 0u : 1u);  // a * b_lo
                        tc_mma_tf32(tmem_d, dA, dB, idesc, 1u);                                      // a * b_hi
                    } else {
                        tc_mma_tf32(tmem_d, dAl, dB, idesc, (first_of_chunk && kk == 0) ? 0u : 1u);  // a_lo * b_hi
                        tc_mma_tf32(tmem_d, dA, dBl, idesc, 1u);                                     // a_hi * b_lo
                        tc_mma_tf32(tmem_d, dA, dB, idesc, 1u);                                      // a_hi * b_hi
                    }
                }
                tc_commit(empty(s));  // frees the stage once these MMAs have read it
                if ((kb % TC_CHUNK_KB) == TC_CHUNK_KB - 1 || kb == num_kb - 1) tc_commit(tmem_full(buf));
            }
        }
    } else if (warp < 6) {
        // ================= transform warps: a_lo = a - trunc_tf32(a), same swizzled offsets =================
        const int t = threadIdx.x - 64;  // 0..127
        for (uint32_t kb = 0; kb < num_kb; kb++) {
            const int s = kb % TC_STAGES;
            const uint32_t ph = (kb / TC_STAGES) & 1;
            mbar_wait(full_raw(s), ph);
            const float4 *ar = reinterpret_cast<const float4 *>(base_ptr + s * TC_STAGE_BYTES);
            float4 *al = reinterpret_cast<float4 *>(base_ptr + s * TC_STAGE_BYTES + TC_A_BYTES);
            const float4 *br = reinterpret_cast<const float4 *>(base_ptr + s * TC_STAGE_BYTES + 2 * TC_A_BYTES);
            float4 *bl = reinterpret_cast<float4 *>(base_ptr + s * TC_STAGE_BYTES + 2 * TC_A_BYTES + TC_B_BYTES);
            auto lo = [](float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); };
            if (WK == WK_Q8) {
                // dequantise in the shared-memory stage: 256 vectors (row group g, k4) of 4 rows x 4 int8
                const uint4 *qt = reinterpret_cast<const uint4 *>(base_ptr + s * TC_STAGE_BYTES + 2 * TC_A_BYTES + 2 * TC_B_BYTES);
                const float4 *dt = reinterpret_cast<const float4 *>(base_ptr + s * TC_STAGE_BYTES + 2 * TC_A_BYTES + 2 * TC_B_BYTES + TC_Q_BYTES);
                float4 *ah = reinterpret_cast<float4 *>(base_ptr + s * TC_STAGE_BYTES);
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const int vec = t + i * 128, g = vec >> 3, k4 = vec & 7;
                    const uint4 w = qt[vec];
                    const float4 sc = dt[g];
                    const uint32_t wr[4] = {w.x, w.y, w.z, w.w};
                    const float sr[4] = {sc.x, sc.y, sc.z, sc.w};
#pragma unroll
                    for (int rr = 0; rr < 4; rr++) {
                        float f[4];
                        tc_unpack4(wr[rr], f);
                        const float4 v = make_float4(__fmul_rn(sr[rr], f[0]), __fmul_rn(sr[rr], f[1]), __fmul_rn(sr[rr], f[2]), __fmul_rn(sr[rr], f[3]));
                        const int row = g * 4 + rr;
                        const int off = row * 8 + (k4 ^ (row & 7));  // float4 index inside the 128-byte-swizzled K-major tile
                        ah[off] = v;
                        al[off] = make_float4(lo(v.x), lo(v.y), lo(v.z), lo(v.w));
                    }
                }
            } else if (WK == WK_F16) {
                // widen in the shared-memory stage: 512 vectors (row, 8 halves) of the unswizzled tile in the a_lo buffer
                const uint4 *ht = reinterpret_cast<const uint4 *>(al);
                float4 *ah = reinterpret_cast<float4 *>(base_ptr + s * TC_STAGE_BYTES);
                uint4 hv[TC_H_BYTES / 16 / 128];
#pragma unroll
                for (int i = 0; i < (int)(TC_H_BYTES / 16 / 128); i++) hv[i] = ht[t + i * 128];
#pragma unroll
                for (int i = 0; i < (int)(TC_H_BYTES / 16 / 128); i++) {
                    const int vec = t + i * 128, row = vec >> 2, k8 = vec & 3;
                    const float2 f0 = __half22float2(*reinterpret_cast<const __half2 *>(&hv[i].x));
                    const float2 f1 = __half22float2(*reinterpret_cast<const __half2 *>(&hv[i].y));
                    const float2 f2 = __half22float2(*reinterpret_cast<const __half2 *>(&hv[i].z));
                    const float2 f3 = __half22float2(*reinterpret_cast<const __half2 *>(&hv[i].w));
                    ah[row * 8 + ((2 * k8) ^ (row & 7))] = make_float4(f0.x, f0.y, f1.x, f1.y);       // float4 index inside the swizzled tile
                    ah[row * 8 + ((2 * k8 + 1) ^ (row & 7))] = make_float4(f2.x, f2.y, f3.x, f3.y);
                }
            } else {
#pragma unroll
                for (int i = 0; i < (int)(TC_A_BYTES / 16 / 128); i++) {
                    float4 v = ar[t + i * 128];
                    al[t + i * 128] = make_float4(lo(v.x), lo(v.y), lo(v.z), lo(v.w));
                }
            }
#pragma unroll
            for (int i = 0; i < (int)(TC_B_BYTES / 16 / 128); i++) {
                float4 v = br[t + i * 128];
                bl[t + i * 128] = make_float4(lo(v.x), lo(v.y), lo(v.z), lo(v.w));
            }
            fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core (async proxy)
            mbar_arrive(full_lo(s));
        }
    } else {
        // ================= accumulate (TMEM chunk -> FP32 registers, RN) + epilogue =================
        const uint32_t q = warp & 3;  // a warp may only touch TMEM lanes [32*(warp%4), +32)
        const uint32_t m = m0 + q * 32 + lane;
        float acc[TC_BN];
#pragma unroll
        for (int j = 0; j < TC_BN; j++) acc[j] = 0.f;
        const uint32_t num_chunks = (num_kb + TC_CHUNK_KB - 1) / TC_CHUNK_KB;
        for (uint32_t chunk = 0; chunk < num_chunks; chunk++) {
            const uint32_t buf = chunk & 1;
            mbar_wait(tmem_full(buf), (chunk >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < TC_BN / 32; c++) {
                float v[32];
                tmem_ld_32x32(tmem_base + buf * TC_BN + ((q * 32u) << 16) + (uint32_t)(c * 32), v);
#pragma unroll
                for (int j = 0; j < 32; j++) acc[c * 32 + j] = __fadd_rn(acc[c * 32 + j], v[j]);
            }
            tc_fence_before();
            mbar_arrive(tmem_empty(buf));
        }
        if (m < M) {
#pragma unroll
            for (int j = 0; j < TC_BN; j++) {
                const uint32_t n = n0 + j;
                if (n < N) {
                    float o = acc[j];
                    if (res) o = __fadd_rn(o, res[(size_t)n * ldy + m]);
                    Y[(size_t)n * ldy + m] = o;  // lanes = consecutive m: coalesced
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 2 * TC_BN);
    }
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        LB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        LB_CHECK(p != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled is not available in this driver");
        fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}
// row-major [rows][cols] FP32 matrix with row pitch ld floats; box = 32 floats (128 B) x box_rows, 128-byte swizzle
static CUtensorMap make_map(const float *ptr, uint32_t rows, uint32_t cols, uint32_t ld, uint32_t box_rows) {
    CUtensorMap m;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {TC_BK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(ptr), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LB_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return m;
}

// generic 2-D tensor map: `cols` elements of `esz` bytes per row, row pitch `pitch_bytes`
static CUtensorMap make_map_raw(const void *ptr, CUtensorMapDataType dt, uint64_t rows, uint64_t cols, uint64_t pitch_bytes,
                                uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle sw) {
    CUtensorMap m;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = get_encode()(&m, dt, 2, const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LB_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return m;
}

bool gemm_tf32x3_supported(uint32_t M, uint32_t K, uint32_t ldx, const float *W, const float *X) {
    (void)M;
    return K >= TC_BK && (K % TC_BK) == 0 && (ldx % 4) == 0 && ((uintptr_t)W % 16) == 0 && ((uintptr_t)X % 16) == 0;
}

template <int WK>
static void set_attr_once() {
    // function attributes are per device: the C-ABI lets one process hold models on several GPUs
    static bool attr[64] = {};
    int dev = 0;
    LB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        LB_CUDA(cudaFuncSetAttribute(gemm_tf32x3_kernel<WK>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
}

void gemm_tf32x3(const float *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N, float *Y, uint32_t ldy,
                 const float *residual, cudaStream_t st) {
    LB_CHECK(gemm_tf32x3_supported(M, K, ldx, W, X), "gemm_tf32x3: unsupported shape (K must be a multiple of 32)");
    if (!M || !N) return;
    set_attr_once<WK_F32>();
    CUtensorMap tmW = make_map(W, M, K, K, TC_BM);
    CUtensorMap tmX = make_map(X, N, K, ldx, TC_BN);
    dim3 grid((M + TC_BM - 1) / TC_BM, (N + TC_BN - 1) / TC_BN);
    gemm_tf32x3_kernel<WK_F32><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(tmW, tmW, tmX, Y, ldy, residual, M, N, K);
    LB_LAUNCH_CHECK();
}

// Q8_0 weights (4-row-interleaved planes of kernels_q8.cu): q plane = [M/4 row groups][K*4 bytes],
// d plane = [M/4][K/32 float4]
void gemm_q8_tc(const int8_t *Q, const float *D, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N, float *Y,
                uint32_t ldy, const float *residual, cudaStream_t st) {
    LB_CHECK(K >= TC_BK && K % TC_BK == 0 && M % 4 == 0 && ldx % 4 == 0 && (uintptr_t)Q % 16 == 0 && (uintptr_t)D % 16 == 0 &&
                 (uintptr_t)X % 16 == 0, "gemm_q8_tc: unsupported shape");
    if (!M || !N) return;
    set_attr_once<WK_Q8>();
    CUtensorMap tmQ = make_map_raw(Q, CU_TENSOR_MAP_DATA_TYPE_UINT8, M / 4, (uint64_t)K * 4, (uint64_t)K * 4, TC_BK * 4, TC_BM / 4,
                                   CU_TENSOR_MAP_SWIZZLE_NONE);
    CUtensorMap tmD = make_map_raw(D, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, M / 4, (uint64_t)(K / 32) * 4, (uint64_t)(K / 32) * 16, 4, TC_BM / 4,
                                   CU_TENSOR_MAP_SWIZZLE_NONE);
    CUtensorMap tmX = make_map(X, N, K, ldx, TC_BN);
    dim3 grid((M + TC_BM - 1) / TC_BM, (N + TC_BN - 1) / TC_BN);
    gemm_tf32x3_kernel<WK_Q8><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(tmQ, tmD, tmX, Y, ldy, residual, M, N, K);
    LB_LAUNCH_CHECK();
}

// F16 weights: row-major [M][K] binary16 plane; box = 32 halves (64 B) x 128 rows, unswizzled (widened by the transform warps)
void gemm_f16_tc(const uint16_t *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N, float *Y, uint32_t ldy,
                 const float *residual, cudaStream_t st) {
    LB_CHECK(K >= TC_BK && K % TC_BK == 0 && ldx % 4 == 0 && (uintptr_t)W % 16 == 0 && (uintptr_t)X % 16 == 0,
             "gemm_f16_tc: unsupported shape (K must be a multiple of 32)");
    if (!M || !N) return;
    set_attr_once<WK_F16>();
    CUtensorMap tmW = make_map_raw(W, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, M, K, (uint64_t)K * 2, TC_BK, TC_BM, CU_TENSOR_MAP_SWIZZLE_NONE);
    CUtensorMap tmX = make_map(X, N, K, ldx, TC_BN);
    dim3 grid((M + TC_BM - 1) / TC_BM, (N + TC_BN - 1) / TC_BN);
    gemm_tf32x3_kernel<WK_F16><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(tmW, tmW, tmX, Y, ldy, residual, M, N, K);
    LB_LAUNCH_CHECK();
}

void gemm_auto(const float *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N, float *Y, uint32_t ldy,
               const float *residual, cudaStream_t st) {
    static const bool no_tc = getenv("LB_NO_TC") != nullptr;
    if (!no_tc && gemm_tf32x3_supported(M, K, ldx, W, X)) gemm_tf32x3(W, M, K, X, ldx, N, Y, ldy, residual, st);
    else gemm_f32(W, M, K, X, ldx, N, Y, ldy, residual, st);
}
void gemm_q8_auto(const int8_t *Q, const float *D, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N, float *Y,
                  uint32_t ldy, const float *residual, cudaStream_t st) {
    static const bool no_tc = getenv("LB_NO_TC") != nullptr;
    if (!no_tc && K >= TC_BK && K % TC_BK == 0) gemm_q8_tc(Q, D, M, K, X, ldx, N, Y, ldy, residual, st);
    else gemm_q8(Q, D, M, K, X, ldx, N, Y, ldy, residual, st);
}

}  // namespace k
}  // namespace lb
