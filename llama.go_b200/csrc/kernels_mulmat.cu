// kernels_mulmat.cu — MulMat family (ComputeForwardMulMatFP32, pkg/ml/ml.go:1976-2098).
//   gemv_f32 / gemv_f32_swiglu : decode (N = 1..8 activation columns), HBM-bound weight streaming
//   gemv_f16 / gemv_f16_swiglu : the same kernels reading binary16 weights (widened in registers)
//   gemm_f32                   : prefill (any N), shared-memory tiled FP32
//   mul_mat_generic            : arbitrary strided operands (the permuted K·Q / V^T·P products
//                                of the op-level API)
// dst[n][m] = sum_k W[m][k] * x[n][k], FP32 multiply-add (the GPU fuses mul+add into FMA; the
// reference's scalar loop and AVX1 vdot do not — a <=1e-6 relative difference, far inside the
// 1e-3 logits budget; summation order likewise differs).
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.cuh"

namespace lb {
namespace k {

// 4 consecutive weights -> float4: FP32 (one streaming 128-bit load) or binary16 (one streaming 64-bit load, widened exactly)
__device__ __forceinline__ float4 ld_w4(const float *p) { return ld_stream_f4(p); }
__device__ __forceinline__ float4 ld_w4(const __half *p) {
    uint32_t a, b;
    asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
    const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&a)), hi = __half22float2(*reinterpret_cast<const __half2 *>(&b));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// ------------------------------------------------------------------------------------------
// Decode GEMV.  One warp owns RPW consecutive weight rows; the 32 lanes stride the row in
// 128-bit pieces (fully coalesced 512 B per warp-load), UNROLL independent loads in flight per
// row, weights bypass L1 (touched once), the tiny activation vector is re-read through L1.
// ------------------------------------------------------------------------------------------
constexpr int GEMV_WARPS = 8;   // swiglu kernel
constexpr int GEMV_UNROLL = 4;

template <typename WT, int NC, int RPW, int WARPS, int UNROLL>
__global__ void __launch_bounds__(WARPS * 32)
gemv_kernel(const WT *__restrict__ W, uint32_t M, uint32_t K, const float *__restrict__ x, uint32_t ldx,
            float *__restrict__ y, uint32_t ldy, const float *__restrict__ res) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t row0 = (blockIdx.x * WARPS + warp) * RPW;
    if (row0 >= M) return;
    float acc[RPW][NC];
#pragma unroll
    for (int r = 0; r < RPW; r++)
#pragma unroll
        for (int c = 0; c < NC; c++) acc[r][c] = 0.f;
    const WT *wr[RPW];
#pragma unroll
    for (int r = 0; r < RPW; r++) wr[r] = W + (size_t)min(row0 + r, M - 1) * K;

    // first batch of weight loads is issued BEFORE waiting on the predecessor grid (weights are
    // read-only): under PDL this CTA streams while the previous kernel drains.
    float4 w[UNROLL][RPW];
    auto load_batch = [&](uint32_t kk) {
#pragma unroll
        for (int u = 0; u < UNROLL; u++) {
            uint32_t kq = kk + u * 128;
#pragma unroll
            for (int r = 0; r < RPW; r++)
                w[u][r] = (kq < K) ? ld_w4(wr[r] + kq) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    pdl_launch_dependents();
    load_batch(lane * 4);
    pdl_wait();
    for (uint32_t kk = lane * 4; kk < K;) {
        float4 xv[UNROLL][NC];
#pragma unroll
        for (int u = 0; u < UNROLL; u++) {
            uint32_t kq = kk + u * 128;
#pragma unroll
            for (int c = 0; c < NC; c++)
                xv[u][c] = (kq < K) ? __ldg(reinterpret_cast<const float4 *>(x + (size_t)c * ldx + kq)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; u++) {
#pragma unroll
            for (int c = 0; c < NC; c++) {
#pragma unroll
                for (int r = 0; r < RPW; r++) {
                    acc[r][c] = fmaf(w[u][r].x, xv[u][c].x, acc[r][c]);
                    acc[r][c] = fmaf(w[u][r].y, xv[u][c].y, acc[r][c]);
                    acc[r][c] = fmaf(w[u][r].z, xv[u][c].z, acc[r][c]);
                    acc[r][c] = fmaf(w[u][r].w, xv[u][c].w, acc[r][c]);
                }
            }
        }
        kk += 128 * UNROLL;
        if (kk < K) load_batch(kk);
    }
#pragma unroll
    for (int r = 0; r < RPW; r++)
#pragma unroll
        for (int c = 0; c < NC; c++) acc[r][c] = warp_sum(acc[r][c]);
    if (lane == 0) {
#pragma unroll
        for (int r = 0; r < RPW; r++) {
            uint32_t row = row0 + r;
            if (row < M) {
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    float v = acc[r][c];
                    if (res) v = __fadd_rn(v, res[(size_t)c * ldy + row]);
                    y[(size_t)c * ldy + row] = v;
                }
            }
        }
    }
}

template <typename WT, int NC>
__global__ void __launch_bounds__(GEMV_WARPS * 32)
gemv_swiglu_kernel(const WT *__restrict__ W1, const WT *__restrict__ W3, uint32_t M, uint32_t K,
                   const float *__restrict__ x, uint32_t ldx, float *__restrict__ act, uint32_t ldy) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t row = blockIdx.x * GEMV_WARPS + warp;
    if (row >= M) return;
    float a1[NC], a3[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) a1[c] = a3[c] = 0.f;
    const WT *w1 = W1 + (size_t)row * K, *w3 = W3 + (size_t)row * K;
    float4 p[GEMV_UNROLL], q[GEMV_UNROLL];
    auto load_batch = [&](uint32_t kk) {
#pragma unroll
        for (int u = 0; u < GEMV_UNROLL; u++) {
            uint32_t kq = kk + u * 128;
            p[u] = (kq < K) ? ld_w4(w1 + kq) : make_float4(0.f, 0.f, 0.f, 0.f);
            q[u] = (kq < K) ? ld_w4(w3 + kq) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    pdl_launch_dependents();
    load_batch(lane * 4);   // weights first, then wait for the predecessor grid (PDL)
    pdl_wait();
    for (uint32_t kk = lane * 4; kk < K;) {
#pragma unroll
        for (int u = 0; u < GEMV_UNROLL; u++) {
            uint32_t kq = kk + u * 128;
            if (kq < K) {
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    float4 xv = __ldg(reinterpret_cast<const float4 *>(x + (size_t)c * ldx + kq));
                    a1[c] = fmaf(p[u].x, xv.x, a1[c]); a1[c] = fmaf(p[u].y, xv.y, a1[c]);
                    a1[c] = fmaf(p[u].z, xv.z, a1[c]); a1[c] = fmaf(p[u].w, xv.w, a1[c]);
                    a3[c] = fmaf(q[u].x, xv.x, a3[c]); a3[c] = fmaf(q[u].y, xv.y, a3[c]);
                    a3[c] = fmaf(q[u].z, xv.z, a3[c]); a3[c] = fmaf(q[u].w, xv.w, a3[c]);
                }
            }
        }
        kk += 128 * GEMV_UNROLL;
        if (kk < K) load_batch(kk);
    }
#pragma unroll
    for (int c = 0; c < NC; c++) { a1[c] = warp_sum(a1[c]); a3[c] = warp_sum(a3[c]); }
    if (lane == 0) {
#pragma unroll
        for (int c = 0; c < NC; c++) act[(size_t)c * ldy + row] = __fmul_rn(silu_ref(a1[c]), a3[c]);
    }
}

// Multi-column (pod batch, NC >= 3) variant: a warp owns 4 weight rows so every activation float4 it
// pulls through L1 is used by 4 rows — with one row per warp the 8 activation columns would need
// ~190 B/clk of L1 bandwidth per SM to keep up with the weight stream (the L1 limit is 128).
template <typename WT, int NC>
__global__ void __launch_bounds__(128)
gemv_cols_kernel(const WT *__restrict__ W, uint32_t M, uint32_t K, const float *__restrict__ x, uint32_t ldx,
                 float *__restrict__ y, uint32_t ldy, const float *__restrict__ res) {
    constexpr int RPW = 4, U = 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t row0 = (blockIdx.x * 4 + warp) * RPW;
    if (row0 >= M) return;
    float acc[RPW][NC];
#pragma unroll
    for (int r = 0; r < RPW; r++)
#pragma unroll
        for (int c = 0; c < NC; c++) acc[r][c] = 0.f;
    const WT *wr[RPW];
#pragma unroll
    for (int r = 0; r < RPW; r++) wr[r] = W + (size_t)min(row0 + r, M - 1) * K;
    float4 w[U][RPW];
    auto load_batch = [&](uint32_t kk) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint32_t kq = kk + u * 128;
#pragma unroll
            for (int r = 0; r < RPW; r++) w[u][r] = (kq < K) ? ld_w4(wr[r] + kq) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    pdl_launch_dependents();
    load_batch(lane * 4);
    pdl_wait();
    for (uint32_t kk = lane * 4; kk < K;) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint32_t kq = kk + u * 128;
            if (kq < K) {
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    const float4 xv = __ldg(reinterpret_cast<const float4 *>(x + (size_t)c * ldx + kq));
#pragma unroll
                    for (int r = 0; r < RPW; r++) {
                        acc[r][c] = fmaf(w[u][r].x, xv.x, acc[r][c]); acc[r][c] = fmaf(w[u][r].y, xv.y, acc[r][c]);
                        acc[r][c] = fmaf(w[u][r].z, xv.z, acc[r][c]); acc[r][c] = fmaf(w[u][r].w, xv.w, acc[r][c]);
                    }
                }
            }
        }
        kk += 128 * U;
        if (kk < K) load_batch(kk);
    }
#pragma unroll
    for (int r = 0; r < RPW; r++)
#pragma unroll
        for (int c = 0; c < NC; c++) acc[r][c] = warp_sum(acc[r][c]);
    if (lane == 0) {
#pragma unroll
        for (int r = 0; r < RPW; r++) {
            const uint32_t row = row0 + r;
            if (row < M) {
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    float v = acc[r][c];
                    if (res) v = __fadd_rn(v, res[(size_t)c * ldy + row]);
                    y[(size_t)c * ldy + row] = v;
                }
            }
        }
    }
}

template <typename WT, int NC>
static void gemv_launch(const WT *W, uint32_t M, uint32_t K, const float *x, uint32_t ldx, float *y, uint32_t ldy,
                        const float *res, cudaStream_t st) {
    // Large M (qkv, lm_head): 2 rows per warp, 8 warps.  Small M (wo, w2: M = dim): one row per warp
    // and 4-warp blocks so that the grid is >= 6 blocks per SM and every SM holds the same number of
    // warps (256 blocks of 16 rows left 1.7 blocks per SM: measured 51-63 % of HBM peak).
    constexpr bool two = (NC <= 2);
    if (NC >= 3) {
        launch_pdl(gemv_cols_kernel<WT, NC>, dim3((M + 15) / 16), dim3(128), 0, st, W, M, K, x, ldx, y, ldy, res);
    } else if (two && M >= 8192) {
        unsigned grid = (M + 15) / 16;
        launch_pdl(gemv_kernel<WT, NC, 2, 8, 4>, dim3(grid), dim3(256), 0, st, W, M, K, x, ldx, y, ldy, res);
    } else {
        unsigned grid = (M + 3) / 4;
        launch_pdl(gemv_kernel<WT, NC, 1, 4, (NC <= 4 ? 8 : 4)>, dim3(grid), dim3(128), 0, st, W, M, K, x, ldx, y, ldy, res);
    }
}

template <typename WT>
static void gemv_any(const char *what, const WT *W, uint32_t M, uint32_t K, const float *x, uint32_t ldx, uint32_t N, float *y,
                     uint32_t ldy, const float *residual, cudaStream_t st) {
    LB_CHECK(N >= 1 && N <= 8, std::string(what) + ": N must be 1..8");
    LB_CHECK((K & 3) == 0 && (ldx & 3) == 0, std::string(what) + ": K and ldx must be multiples of 4");
    switch (N) {
        case 1: gemv_launch<WT, 1>(W, M, K, x, ldx, y, ldy, residual, st); break;
        case 2: gemv_launch<WT, 2>(W, M, K, x, ldx, y, ldy, residual, st); break;
        case 3: gemv_launch<WT, 3>(W, M, K, x, ldx, y, ldy, residual, st); break;
        case 4: gemv_launch<WT, 4>(W, M, K, x, ldx, y, ldy, residual, st); break;
        case 5: gemv_launch<WT, 5>(W, M, K, x, ldx, y, ldy, residual, st); break;
        case 6: gemv_launch<WT, 6>(W, M, K, x, ldx, y, ldy, residual, st); break;
        case 7: gemv_launch<WT, 7>(W, M, K, x, ldx, y, ldy, residual, st); break;
        default: gemv_launch<WT, 8>(W, M, K, x, ldx, y, ldy, residual, st); break;
    }
}
void gemv_f32(const float *W, uint32_t M, uint32_t K, const float *x, uint32_t ldx, uint32_t N, float *y,
              uint32_t ldy, const float *residual, cudaStream_t st) {
    gemv_any("gemv_f32", W, M, K, x, ldx, N, y, ldy, residual, st);
}
void gemv_f16(const uint16_t *W, uint32_t M, uint32_t K, const float *x, uint32_t ldx, uint32_t N, float *y,
              uint32_t ldy, const float *residual, cudaStream_t st) {
    gemv_any("gemv_f16", reinterpret_cast<const __half *>(W), M, K, x, ldx, N, y, ldy, residual, st);
}

template <typename WT, int NC>
static void swiglu_launch(const WT *W1, const WT *W3, uint32_t M, uint32_t K, const float *x, uint32_t ldx,
                          float *act, uint32_t ldy, cudaStream_t st) {
    unsigned grid = (M + GEMV_WARPS - 1) / GEMV_WARPS;
    launch_pdl(gemv_swiglu_kernel<WT, NC>, dim3(grid), dim3(GEMV_WARPS * 32), 0, st, W1, W3, M, K, x, ldx, act, ldy);
}
template <typename WT>
static void swiglu_any(const char *what, const WT *W1, const WT *W3, uint32_t M, uint32_t K, const float *x, uint32_t ldx,
                       uint32_t N, float *act, uint32_t ldy, cudaStream_t st) {
    LB_CHECK(N >= 1 && N <= 8, std::string(what) + ": N must be 1..8");
    LB_CHECK((K & 3) == 0 && (ldx & 3) == 0, std::string(what) + ": K and ldx must be multiples of 4");
    switch (N) {
        case 1: swiglu_launch<WT, 1>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        case 2: swiglu_launch<WT, 2>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        case 3: swiglu_launch<WT, 3>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        case 4: swiglu_launch<WT, 4>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        case 5: swiglu_launch<WT, 5>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        case 6: swiglu_launch<WT, 6>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        case 7: swiglu_launch<WT, 7>(W1, W3, M, K, x, ldx, act, ldy, st); break;
        default: swiglu_launch<WT, 8>(W1, W3, M, K, x, ldx, act, ldy, st); break;
    }
}
void gemv_f32_swiglu(const float *W1, const float *W3, uint32_t M, uint32_t K, const float *x, uint32_t ldx,
                     uint32_t N, float *act, uint32_t ldy, cudaStream_t st) {
    swiglu_any("gemv_f32_swiglu", W1, W3, M, K, x, ldx, N, act, ldy, st);
}
void gemv_f16_swiglu(const uint16_t *W1, const uint16_t *W3, uint32_t M, uint32_t K, const float *x, uint32_t ldx,
                     uint32_t N, float *act, uint32_t ldy, cudaStream_t st) {
    swiglu_any("gemv_f16_swiglu", reinterpret_cast<const __half *>(W1), reinterpret_cast<const __half *>(W3), M, K, x, ldx, N, act, ldy, st);
}

// ------------------------------------------------------------------------------------------
// Prefill GEMM (FP32 CUDA cores): Y[n][m] = sum_k W[m][k] X[n][k].  128(m) x 64(n) x 16(k) tiles,
// 256 threads, 8x4 register micro-tile, operands staged k-major in shared memory.
// ------------------------------------------------------------------------------------------
constexpr int GM = 128, GN = 64, GK = 16;
__global__ void __launch_bounds__(256)
gemm_kernel(const float *__restrict__ W, uint32_t M, uint32_t K, const float *__restrict__ X, uint32_t ldx,
            uint32_t N, float *__restrict__ Y, uint32_t ldy, const float *__restrict__ res) {
    __shared__ float As[GK][GM + 4];
    __shared__ float Bs[GK][GN + 4];
    const uint32_t m0 = blockIdx.x * GM, n0 = blockIdx.y * GN;
    const int tid = threadIdx.x;
    const int tm = (tid & 15) * 8;   // 16 threads along m, 8 rows each
    const int tn = (tid >> 4) * 4;   // 16 threads along n, 4 cols each
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.f;

    for (uint32_t k0 = 0; k0 < K; k0 += GK) {
        // W tile: 128 rows x 16 k = 512 float4, two per thread
#pragma unroll
        for (int i = 0; i < 2; i++) {
            int f = tid + i * 256;
            int r = f >> 2, kq = (f & 3) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m0 + r < M && k0 + kq < K) v = *reinterpret_cast<const float4 *>(W + (size_t)(m0 + r) * K + k0 + kq);
            As[kq + 0][r] = v.x; As[kq + 1][r] = v.y; As[kq + 2][r] = v.z; As[kq + 3][r] = v.w;
        }
        {
            int r = tid >> 2, kq = (tid & 3) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n0 + r < N && k0 + kq < K) v = *reinterpret_cast<const float4 *>(X + (size_t)(n0 + r) * ldx + k0 + kq);
            Bs[kq + 0][r] = v.x; Bs[kq + 1][r] = v.y; Bs[kq + 2][r] = v.z; Bs[kq + 3][r] = v.w;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; kk++) {
            float a[8], b[4];
            *reinterpret_cast<float4 *>(a) = *reinterpret_cast<const float4 *>(&As[kk][tm]);
            *reinterpret_cast<float4 *>(a + 4) = *reinterpret_cast<const float4 *>(&As[kk][tm + 4]);
            *reinterpret_cast<float4 *>(b) = *reinterpret_cast<const float4 *>(&Bs[kk][tn]);
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
        uint32_t n = n0 + tn + j;
        if (n >= N) continue;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint32_t m = m0 + tm + i;
            if (m < M) {
                float v = acc[i][j];
                if (res) v = __fadd_rn(v, res[(size_t)n * ldy + m]);
                Y[(size_t)n * ldy + m] = v;
            }
        }
    }
}
void gemm_f32(const float *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N, float *Y,
              uint32_t ldy, const float *residual, cudaStream_t st) {
    LB_CHECK((K & 3) == 0 && (ldx & 3) == 0, "gemm_f32: K and ldx must be multiples of 4");
    if (!N || !M) return;
    dim3 grid((M + GM - 1) / GM, (N + GN - 1) / GN);
    gemm_kernel<<<grid, 256, 0, st>>>(W, M, K, X, ldx, N, Y, ldy, residual);
    LB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------------------------------
// Generic strided MulMat: one warp per dst element (src0/src1 unit-stride along dim 0, every other
// stride arbitrary — exactly what the reference's generic path supports, ml.go:2039-2091).
// dst NE = [a.ne1, b.ne1, a.ne2, b.ne3].
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mul_mat_generic_kernel(TView a, TView b, TView d, size_t total) {
    const int lane = threadIdx.x & 31;
    size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t e = warp; e < total; e += nwarps) {
        size_t r = e;
        uint32_t i01 = (uint32_t)(r % a.ne[1]); r /= a.ne[1];
        uint32_t ic = (uint32_t)(r % b.ne[1]); r /= b.ne[1];
        uint32_t i02 = (uint32_t)(r % a.ne[2]); r /= a.ne[2];
        uint32_t i03 = (uint32_t)r;
        const float *pa = a.data + (size_t)i01 * a.nb[1] + (size_t)i02 * a.nb[2] + (size_t)i03 * a.nb[3];
        const float *pb = b.data + (size_t)ic * b.nb[1] + (size_t)i02 * b.nb[2] + (size_t)i03 * b.nb[3];
        float acc = 0.f;
        for (uint32_t kq = lane; kq < a.ne[0]; kq += 32) acc = fmaf(pa[kq], pb[kq], acc);
        acc = warp_sum(acc);
        if (lane == 0)
            d.data[(size_t)i01 * d.nb[0] + (size_t)ic * d.nb[1] + (size_t)i02 * d.nb[2] + (size_t)i03 * d.nb[3]] = acc;
    }
}
void mul_mat_generic(const TView &a, const TView &b, const TView &dst, cudaStream_t st) {
    size_t total = (size_t)a.ne[1] * b.ne[1] * a.ne[2] * b.ne[3];
    if (!total) return;
    size_t blocks = (total + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    mul_mat_generic_kernel<<<(unsigned)blocks, 256, 0, st>>>(a, b, dst, total);
    LB_LAUNCH_CHECK();
}

}  // namespace k
}  // namespace lb
