// kernels_elementwise.cu — memory-bound op kernels: one CUDA kernel per reference
// ComputeForward* (pkg/ml/ml.go:1711-2644), warp-shuffle reductions, 128-bit accesses where the
// layout allows.  Numerics follow the reference op for op (see each kernel).
#include "common.cuh"
#include "kernels.cuh"

#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>

namespace lb {
std::atomic<uint64_t> g_launches{0};
bool g_use_pdl = getenv("LB_NO_PDL") == nullptr;
namespace k {

static inline unsigned blocks_for(size_t n, unsigned per_block, unsigned cap = 148 * 16) {
    size_t b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > cap) b = cap;
    return (unsigned)b;
}

// ---- GetRows: ComputeForwardGetRows, ml.go:1711-1750 (ids travel as float32, llama.go:239-242)
template <typename IdT>
__global__ void get_rows_kernel(const float *__restrict__ table, uint32_t nc, const IdT *__restrict__ ids,
                                float *__restrict__ dst) {
    uint32_t row = blockIdx.x;
    size_t r = (size_t)(uint32_t)ids[row];
    const float *src = table + r * nc;
    float *d = dst + (size_t)row * nc;
    if ((nc & 3) == 0) {
        for (uint32_t i = threadIdx.x * 4; i < nc; i += blockDim.x * 4)
            *reinterpret_cast<float4 *>(d + i) = *reinterpret_cast<const float4 *>(src + i);
    } else {
        for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) d[i] = src[i];
    }
}
void get_rows_f32ids(const float *table, uint32_t nc, const float *ids, uint32_t nr, float *dst, cudaStream_t st) {
    if (!nr) return;
    get_rows_kernel<float><<<nr, 256, 0, st>>>(table, nc, ids, dst);
    LB_LAUNCH_CHECK();
}
void get_rows_u32ids(const float *table, uint32_t nc, const uint32_t *ids, uint32_t nr, float *dst, cudaStream_t st) {
    if (!nr) return;
    get_rows_kernel<uint32_t><<<nr, 256, 0, st>>>(table, nc, ids, dst);
    LB_LAUNCH_CHECK();
}

// ---- RMSNorm (+ optional weight multiply): ComputeForwardRMSNormFP32, ml.go:1753-1812 and the
// following Mul(Repeat(w), cur) (llama.go:255-259).  f32 square, f64 accumulate, /n, +eps,
// 1/sqrt in f64, cast to f32 scale, f32 multiply; then a second f32 multiply by the weight.
__global__ void __launch_bounds__(256) rms_norm_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                                       float *__restrict__ y, uint32_t nc) {
    __shared__ double red[8];
    __shared__ float s_scale;
    const float *xr = x + (size_t)blockIdx.x * nc;
    float *yr = y + (size_t)blockIdx.x * nc;
    double acc = 0.0;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) {
        float v = xr[i];
        acc += (double)__fmul_rn(v, v);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += red[i];
        double mean = t / (double)nc;
        s_scale = (float)(1.0 / sqrt(mean + 1e-5));
    }
    __syncthreads();
    float sc = s_scale;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) {
        float v = __fmul_rn(xr[i], sc);
        yr[i] = w ? __fmul_rn(w[i], v) : v;
    }
}
// Fast path (nc % 4 == 0, nc <= 8192): the row is read ONCE with 128-bit loads into registers
// (all loads issued before the first use), reduced, and written back from registers.
template <int VPT>  // float4 per thread
__global__ void __launch_bounds__(256) rms_norm_reg_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                                           float *__restrict__ y, uint32_t nc) {
    __shared__ double red[8];
    __shared__ float s_scale;
    const float4 *xr = reinterpret_cast<const float4 *>(x + (size_t)blockIdx.x * nc);
    float4 *yr = reinterpret_cast<float4 *>(y + (size_t)blockIdx.x * nc);
    const uint32_t n4 = nc >> 2;
    pdl_launch_dependents();
    pdl_wait();
    float4 v[VPT];
#pragma unroll
    for (int i = 0; i < VPT; i++) {
        uint32_t idx = threadIdx.x + i * 256;
        v[i] = idx < n4 ? xr[idx] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < VPT; i++) {
        acc += (double)__fmul_rn(v[i].x, v[i].x);
        acc += (double)__fmul_rn(v[i].y, v[i].y);
        acc += (double)__fmul_rn(v[i].z, v[i].z);
        acc += (double)__fmul_rn(v[i].w, v[i].w);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; i++) t += red[i];
        s_scale = (float)(1.0 / sqrt(t / (double)nc + 1e-5));
    }
    __syncthreads();
    const float sc = s_scale;
    const float4 *wr = reinterpret_cast<const float4 *>(w);
#pragma unroll
    for (int i = 0; i < VPT; i++) {
        uint32_t idx = threadIdx.x + i * 256;
        if (idx < n4) {
            float4 o;
            o.x = __fmul_rn(v[i].x, sc); o.y = __fmul_rn(v[i].y, sc); o.z = __fmul_rn(v[i].z, sc); o.w = __fmul_rn(v[i].w, sc);
            if (w) {
                float4 ww = __ldg(wr + idx);
                o.x = __fmul_rn(ww.x, o.x); o.y = __fmul_rn(ww.y, o.y); o.z = __fmul_rn(ww.z, o.z); o.w = __fmul_rn(ww.w, o.w);
            }
            yr[idx] = o;
        }
    }
}
void rms_norm(const float *x, const float *w, float *y, uint32_t nc, uint32_t nr, cudaStream_t st) {
    if (!nr) return;
    const bool aligned = (nc & 3) == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 15) == 0 && ((uintptr_t)w & 15) == 0;
    if (aligned && nc <= 4096) { launch_pdl(rms_norm_reg_kernel<4>, dim3(nr), dim3(256), 0, st, x, w, y, nc); return; }
    if (aligned && nc <= 8192) { launch_pdl(rms_norm_reg_kernel<8>, dim3(nr), dim3(256), 0, st, x, w, y, nc); return; }
    rms_norm_kernel<<<nr, 256, 0, st>>>(x, w, y, nc);
    LB_LAUNCH_CHECK();
}

// ---- Repeat: ComputeForwardRepeatFP32, ml.go:1822-1868 (2-D)
__global__ void repeat_kernel(const float *__restrict__ a, uint32_t nc0, uint32_t nr0, float *__restrict__ dst,
                              uint32_t nc, uint32_t nr) {
    size_t n = (size_t)nc * nr;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        uint32_t r = (uint32_t)(i / nc), c = (uint32_t)(i % nc);
        dst[i] = a[(size_t)(r % nr0) * nc0 + (c % nc0)];
    }
}
void repeat_rows(const float *a, uint32_t nc0, uint32_t nr0, float *dst, uint32_t nc, uint32_t nr, cudaStream_t st) {
    repeat_kernel<<<blocks_for((size_t)nc * nr, 256), 256, 0, st>>>(a, nc0, nr0, dst, nc, nr);
    LB_LAUNCH_CHECK();
}

// ---- Mul / Add / Scale / Silu: ml.go:1877-1914, 2515-2584, 2331-2374, 2587-2644
enum { OP_MUL, OP_ADD, OP_SILU, OP_SWIGLU };
template <int OP>
__global__ void ewise_kernel(const float *__restrict__ a, const float *__restrict__ b, float *__restrict__ dst, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float r;
        if (OP == OP_MUL) r = __fmul_rn(a[i], b[i]);
        else if (OP == OP_ADD) r = __fadd_rn(a[i], b[i]);
        else if (OP == OP_SILU) r = silu_ref(a[i]);
        else r = __fmul_rn(silu_ref(a[i]), b[i]);
        dst[i] = r;
    }
}
void mul(const float *a, const float *b, float *dst, size_t n, cudaStream_t st) {
    ewise_kernel<OP_MUL><<<blocks_for(n, 256), 256, 0, st>>>(a, b, dst, n);
    LB_LAUNCH_CHECK();
}
void add(const float *a, const float *b, float *dst, size_t n, cudaStream_t st) {
    ewise_kernel<OP_ADD><<<blocks_for(n, 256), 256, 0, st>>>(a, b, dst, n);
    LB_LAUNCH_CHECK();
}
void silu(const float *x, float *y, size_t n, cudaStream_t st) {
    ewise_kernel<OP_SILU><<<blocks_for(n, 256), 256, 0, st>>>(x, nullptr, y, n);
    LB_LAUNCH_CHECK();
}
void swiglu(const float *gate, const float *up, float *dst, size_t n, cudaStream_t st) {
    ewise_kernel<OP_SWIGLU><<<blocks_for(n, 256), 256, 0, st>>>(gate, up, dst, n);
    LB_LAUNCH_CHECK();
}
__global__ void scale_kernel(float *x, float v, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] = __fmul_rn(x[i], v);
}
void scale_inplace(float *x, float v, size_t n, cudaStream_t st) {
    scale_kernel<<<blocks_for(n, 256), 256, 0, st>>>(x, v, n);
    LB_LAUNCH_CHECK();
}

// ---- DiagMaskInf: ml.go:2377-2414.  x is [ne0=T, ne1=N, ne2=H]; x[k][j][i] = -inf for i > past + j
__global__ void diag_mask_kernel(float *x, uint32_t ne0, uint32_t ne1, size_t n, uint32_t past) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += stride) {
        uint32_t i = (uint32_t)(idx % ne0);
        uint32_t j = (uint32_t)((idx / ne0) % ne1);
        if (i > past + j) x[idx] = -INFINITY;
    }
}
void diag_mask_inf(float *x, uint32_t ne0, uint32_t ne1, uint32_t ne2, uint32_t past, cudaStream_t st) {
    size_t n = (size_t)ne0 * ne1 * ne2;
    diag_mask_kernel<<<blocks_for(n, 256), 256, 0, st>>>(x, ne0, ne1, n, past);
    LB_LAUNCH_CHECK();
}

// ---- SoftMax: ComputeForwardSoftMaxFP32, ml.go:2432-2505.  f32 max; e = f32(exp(f64(p - max)));
// -inf -> 0; multiply by f32(1/sum).  Deviation: the f32 sum is a tree (warp shuffle), the
// reference's is sequential in i — an O(1e-7) relative difference.
__global__ void __launch_bounds__(256) soft_max_kernel(float *x, uint32_t nc) {
    __shared__ float red[8];
    __shared__ float s_val;
    float *p = x + (size_t)blockIdx.x * nc;
    float m = -INFINITY;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) m = fmaxf(m, p[i]);
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = red[0];
        for (int i = 1; i < (int)(blockDim.x >> 5); i++) t = fmaxf(t, red[i]);
        s_val = t;
    }
    __syncthreads();
    m = s_val;
    float sum = 0.f;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) {
        float v = p[i];
        float e = (v == -INFINITY) ? 0.f : (float)exp((double)__fsub_rn(v, m));
        p[i] = e;
        sum += e;
    }
    sum = warp_sum(sum);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += red[i];
        s_val = __fdiv_rn(1.0f, t);
    }
    __syncthreads();
    float inv = s_val;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) p[i] = __fmul_rn(p[i], inv);
}
void soft_max_rows(float *x, uint32_t nc, uint32_t nr, cudaStream_t st) {
    if (!nr) return;
    soft_max_kernel<<<nr, 256, 0, st>>>(x, nc);
    LB_LAUNCH_CHECK();
}

// ---- Copy (OP_CPY): ComputeForwardDupFP32, ml.go:2110-2240 — strided source to contiguous dst
__global__ void cpy_kernel(TView s, float *__restrict__ dst, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < n; id += stride) {
        size_t r = id;
        uint32_t i0 = (uint32_t)(r % s.ne[0]); r /= s.ne[0];
        uint32_t i1 = (uint32_t)(r % s.ne[1]); r /= s.ne[1];
        uint32_t i2 = (uint32_t)(r % s.ne[2]); r /= s.ne[2];
        uint32_t i3 = (uint32_t)r;
        dst[id] = s.data[(size_t)i0 * s.nb[0] + (size_t)i1 * s.nb[1] + (size_t)i2 * s.nb[2] + (size_t)i3 * s.nb[3]];
    }
}
void cpy_strided(const TView &src, float *dst, cudaStream_t st) {
    size_t n = (size_t)src.ne[0] * src.ne[1] * src.ne[2] * src.ne[3];
    if (!n) return;
    cpy_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, dst, n);
    LB_LAUNCH_CHECK();
}

// ---- RoPE: ComputeForwardRopeFP32, ml.go:2253-2328.  theta = pow(10000, -i0/dims), angle p*theta,
// cos/sin and the 2x2 rotation in f64, cast to f32.  mode 0: rows i2=0.., p = past+i2;
// mode 1: rows i2 = past.., p = i2.
__device__ __forceinline__ void rope_pair(float *d, uint32_t p, int i0, uint32_t dims) {
    double theta = pow(10000.0, ((double)(-i0)) / (double)dims);
    double s, c;
    sincos((double)p * theta, &s, &c);
    double x0 = (double)d[0], x1 = (double)d[1];
    d[0] = (float)(__dsub_rn(__dmul_rn(x0, c), __dmul_rn(x1, s)));
    d[1] = (float)(__dadd_rn(__dmul_rn(x0, s), __dmul_rn(x1, c)));
}
__global__ void rope_kernel(float *x, uint32_t ne0, uint32_t ne1, uint32_t ne2, uint32_t past, uint32_t dims,
                            uint32_t mode, uint32_t i2_begin) {
    uint32_t half = dims / 2;
    size_t n = (size_t)half * ne1 * (ne2 - i2_begin);
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += stride) {
        uint32_t j = (uint32_t)(idx % half);
        uint32_t i1 = (uint32_t)((idx / half) % ne1);
        uint32_t i2 = (uint32_t)(idx / ((size_t)half * ne1)) + i2_begin;
        uint32_t p = mode == 0 ? past + i2 : i2;
        rope_pair(x + ((size_t)i2 * ne1 + i1) * ne0 + 2 * j, p, (int)(2 * j), dims);
    }
}
void rope(float *x, uint32_t ne0, uint32_t ne1, uint32_t ne2, uint32_t past, uint32_t dims, uint32_t mode, cudaStream_t st) {
    uint32_t begin = mode == 0 ? 0 : past;
    if (begin >= ne2) return;
    size_t n = (size_t)(dims / 2) * ne1 * (ne2 - begin);
    if (!n) return;
    rope_kernel<<<blocks_for(n, 128), 128, 0, st>>>(x, ne0, ne1, ne2, past, dims, mode, begin);
    LB_LAUNCH_CHECK();
}

// fused hot-path variant: rotate q in place, rotate k into the cache, copy v into the cache.
__global__ void rope_qk_store_kernel(float *q, const float *__restrict__ k, const float *__restrict__ v, uint32_t ld,
                                     float *__restrict__ Kc, float *__restrict__ Vc, uint32_t N,
                                     const uint32_t *__restrict__ past_dev, uint32_t dim, uint32_t hd) {
    pdl_launch_dependents();
    pdl_wait();
    const uint32_t past = *past_dev;
    uint32_t half = dim / 2;
    size_t n = (size_t)half * N;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += stride) {
        uint32_t pr = (uint32_t)(idx % half);   // pair index within the row
        uint32_t t = (uint32_t)(idx / half);
        uint32_t e = 2 * pr;                    // element index in [0, dim)
        int i0 = (int)(e % hd);                 // pair offset inside the head
        uint32_t p = past + t;
        double theta = pow(10000.0, ((double)(-i0)) / (double)hd);
        double s, c;
        sincos((double)p * theta, &s, &c);
        float *qd = q + (size_t)t * ld + e;
        double x0 = (double)qd[0], x1 = (double)qd[1];
        qd[0] = (float)(__dsub_rn(__dmul_rn(x0, c), __dmul_rn(x1, s)));
        qd[1] = (float)(__dadd_rn(__dmul_rn(x0, s), __dmul_rn(x1, c)));
        const float *kd = k + (size_t)t * ld + e;
        x0 = (double)kd[0]; x1 = (double)kd[1];
        float2 kr;
        kr.x = (float)(__dsub_rn(__dmul_rn(x0, c), __dmul_rn(x1, s)));
        kr.y = (float)(__dadd_rn(__dmul_rn(x0, s), __dmul_rn(x1, c)));
        *reinterpret_cast<float2 *>(Kc + (size_t)(past + t) * dim + e) = kr;
        *reinterpret_cast<float2 *>(Vc + (size_t)(past + t) * dim + e) =
            *reinterpret_cast<const float2 *>(v + (size_t)t * ld + e);
    }
}
void rope_qk_store(float *q, const float *k, const float *v, uint32_t ld, float *Kc, float *Vc, uint32_t N,
                   const uint32_t *past_dev, uint32_t dim, uint32_t heads, cudaStream_t st) {
    size_t n = (size_t)(dim / 2) * N;
    launch_pdl(rope_qk_store_kernel, dim3(blocks_for(n, 128)), dim3(128), 0, st, q, k, v, ld, Kc, Vc, N, past_dev, dim, dim / heads);
}

// ---- pod-batch variants (SURVEY §8f-1): row b belongs to sequence b
__global__ void rope_qk_store_pods_kernel(float *q, const float *__restrict__ k, const float *__restrict__ v, uint32_t ld,
                                          uint32_t B, PodPtrs pods, uint32_t dim, uint32_t hd) {
    pdl_launch_dependents();
    pdl_wait();
    const uint32_t half = dim / 2;
    const size_t n = (size_t)half * B;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += stride) {
        const uint32_t pr = (uint32_t)(idx % half), b = (uint32_t)(idx / half);
        const uint32_t e = 2 * pr;
        const int i0 = (int)(e % hd);
        const uint32_t p = pods.pasts[b];
        double sn, cs;
        sincos((double)p * pow(10000.0, ((double)(-i0)) / (double)hd), &sn, &cs);
        float *qd = q + (size_t)b * ld + e;
        double x0 = (double)qd[0], x1 = (double)qd[1];
        qd[0] = (float)(__dsub_rn(__dmul_rn(x0, cs), __dmul_rn(x1, sn)));
        qd[1] = (float)(__dadd_rn(__dmul_rn(x0, sn), __dmul_rn(x1, cs)));
        const float *kd = k + (size_t)b * ld + e;
        x0 = (double)kd[0]; x1 = (double)kd[1];
        float2 kr;
        kr.x = (float)(__dsub_rn(__dmul_rn(x0, cs), __dmul_rn(x1, sn)));
        kr.y = (float)(__dadd_rn(__dmul_rn(x0, sn), __dmul_rn(x1, cs)));
        *reinterpret_cast<float2 *>(pods.K[b] + pods.layer_off + (size_t)p * dim + e) = kr;
        *reinterpret_cast<float2 *>(pods.V[b] + pods.layer_off + (size_t)p * dim + e) =
            *reinterpret_cast<const float2 *>(v + (size_t)b * ld + e);
    }
}
void rope_qk_store_pods(float *q, const float *k, const float *v, uint32_t ld, uint32_t B, const PodPtrs &pods, uint32_t dim,
                        uint32_t heads, cudaStream_t st) {
    const size_t n = (size_t)(dim / 2) * B;
    launch_pdl(rope_qk_store_pods_kernel, dim3(blocks_for(n, 128)), dim3(128), 0, st, q, k, v, ld, B, pods, dim, dim / heads);
}
__global__ void get_rows_pods_kernel(const float *__restrict__ table, uint32_t nc, const uint32_t *__restrict__ tokens,
                                     uint32_t row_stride, const uint32_t *__restrict__ step_dev, float *__restrict__ dst) {
    pdl_launch_dependents();
    pdl_wait();
    const uint32_t row = blockIdx.x;
    const size_t r = tokens[(size_t)row * row_stride + *step_dev];
    const float *src = table + r * nc;
    float *d = dst + (size_t)row * nc;
    for (uint32_t i = threadIdx.x * 4; i < nc; i += blockDim.x * 4)
        *reinterpret_cast<float4 *>(d + i) = *reinterpret_cast<const float4 *>(src + i);
}
void get_rows_pods(const float *table, uint32_t nc, const uint32_t *tokens, uint32_t row_stride, const uint32_t *step_dev,
                   uint32_t B, float *dst, cudaStream_t st) {
    LB_CHECK((nc & 3) == 0, "get_rows_pods: row length must be a multiple of 4");
    launch_pdl(get_rows_pods_kernel, dim3(B), dim3(256), 0, st, table, nc, tokens, row_stride, step_dev, dst);
}
__global__ void advance_pods_kernel(uint32_t *pasts, uint32_t *state, uint32_t B) {
    pdl_wait();
    if (threadIdx.x < B) pasts[threadIdx.x] += 1;
    if (threadIdx.x == 0) state[1] += 1;
}
void advance_pods(uint32_t *pasts, uint32_t *state, uint32_t B, cudaStream_t st) {
    launch_pdl(advance_pods_kernel, dim3(1), dim3(32), 0, st, pasts, state, B);
}

__global__ void get_rows_indirect_kernel(const float *__restrict__ table, uint32_t nc, const uint32_t *__restrict__ tokens,
                                         const uint32_t *__restrict__ step_dev, float *__restrict__ dst) {
    uint32_t row = blockIdx.x;
    pdl_launch_dependents();
    pdl_wait();
    size_t r = tokens[*step_dev + row];
    const float *src = table + r * nc;
    float *d = dst + (size_t)row * nc;
    for (uint32_t i = threadIdx.x * 4; i < nc; i += blockDim.x * 4)
        *reinterpret_cast<float4 *>(d + i) = *reinterpret_cast<const float4 *>(src + i);
}
void get_rows_indirect(const float *table, uint32_t nc, const uint32_t *tokens, const uint32_t *step_dev, uint32_t nr,
                       float *dst, cudaStream_t st) {
    LB_CHECK((nc & 3) == 0, "get_rows_indirect: row length must be a multiple of 4");
    launch_pdl(get_rows_indirect_kernel, dim3(nr), dim3(256), 0, st, table, nc, tokens, step_dev, dst);
}
__global__ void advance_state_kernel(uint32_t *state, uint32_t dp, uint32_t ds, uint32_t *seq) {
    pdl_wait();
    state[0] += dp;
    state[1] += ds;
    if (seq) *seq += 1;
}
void advance_state(uint32_t *state, uint32_t dp, uint32_t ds, cudaStream_t st, uint32_t *seq) {
    launch_pdl(advance_state_kernel, dim3(1), dim3(1), 0, st, state, dp, ds, seq);
}

// ---- greedy sampler on the device (SURVEY.md §8f-2): the reference's SampleTopPTopK at temp -> 0
// (pkg/llama/llama.go:455-707) degenerates to argmax of the repetition-penalised logits: every id present
// in the last-`ring_size` ring gets  l < 0 ? l*scale*penalty : l*scale/penalty  (FP32, in that order,
// llama.go:515-522; scale = float32(1/temp)).  One CTA: penalise + argmax (lowest index on ties), append the
// token to tokens[*step] for the next decode step and update the ring and its per-id presence counts.
__global__ void __launch_bounds__(1024) sample_greedy_kernel(const float *__restrict__ logits, uint32_t V, float scale,
                                                             float penalty, uint32_t *__restrict__ present,
                                                             uint32_t *__restrict__ ring, uint32_t ring_size,
                                                             uint32_t *__restrict__ ring_pos, uint32_t *__restrict__ tokens,
                                                             const uint32_t *__restrict__ state) {
    __shared__ float bv[32];
    __shared__ uint32_t bi[32];
    pdl_wait();
    float best = -INFINITY;
    uint32_t best_i = 0xFFFFFFFFu;
    for (uint32_t i = threadIdx.x; i < V; i += blockDim.x) {
        float l = __fmul_rn(logits[i], scale);
        if (present[i]) l = logits[i] < 0.0f ? __fmul_rn(l, penalty) : __fdiv_rn(l, penalty);
        if (l > best || (l == best && i < best_i)) { best = l; best_i = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, best, o);
        uint32_t oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (ov > best || (ov == best && oi < best_i)) { best = ov; best_i = oi; }
    }
    if ((threadIdx.x & 31) == 0) { bv[threadIdx.x >> 5] = best; bi[threadIdx.x >> 5] = best_i; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); w++)
            if (bv[w] > best || (bv[w] == best && bi[w] < best_i)) { best = bv[w]; best_i = bi[w]; }
        tokens[state[1]] = best_i;                 // consumed by the next single-token eval
        const uint32_t pos = *ring_pos;
        const uint32_t evict = ring[pos];
        if (present[evict]) present[evict]--;
        ring[pos] = best_i;
        present[best_i]++;
        *ring_pos = (pos + 1) % ring_size;
    }
}
void sample_greedy(const float *logits, uint32_t V, float scale, float penalty, uint32_t *present, uint32_t *ring,
                   uint32_t ring_size, uint32_t *ring_pos, uint32_t *tokens, const uint32_t *state, cudaStream_t st) {
    launch_pdl(sample_greedy_kernel, dim3(1), dim3(1024), 0, st, logits, V, scale, penalty, present, ring, ring_size, ring_pos, tokens, state);
}

// ---- synthetic weights: same integer recipe as llama.go_b200/synth.py (bit-identical)
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void init_random_kernel(float *__restrict__ dst, uint64_t count, uint64_t base, float mean, float sscale) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        uint64_t h = splitmix64(base + i);
        int s = (int)(h & 0xFFFF) + (int)((h >> 16) & 0xFFFF) + (int)((h >> 32) & 0xFFFF) + (int)(h >> 48);
        float t = __fmul_rn((float)(s - 131070), sscale);
        dst[i] = __fadd_rn(mean, t);
    }
}
void init_random(float *dst, uint64_t count, uint64_t seed, uint64_t tid, float mean, float sigma_scale, cudaStream_t st) {
    if (!count) return;
    uint64_t base = seed * 0x9E3779B97F4A7C15ull + tid * 0xD1B54A32D192ED03ull;
    init_random_kernel<<<148 * 8, 256, 0, st>>>(dst, count, base, mean, sigma_scale);
    LB_LAUNCH_CHECK();
}

__global__ void f16_to_f32_kernel(const __half *__restrict__ src, float *__restrict__ dst, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = __half2float(src[i]);
}
void f16_to_f32(const uint16_t *src, float *dst, size_t n, cudaStream_t st) {
    if (!n) return;
    f16_to_f32_kernel<<<blocks_for(n, 256), 256, 0, st>>>(reinterpret_cast<const __half *>(src), dst, n);
    LB_LAUNCH_CHECK();
}

// __float2half_rn rounds to nearest even with gradual underflow, exactly like numpy's float32 -> float16 cast
__global__ void f32_to_f16_kernel(const float *__restrict__ src, __half *__restrict__ dst, size_t n, unsigned *overflow) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    bool over = false;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float v = src[i];
        const __half h = __float2half_rn(v);
        over |= isfinite(v) && __hisinf(h);
        dst[i] = h;
    }
    if (over) atomicExch(overflow, 1u);
}
void f32_to_f16(const float *src, uint16_t *dst, size_t n, unsigned *overflow, cudaStream_t st) {
    if (!n) return;
    f32_to_f16_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, reinterpret_cast<__half *>(dst), n, overflow);
    LB_LAUNCH_CHECK();
}

}  // namespace k
}  // namespace lb
