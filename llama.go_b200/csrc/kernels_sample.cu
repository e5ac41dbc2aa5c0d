// kernels_sample.cu — SampleTopPTopK on the device (pkg/llama/llama.go:455-707, SURVEY §8f-2).
//
// One CTA of 1024 threads on the context's logits (already in HBM: no 128 KB D2H per token, no O(V * ring)
// host scan, llama.go:501-527):
//   1. v[i] = logits[i] * scale, and for ids present in the last-N ring  v < 0 ? v * penalty : v / penalty
//      (FP32, in that order: llama.go:515-522; scale = float32(1/temp), :500), kept in shared memory;
//   2. the top-K by K rounds of block-wide arg-max (descending, ties -> lower id: the reference's sort.Slice
//      is unstable, :548-552, so any tie order is "the reference's");
//   3. thread 0 walks the K candidates exactly like the reference: p = f32(exp(f64(v - max))), f64 sum,
//      p /= f32(sum) (:579-599); top-p cut at the first cumsum >= topP with the FP32 sequential cumsum and the
//      renormalisation by f32(1/cumsum) (:614-629);
//   4. the pick (:658-673): argmax_i p_i * p_i * f_i * f_i with f_i = float32(Int63)/2^63.  The reference seeds
//      its generator with time.Now() (:655), so no implementation can reproduce its draws; here Int63 comes from
//      splitmix64(seed + i), i.e. the same formula with a caller-supplied seed.  The candidate set (ids and
//      probabilities after both cuts) is the parity target (tests/test_gpu_sample.py vs oracle.sample_candidates).
//
// sample_top_p_top_k_pods_kernel runs the same row sampler (one __device__ function) on B pods, one CTA each, and in the
// pods generate loop (pods.cpp PodBatch::generate) also keeps each pod's last-N ring and produced count on the device and
// writes the picked id straight into the next pod step's token buffer.
#include "common.cuh"
#include "kernels.cuh"

namespace lb {
namespace k {

constexpr int SMP_THREADS = 1024;

__device__ __forceinline__ uint64_t smp_splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// The whole sampler on one row of logits, run by all SMP_THREADS threads of a CTA; smem = dynamic shared memory of
// sample_top_p_top_k_smem(V, top_k) bytes: vals[V] | cand_val[K] | cand_id[K] | present bitmask[(V + 31) / 32].
// out_ids / out_probs (optional) receive the candidate set after both cuts.  Returns the picked id in thread 0 (and
// the candidate count in *n_cand there); the other threads' return value is meaningless.
__device__ __forceinline__ uint32_t sample_top_p_top_k_row(float *smp_smem, const float *__restrict__ logits, uint32_t V,
                                                           const uint32_t *last_n, uint32_t n_last, uint32_t top_k, float top_p,
                                                           float scale, float penalty, uint64_t seed, uint32_t *__restrict__ out_ids,
                                                           float *__restrict__ out_probs, uint32_t *n_cand) {
    float *vals = smp_smem;
    float *cand_val = vals + V;
    uint32_t *cand_id = reinterpret_cast<uint32_t *>(cand_val + top_k);
    uint32_t *present = cand_id + top_k;
    __shared__ float bv[32];
    __shared__ uint32_t bi[32];
    __shared__ uint32_t win;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t words = (V + 31) / 32;
    for (uint32_t i = threadIdx.x; i < words; i += SMP_THREADS) present[i] = 0u;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n_last; i += SMP_THREADS) {
        const uint32_t tkn = last_n[i];
        if (tkn < V) atomicOr(&present[tkn >> 5], 1u << (tkn & 31));
    }
    __syncthreads();
    float best = -INFINITY;
    uint32_t best_i = 0xFFFFFFFFu;
    for (uint32_t i = threadIdx.x; i < V; i += SMP_THREADS) {
        const float lg = logits[i];
        float l = __fmul_rn(lg, scale);
        if (present[i >> 5] >> (i & 31) & 1u) l = lg < 0.0f ? __fmul_rn(l, penalty) : __fdiv_rn(l, penalty);
        vals[i] = l;
        if (l > best || (l == best && i < best_i)) { best = l; best_i = i; }
    }
    for (uint32_t r = 0; r < top_k; r++) {
        float bvv = best;
        uint32_t bii = best_i;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bvv, o);
            const uint32_t oi = __shfl_xor_sync(0xffffffffu, bii, o);
            if (ov > bvv || (ov == bvv && oi < bii)) { bvv = ov; bii = oi; }
        }
        if (lane == 0) { bv[warp] = bvv; bi[warp] = bii; }
        __syncthreads();
        if (warp == 0) {
            bvv = bv[lane];
            bii = bi[lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bvv, o);
                const uint32_t oi = __shfl_xor_sync(0xffffffffu, bii, o);
                if (ov > bvv || (ov == bvv && oi < bii)) { bvv = ov; bii = oi; }
            }
            if (lane == 0) {
                cand_val[r] = bvv;
                cand_id[r] = bii;
                win = bii;
            }
        }
        __syncthreads();
        const uint32_t w = win;
        if (w != 0xFFFFFFFFu && (w % SMP_THREADS) == threadIdx.x) {   // the owner removes it and rescans its elements
            vals[w] = -INFINITY;
            best = -INFINITY;
            best_i = 0xFFFFFFFFu;
            for (uint32_t i = threadIdx.x; i < V; i += SMP_THREADS) {
                const float l = vals[i];
                if (l != -INFINITY && (l > best || (l == best && i < best_i))) { best = l; best_i = i; }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t n = top_k;
        const float maxl = cand_val[0];
        double sum = 0.0;
        for (uint32_t i = 0; i < n; i++) {
            const double pe = exp((double)__fsub_rn(cand_val[i], maxl));
            cand_val[i] = (float)pe;
            sum += pe;
        }
        const float fsum = (float)sum;
        for (uint32_t i = 0; i < n; i++) cand_val[i] = __fdiv_rn(cand_val[i], fsum);
        if (top_p < 1.0f) {
            float cumsum = 0.0f;
            for (uint32_t i = 0; i < n; i++) {
                cumsum = __fadd_rn(cumsum, cand_val[i]);
                if (cumsum >= top_p) { n = i + 1; break; }
            }
            cumsum = __fdiv_rn(1.0f, cumsum);
            for (uint32_t i = 0; i < n; i++) cand_val[i] = __fmul_rn(cand_val[i], cumsum);
        }
        uint32_t idx = 0;
        float maxp = 0.0f;
        for (uint32_t i = 0; i < n; i++) {
            if (out_ids) out_ids[i] = cand_id[i];
            if (out_probs) out_probs[i] = cand_val[i];
            const float f = __fmul_rn((float)(long long)(smp_splitmix64(seed + i) >> 1), 1.0842021724855044e-19f);  // float32(Int63) / 2^63
            const float pp = __fmul_rn(__fmul_rn(__fmul_rn(cand_val[i], cand_val[i]), f), f);                       // p*p*f*f, llama.go:660
            if (i == 0 || pp > maxp) { idx = i; maxp = pp; }                                                          // :663-670
        }
        *n_cand = n;
        return cand_id[idx];
    }
    return 0u;
}

__global__ void __launch_bounds__(SMP_THREADS)
sample_top_p_top_k_kernel(const float *__restrict__ logits, uint32_t V, const uint32_t *__restrict__ last_n, uint32_t n_last,
                          uint32_t top_k, float top_p, float scale, float penalty, uint64_t seed,
                          uint32_t *__restrict__ out_ids, float *__restrict__ out_probs, uint32_t *__restrict__ out_n_token) {
    extern __shared__ float smp_smem[];
    uint32_t n = 0;
    const uint32_t tok = sample_top_p_top_k_row(smp_smem, logits, V, last_n, n_last, top_k, top_p, scale, penalty, seed, out_ids,
                                                 out_probs, &n);
    if (threadIdx.x == 0) {
        out_n_token[0] = n;
        out_n_token[1] = tok;
    }
}

// One CTA per pod b on row b of the batch logits, the same row sampler.  last_n rows are n_last apart (in the generate
// loop they are the pods' rings, g.ring).  Pod b's seed is seeds[b] + g.produced[b] (seeds[b] without g.produced).  After
// the pick thread 0 stores the id into the optional outputs and, in the generate loop, into the ring, out[b][produced]
// and tokens[b * tok_stride + state[1]] — the input of the next pod step — with no host copy in between.
__global__ void __launch_bounds__(SMP_THREADS)
sample_top_p_top_k_pods_kernel(const float *__restrict__ logits, uint32_t V, const uint32_t *last_n, uint32_t n_last, uint32_t top_k,
                               float top_p, float scale, float penalty, const uint64_t *__restrict__ seeds, uint32_t *__restrict__ out_ids,
                               float *__restrict__ out_probs, uint32_t *__restrict__ out_n, uint32_t *__restrict__ out_tok,
                               PodSampleState g) {
    extern __shared__ float smp_smem[];
    const uint32_t b = blockIdx.x;
    const uint32_t produced = g.produced ? g.produced[b] : 0u;
    uint32_t n = 0;
    const uint32_t tok = sample_top_p_top_k_row(smp_smem, logits + (size_t)b * V, V, last_n + (size_t)b * n_last, n_last, top_k, top_p,
                                                 scale, penalty, seeds[b] + produced, out_ids ? out_ids + (size_t)b * top_k : nullptr,
                                                 out_probs ? out_probs + (size_t)b * top_k : nullptr, &n);
    if (threadIdx.x != 0) return;
    if (out_n) out_n[b] = n;
    if (out_tok) out_tok[b] = tok;
    if (g.ring) {                       // lastNTokens.Value = id; lastNTokens = lastNTokens.Next() (server.go:207-208)
        const uint32_t pos = g.ring_pos[b];
        g.ring[(size_t)b * n_last + pos] = tok;
        g.ring_pos[b] = pos + 1 == n_last ? 0u : pos + 1;
    }
    if (g.produced) {
        g.out[(size_t)b * g.out_stride + produced] = tok;
        g.produced[b] = produced + 1;
    }
    if (g.tokens) g.tokens[(size_t)b * g.tok_stride + g.state[1]] = tok;
}

size_t sample_top_p_top_k_smem(uint32_t V, uint32_t top_k) {
    return ((size_t)V + 2 * (size_t)top_k + (V + 31) / 32) * sizeof(float);
}

// checks shared by both launchers; returns float32(1.0 / temp), llama.go:500 (the Go constant expression is evaluated in
// float32 here too)
template <typename Kernel>
static float sample_prepare(Kernel kernel, uint32_t V, uint32_t top_k, float temp) {
    LB_CHECK(top_k >= 1 && top_k <= V, "SampleTopPTopK : topK must be in 1..vocab (the reference slices logitsID[:topK], llama.go:565)");
    LB_CHECK(temp > 0.f, "SampleTopPTopK : temp must be > 0 (the reference replaces 0 by 0.5, main.go:379-381)");
    LB_CHECK(sample_top_p_top_k_smem(V, top_k) <= 200 * 1024, "SampleTopPTopK : vocab + 2 topK floats must fit 200 KB of shared memory");
    static bool attr[64] = {};  // function attributes are per device (one table per kernel: one per instantiation)
    int dev = 0;
    LB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        LB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    return 1.0f / temp;
}

void sample_top_p_top_k(const float *logits, uint32_t V, const uint32_t *last_n_dev, uint32_t n_last, uint32_t top_k, float top_p,
                        float temp, float penalty, uint64_t seed, uint32_t *out_ids, float *out_probs, uint32_t *out_n_token,
                        cudaStream_t st) {
    const float scale = sample_prepare(sample_top_p_top_k_kernel, V, top_k, temp);
    sample_top_p_top_k_kernel<<<1, SMP_THREADS, sample_top_p_top_k_smem(V, top_k), st>>>(logits, V, last_n_dev, n_last, top_k, top_p,
                                                                                          scale, penalty, seed, out_ids, out_probs,
                                                                                          out_n_token);
    LB_LAUNCH_CHECK();
}

void sample_top_p_top_k_pods(const float *logits, uint32_t V, uint32_t B, const uint32_t *last_n_dev, uint32_t n_last, uint32_t top_k,
                             float top_p, float temp, float penalty, const uint64_t *seeds_dev, uint32_t *out_ids, float *out_probs,
                             uint32_t *out_n, uint32_t *out_tok, const PodSampleState &g, cudaStream_t st) {
    const float scale = sample_prepare(sample_top_p_top_k_pods_kernel, V, top_k, temp);
    sample_top_p_top_k_pods_kernel<<<B, SMP_THREADS, sample_top_p_top_k_smem(V, top_k), st>>>(
        logits, V, last_n_dev, n_last, top_k, top_p, scale, penalty, seeds_dev, out_ids, out_probs, out_n, out_tok, g);
    LB_LAUNCH_CHECK();
}

}  // namespace k
}  // namespace lb
