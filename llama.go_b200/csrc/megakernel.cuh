// megakernel.cuh — device code shared by the persistent decode kernels: kernels_mega.cu, kernels_ring.cu,
// kernels_ring_q8.cu (single sequence) and kernels_mega_pods.cu, kernels_ring_pods.cu (pod batches).
// What differs between those kernels is the weight stream and the MulMat consumer; what is here is what they have in
// common: PTX wrappers, the grid barrier, the RoPE table, the split attention phase and the statistics of its merge.
// Functions that involve CTA barriers take the number of threads that reach them (NT: all warps of a register-fed
// kernel, the consumer warps of a ring kernel); the producer warp of a ring kernel never reaches one.
#pragma once
#include "common.cuh"

namespace lb {
namespace k {

// ---- PTX wrappers ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// named barrier 1 over the NT threads / barrier 2 + half over one half of them (the attention phase runs two items at a time)
template <int NT>
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); }
template <int NT>
__device__ __forceinline__ void hsync(int half) { asm volatile("bar.sync %0, %1;" ::"r"(2 + half), "n"(NT / 2) : "memory"); }
// L2 load of data other CTAs wrote during this launch
__device__ __forceinline__ float4 ldcg4(const float *p) { return __ldcg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done != 0;
}
// Wait for the phase `parity` of an mbarrier to complete.  try_wait suspends the thread in hardware for a bounded time;
// the spin counter only exists so that a pipeline bug traps after MAX_SPINS failed polls instead of hanging the GPU (no
// clock read per iteration: ncu r02n counted 3.5-6.5 % CS2R instructions in the ring kernels).  FAST_PATH: one poll
// before the loop.  backoff_ns: sleep between polls (polling burns issue slots and power, and 16 warps polling one
// mbarrier compete with the producer's and the copy engine's updates of it).
template <uint32_t MAX_SPINS, bool FAST_PATH = false>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t backoff_ns = 0) {
    if (FAST_PATH && mbar_try(bar, parity)) return;
    uint32_t spins = 0;
    while (!mbar_try(bar, parity)) {
        if (backoff_ns) __nanosleep(backoff_ns);
        if (++spins > MAX_SPINS) __trap();
    }
}
// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier (TMA engine, no tensor map)
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// ring entry and mbarrier phase parity of the next slot of a shared-memory ring (no division on the hot path: ncu r02n)
struct RingPos {
    uint32_t slot, phase;
    __device__ __forceinline__ void next(uint32_t n_slots) {
        if (++slot == n_slots) { slot = 0; phase ^= 1u; }
    }
};

// D(16x8, f32) += A(16x8, tf32, row) * B(8x8, tf32, col)
__device__ __forceinline__ void mma_tf32(float (&d)[4], float a0, float a1, float a2, float a3, float b0, float b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(__float_as_uint(a0)), "r"(__float_as_uint(a1)), "r"(__float_as_uint(a2)), "r"(__float_as_uint(a3)),
          "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}
// v - trunc_tf32(v): exact in FP32 (the tensor core reads only the upper 19 bits of an operand register)
__device__ __forceinline__ float tf32_lo(float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }
__device__ __forceinline__ float4 tf32_lo4(float4 v) { return make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)); }

// ---- fused pipeline-stage hand-off over NVLink peer memory (multi-GPU layer sharding, SURVEY 8e) ----------------
__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u32(unsigned *p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// spin (one thread) until *flag >= want; traps after ~10 s instead of hanging the GPU if the peer stage died
__device__ __forceinline__ void p2p_wait(const unsigned *flag, unsigned want) {
    const long long t0 = clock64();
    while (ld_acquire_sys_u32(flag) < want) {
        if (clock64() - t0 > 20000000000LL) __trap();
    }
}

// ---- grid barrier among the NT threads of every CTA: a monotonically increasing counter, zeroed before each launch.
// sys: this CTA's stores to a peer GPU are ordered before the hand-off flag; arrive (profiling aid): per-CTA arrival time.
template <int NT>
__device__ __forceinline__ void grid_barrier(unsigned *bar, unsigned &target, unsigned nctas, bool sys = false,
                                             unsigned long long *arrive = nullptr) {
    target += nctas;
    csync<NT>();
    if (threadIdx.x == 0) {
        if (arrive) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            arrive[blockIdx.x] = t;
        }
        if (sys) __threadfence_system();
        else __threadfence();
        atomicAdd(bar, 1u);
        const long long t0 = clock64();
        while (ld_acquire_u32(bar) < target) {
            if (clock64() - t0 > 4000000000LL) __trap();  // never hang the GPU on a scheduling bug
        }
        __threadfence();
    }
    csync<NT>();
}

// ---- RoPE table: cos, sin(past * 10000^(-2j/HD)), j < HD/2, in f64 (ComputeForwardRopeFP32's pow/cos/sin, ml.go:2307-2310)
template <int HD, typename SH>
__device__ __forceinline__ void rope_table(SH &sh, uint32_t past) {
    if (threadIdx.x < HD / 2) {
        double sn, c;
        sincos((double)past * pow(10000.0, ((double)(-(int)(2 * threadIdx.x))) / (double)HD), &sn, &c);
        sh.rope_cs[threadIdx.x][0] = c;
        sh.rope_cs[threadIdx.x][1] = sn;
    }
}

// ---- attention phase of one sequence: items (head, split); each CTA runs up to two items CONCURRENTLY, one per half of
// its NT threads (own named barrier), so the latency chain of an item is paid once per layer.  Per item: RoPE of q and,
// in the item that owns position `past`, of k; store k, v (ComputeForwardRopeFP32 ml.go:2253-2328; llama.go:274-297 — K
// is cached rotated); scores K·q * 1/sqrt(HD); the split's softmax statistics (m, l) to part_ml and its unnormalised
// P·V to part_o, merged in the next phase (merge_stats).  P: the kernel's parameters (dim, heads, splits, chunk_cap, qkv,
// part_o, part_ml); SH: its shared memory (rope_cs, fred, hbcast, pv); scores_all: 2 x chunk_cap floats.
template <int HD, int NT, typename P, typename SH>
__device__ __forceinline__ void attention_phase(const P &p, const MegaLayerHost &L, uint32_t past, SH &sh, float *scores_all) {
    constexpr int LANES = HD / 4;
    constexpr int HALF = NT / 2;
    constexpr int HW = HALF / 32;      // warps per half
    constexpr int KG = HALF / LANES;   // P·V key groups per half: thread (kg, dl) takes keys kg, kg + KG, ... for 4 dims
    constexpr int AU = 8;              // K rows per warp / V rows per thread in flight
    const int half = threadIdx.x / HALF, ht = threadIdx.x % HALF;
    const int hwarp = ht >> 5, lane = threadIdx.x & 31;
    const uint32_t dim = p.dim, S = p.splits, Tn = past + 1;
    const float scale = (float)(1.0 / sqrt((double)HD));  // f32(1/sqrt(dim/heads)), llama.go:306
    const uint32_t chunk = min((Tn + S - 1) / S, p.chunk_cap);
    const uint32_t items = p.heads * S;
    float *scores = scores_all + (size_t)half * p.chunk_cap;
    float4 *pv = sh.pv + half * HALF;
    const uint32_t kg = ht / LANES, dl = ht % LANES;
    for (uint32_t item = blockIdx.x * 2 + half; item < items; item += gridDim.x * 2) {
        const uint32_t h = item / S, sp = item % S;
        const uint32_t t0 = min(sp * chunk, Tn), t1 = min(t0 + chunk, Tn), nk = t1 - t0;
        float *Kh = L.Kc + (size_t)h * HD;
        float *Vh = L.Vc + (size_t)h * HD;
        float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (lane < LANES) {
            const float4 qr = ldcg4(p.qkv + (size_t)h * HD + lane * 4);
            const double c0 = sh.rope_cs[lane * 2][0], s0 = sh.rope_cs[lane * 2][1];
            const double c1 = sh.rope_cs[lane * 2 + 1][0], s1 = sh.rope_cs[lane * 2 + 1][1];
            qv.x = (float)(__dsub_rn(__dmul_rn((double)qr.x, c0), __dmul_rn((double)qr.y, s0)));
            qv.y = (float)(__dadd_rn(__dmul_rn((double)qr.x, s0), __dmul_rn((double)qr.y, c0)));
            qv.z = (float)(__dsub_rn(__dmul_rn((double)qr.z, c1), __dmul_rn((double)qr.w, s1)));
            qv.w = (float)(__dadd_rn(__dmul_rn((double)qr.z, s1), __dmul_rn((double)qr.w, c1)));
            if (hwarp == 0 && past >= t0 && past < t1) {
                const float4 kr = ldcg4(p.qkv + dim + (size_t)h * HD + lane * 4);
                float4 ko;
                ko.x = (float)(__dsub_rn(__dmul_rn((double)kr.x, c0), __dmul_rn((double)kr.y, s0)));
                ko.y = (float)(__dadd_rn(__dmul_rn((double)kr.x, s0), __dmul_rn((double)kr.y, c0)));
                ko.z = (float)(__dsub_rn(__dmul_rn((double)kr.z, c1), __dmul_rn((double)kr.w, s1)));
                ko.w = (float)(__dadd_rn(__dmul_rn((double)kr.z, s1), __dmul_rn((double)kr.w, c1)));
                *reinterpret_cast<float4 *>(Kh + (size_t)past * dim + lane * 4) = ko;
                *reinterpret_cast<float4 *>(Vh + (size_t)past * dim + lane * 4) = ldcg4(p.qkv + 2 * dim + (size_t)h * HD + lane * 4);
            }
        }
        hsync<NT>(half);  // the freshly stored K/V row is visible to this half (read back through L2)
        // scores (MulMat K·Q, Scale): warp w takes keys w, w+HW, ... (AU keys in flight: one HBM round trip for the 7B
        // chunk of <= 57 keys)
        for (uint32_t i = hwarp; i < nk; i += HW * AU) {
            float4 kk[AU];
#pragma unroll
            for (int u = 0; u < AU; u++) {
                const uint32_t ii = i + u * HW;
                kk[u] = (ii < nk && lane < LANES) ? ldcg4(Kh + (size_t)(t0 + ii) * dim + lane * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < AU; u++) {
                const uint32_t ii = i + u * HW;
                float dd = kk[u].x * qv.x;
                dd = fmaf(kk[u].y, qv.y, dd); dd = fmaf(kk[u].z, qv.z, dd); dd = fmaf(kk[u].w, qv.w, dd);
                dd = warp_sum(dd);
                if (lane == 0 && ii < nk) scores[ii] = __fmul_rn(dd, scale);
            }
        }
        // the first AU V rows of this thread do not depend on the scores: fetch them now, under the softmax
        float4 vf[AU];
#pragma unroll
        for (int u = 0; u < AU; u++) {
            const uint32_t key = kg + u * KG;
            vf[u] = key < nk ? ldcg4(Vh + (size_t)(t0 + key) * dim + dl * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        hsync<NT>(half);
        // local softmax statistics (SoftMax, ml.go:2472-2499, per split)
        float m = -INFINITY;
        for (uint32_t i = ht; i < nk; i += HALF) m = fmaxf(m, scores[i]);
        m = warp_max(m);
        if (lane == 0) sh.fred[half][hwarp] = m;
        hsync<NT>(half);
        if (ht == 0) {
            float t = sh.fred[half][0];
            for (int i = 1; i < HW; i++) t = fmaxf(t, sh.fred[half][i]);
            sh.hbcast[half] = t;
        }
        hsync<NT>(half);
        m = sh.hbcast[half];
        float l = 0.f;
        for (uint32_t i = ht; i < nk; i += HALF) {
            float e = (float)exp((double)__fsub_rn(scores[i], m));
            scores[i] = e;
            l += e;
        }
        l = warp_sum(l);
        hsync<NT>(half);
        if (lane == 0) sh.fred[half][hwarp] = l;
        hsync<NT>(half);
        if (ht == 0) {
            float t = 0.f;
            for (int i = 0; i < HW; i++) t += sh.fred[half][i];
            p.part_ml[((size_t)h * S + sp) * 2 + 0] = m;
            p.part_ml[((size_t)h * S + sp) * 2 + 1] = t;
        }
        // partial P·V: sequential over this thread's keys, then over the key groups (fixed order)
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (uint32_t base = 0; base < nk; base += KG * AU) {
            if (base) {
#pragma unroll
                for (int u = 0; u < AU; u++) {
                    const uint32_t key = base + kg + u * KG;
                    vf[u] = key < nk ? ldcg4(Vh + (size_t)(t0 + key) * dim + dl * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
#pragma unroll
            for (int u = 0; u < AU; u++) {
                const uint32_t key = base + kg + u * KG;
                if (key < nk) {
                    const float sc = scores[key];
                    acc.x = fmaf(vf[u].x, sc, acc.x); acc.y = fmaf(vf[u].y, sc, acc.y);
                    acc.z = fmaf(vf[u].z, sc, acc.z); acc.w = fmaf(vf[u].w, sc, acc.w);
                }
            }
        }
        pv[ht] = acc;  // [kg][dl]
        hsync<NT>(half);
        if (ht < HD) {
            const float *pvf = reinterpret_cast<const float *>(pv);
            float r = 0.f;
            for (int i = 0; i < KG; i++) r += pvf[i * HD + ht];
            p.part_o[((size_t)h * S + sp) * HD + ht] = r;
        }
        hsync<NT>(half);  // scores / pv buffers are reused by the next item of this half
    }
}

// ---- the same for a pod batch: items (pod, head, split), pod b at position p.pasts[b] with its own cache p.Kb[b] / p.Vb[b]
// (+ layer_off).  With S == 1 the normalised output goes straight to p.attn[pod][h*HD..]; with S > 1 the split
// partials go to part_ml / part_o.  P also provides B and attn; SH has one RoPE table per pod.
template <int HD, int NT, typename P, typename SH>
__device__ __forceinline__ void attention_pods(const P &p, size_t layer_off, SH &sh, float *scores_all) {
    constexpr int LANES = HD / 4;
    constexpr int HALF = NT / 2;
    constexpr int HW = HALF / 32;
    constexpr int KG = HALF / LANES;
    constexpr int AU = 8;
    const int half = threadIdx.x / HALF, ht = threadIdx.x % HALF;
    const int hwarp = ht >> 5, lane = threadIdx.x & 31;
    const uint32_t dim = p.dim, S = p.splits;
    const float scale = (float)(1.0 / sqrt((double)HD));  // f32(1/sqrt(dim/heads)), llama.go:306
    const uint32_t items = p.B * p.heads * S;
    float *scores = scores_all + (size_t)half * p.chunk_cap;
    float4 *pv = sh.pv + half * HALF;
    const uint32_t kg = ht / LANES, dl = ht % LANES;
    for (uint32_t item = blockIdx.x * 2 + half; item < items; item += gridDim.x * 2) {
        const uint32_t sp = item % S, bh = item / S, h = bh % p.heads, b = bh / p.heads;
        const uint32_t past = p.pasts[b], Tn = past + 1;
        const uint32_t chunk = min((Tn + S - 1) / S, p.chunk_cap);
        const uint32_t t0 = min(sp * chunk, Tn), t1 = min(t0 + chunk, Tn), nk = t1 - t0;
        float *Kh = p.Kb[b] + layer_off + (size_t)h * HD;
        float *Vh = p.Vb[b] + layer_off + (size_t)h * HD;
        const float *qkv = p.qkv + (size_t)b * 3 * dim;
        float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (lane < LANES) {
            const float4 qr = ldcg4(qkv + (size_t)h * HD + lane * 4);
            const double c0 = sh.rope_cs[b][lane * 2][0], s0 = sh.rope_cs[b][lane * 2][1];
            const double c1 = sh.rope_cs[b][lane * 2 + 1][0], s1 = sh.rope_cs[b][lane * 2 + 1][1];
            qv.x = (float)(__dsub_rn(__dmul_rn((double)qr.x, c0), __dmul_rn((double)qr.y, s0)));
            qv.y = (float)(__dadd_rn(__dmul_rn((double)qr.x, s0), __dmul_rn((double)qr.y, c0)));
            qv.z = (float)(__dsub_rn(__dmul_rn((double)qr.z, c1), __dmul_rn((double)qr.w, s1)));
            qv.w = (float)(__dadd_rn(__dmul_rn((double)qr.z, s1), __dmul_rn((double)qr.w, c1)));
            if (hwarp == 0 && past >= t0 && past < t1) {  // the item that owns position `past` stores the new K (rotated) and V rows
                const float4 kr = ldcg4(qkv + dim + (size_t)h * HD + lane * 4);
                float4 ko;
                ko.x = (float)(__dsub_rn(__dmul_rn((double)kr.x, c0), __dmul_rn((double)kr.y, s0)));
                ko.y = (float)(__dadd_rn(__dmul_rn((double)kr.x, s0), __dmul_rn((double)kr.y, c0)));
                ko.z = (float)(__dsub_rn(__dmul_rn((double)kr.z, c1), __dmul_rn((double)kr.w, s1)));
                ko.w = (float)(__dadd_rn(__dmul_rn((double)kr.z, s1), __dmul_rn((double)kr.w, c1)));
                *reinterpret_cast<float4 *>(Kh + (size_t)past * dim + lane * 4) = ko;
                *reinterpret_cast<float4 *>(Vh + (size_t)past * dim + lane * 4) = ldcg4(qkv + 2 * dim + (size_t)h * HD + lane * 4);
            }
        }
        hsync<NT>(half);
        for (uint32_t i = hwarp; i < nk; i += HW * AU) {
            float4 kk[AU];
#pragma unroll
            for (int u = 0; u < AU; u++) {
                const uint32_t ii = i + u * HW;
                kk[u] = (ii < nk && lane < LANES) ? ldcg4(Kh + (size_t)(t0 + ii) * dim + lane * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < AU; u++) {
                const uint32_t ii = i + u * HW;
                float dd = kk[u].x * qv.x;
                dd = fmaf(kk[u].y, qv.y, dd); dd = fmaf(kk[u].z, qv.z, dd); dd = fmaf(kk[u].w, qv.w, dd);
                dd = warp_sum(dd);
                if (lane == 0 && ii < nk) scores[ii] = __fmul_rn(dd, scale);
            }
        }
        float4 vf[AU];
#pragma unroll
        for (int u = 0; u < AU; u++) {
            const uint32_t key = kg + u * KG;
            vf[u] = key < nk ? ldcg4(Vh + (size_t)(t0 + key) * dim + dl * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        hsync<NT>(half);
        float m = -INFINITY;
        for (uint32_t i = ht; i < nk; i += HALF) m = fmaxf(m, scores[i]);
        m = warp_max(m);
        if (lane == 0) sh.fred[half][hwarp] = m;
        hsync<NT>(half);
        if (ht == 0) {
            float t = sh.fred[half][0];
            for (int i = 1; i < HW; i++) t = fmaxf(t, sh.fred[half][i]);
            sh.hbcast[half] = t;
        }
        hsync<NT>(half);
        m = sh.hbcast[half];
        float l = 0.f;
        for (uint32_t i = ht; i < nk; i += HALF) {
            float e = (float)exp((double)__fsub_rn(scores[i], m));
            scores[i] = e;
            l += e;
        }
        l = warp_sum(l);
        hsync<NT>(half);
        if (lane == 0) sh.fred[half][hwarp] = l;
        hsync<NT>(half);
        if (ht == 0) {
            float t = 0.f;
            for (int i = 0; i < HW; i++) t += sh.fred[half][i];
            sh.hbcast[half] = t;
            if (S > 1) {
                p.part_ml[((size_t)bh * S + sp) * 2 + 0] = m;
                p.part_ml[((size_t)bh * S + sp) * 2 + 1] = t;
            }
        }
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (uint32_t base = 0; base < nk; base += KG * AU) {
            if (base) {
#pragma unroll
                for (int u = 0; u < AU; u++) {
                    const uint32_t key = base + kg + u * KG;
                    vf[u] = key < nk ? ldcg4(Vh + (size_t)(t0 + key) * dim + dl * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
#pragma unroll
            for (int u = 0; u < AU; u++) {
                const uint32_t key = base + kg + u * KG;
                if (key < nk) {
                    const float sc = scores[key];
                    acc.x = fmaf(vf[u].x, sc, acc.x); acc.y = fmaf(vf[u].y, sc, acc.y);
                    acc.z = fmaf(vf[u].z, sc, acc.z); acc.w = fmaf(vf[u].w, sc, acc.w);
                }
            }
        }
        pv[ht] = acc;
        hsync<NT>(half);  // also publishes hbcast = l
        if (ht < HD) {
            const float *pvf = reinterpret_cast<const float *>(pv);
            float r = 0.f;
            for (int i = 0; i < KG; i++) r += pvf[i * HD + ht];
            if (S > 1) p.part_o[((size_t)bh * S + sp) * HD + ht] = r;
            else p.attn[(size_t)b * dim + (size_t)h * HD + ht] = __fmul_rn(r, __fdiv_rn(1.0f, sh.hbcast[half]));  // p = e * f32(1/sum), ml.go:2493-2499
        }
        hsync<NT>(half);
    }
}

// ---- statistics of the merge of the attention splits, for `groups` (heads, or pods x heads) of S splits each:
// sh.mrg_m/mrg_l[g * S + s] = (m_s, l_s) of part_ml, mrg_w[g * S + s] = w_s = expf(m_s - max_s m_s) (0 for an empty
// split), mrg_inv[g] = f32(1 / sum_s l_s w_s).  The caller then forms out = (sum_s O_s w_s) * mrg_inv.  (The split/merge
// is this engine's reassociation of the reference's single-pass softmax; the merge weights use the FP32 expf — an f64
// exp per lane and split measured 8 us per layer — while the softmax terms themselves keep the reference's f64 exp.)
// One thread per (group, split) and then per group, through shared memory: a per-lane loop "read m, l -> if l > 0 read
// O_s" is a chain of 2 dependent L2 round trips per split (9 splits cost ~5 us per layer).
template <int NT, typename P, typename SH>
__device__ __forceinline__ void merge_stats(const P &p, uint32_t groups, SH &sh) {
    const uint32_t S = p.splits, items = groups * S;
    for (uint32_t i = threadIdx.x; i < items; i += NT) {
        const float2 ml = __ldcg(reinterpret_cast<const float2 *>(p.part_ml) + i);
        sh.mrg_m[i] = ml.x;
        sh.mrg_l[i] = ml.y;
    }
    csync<NT>();
    for (uint32_t g = threadIdx.x; g < groups; g += NT) {
        float M = -INFINITY;
        for (uint32_t s = 0; s < S; s++) M = fmaxf(M, sh.mrg_m[g * S + s]);
        float Lsum = 0.f;
        for (uint32_t s = 0; s < S; s++) {
            const float l = sh.mrg_l[g * S + s];
            float wgt = 0.f;
            if (l > 0.f) {
                wgt = expf(__fsub_rn(sh.mrg_m[g * S + s], M));
                Lsum = fmaf(l, wgt, Lsum);
            }
            sh.mrg_w[g * S + s] = wgt;
        }
        sh.mrg_inv[g] = __fdiv_rn(1.0f, Lsum);
    }
    csync<NT>();
}

}  // namespace k
}  // namespace lb
