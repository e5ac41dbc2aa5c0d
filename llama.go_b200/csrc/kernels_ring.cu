// kernels_ring.cu — the single-token forward pass (llama.Eval with N = 1, pkg/llama/llama.go:211-426) as ONE
// persistent cooperative kernel whose weight stream never stops: a dedicated producer warp copies every weight
// this CTA will need, in schedule order, from HBM into a shared-memory ring with cp.async.bulk (the TMA copy
// engine, completion on mbarriers), and runs AHEAD of the 16 consumer warps — across rows, across phases,
// across the grid barriers and the attention phase.  Weights do not depend on anything computed in the launch,
// so the only thing that ever stops the stream is a full ring.
//
// Why (profiles/README.md): the register-fed megakernel (kernels_mega.cu) streams its four MulMat phases at ~7.0 TB/s
// but leaves HBM idle for ~11 us of grid barriers and ~4 us of attention per 137 us layer (0.905-0.914 of the
// measured-peak roofline); L2 prefetch hints around the barriers and a shared-memory head start of the next phase
// measured no gain or a loss (r02a, r02j).
//
// Version 3 (r02m).  Versions 1-2 gave every ring slot (one row, 16 KB) to ONE consumer warp and kept the activation
// vector in shared memory: a slot stayed occupied for the ~0.6 us a single warp needs to walk 16 KB, only 9 slots fit
// next to the 44 KB vector, and the kernel ended 3 % BEHIND the register-fed one (r02i/r02j: 215.8 vs 221.5 tok/s) — the
// ring was latency-bound: 9 x 16 KB / (HBM latency + 0.6 us) is no more than an SM's share of the HBM rate.  Now
//   * every slot is consumed by ALL 16 warps at once: warp w owns the fixed 1/16 slice of the slot's K range and keeps
//     that slice of the activation vector in REGISTERS for the whole phase (the register-fed kernel's decomposition),
//     reads its 1 KB of the row with two conflict-free LDS.128, and releases the slot (mbarrier count 16) ~50 ns after
//     the bytes have landed;
//   * no activation vector in shared memory: the ring is 12 x 16 KB = 192 KB per SM (4 us of stream);
//   * per-warp partial sums go through shared memory and are combined in a fixed order once per 32 rows (deterministic).
// Layout of the stream: a MulMat phase gives CTA c a contiguous block of ~0.8 M/148 output rows plus rows drawn from a
// ticket pool; one ring slot = one row (K <= 4096) or one K chunk of a longer row, filled by ONE bulk copy of up to
// 16 KB (1 KB copies were measured copy-engine bound at ~75 clk per copy: 4 TB/s, profiles/README.md r02f).
// Slot q lives in ring entry q % n; full[] (expect_tx + the copy's complete_tx) / empty[] (the 16 warps' arrivals).
// Numerics are those of kernels_mega.cu (f64 RMSNorm sums, f64 RoPE, f64 exp softmax terms, K-slice partial sums combined
// in warp order); only the chunking of K > 4096 rows differs in the association order of the FP32 dot products.
//
// F16 weights (WT = __half): the same kernel streams the binary16 matrices.  The K chunking stays 4096 ELEMENTS per slot
// (8 KB, so twice as many slots fit in the ring), and each lane reads the same elements as in the FP32 ring — two LDS.64
// instead of two LDS.128 — widens them exactly and issues the same FMAs in the same order: every product and partial sum
// equals the FP32 ring's on the widened weights, so the logits are bit-identical to an FP32 model holding those weights.
// The attention phase, grid barrier and PTX wrappers are shared with the other decode kernels (megakernel.cuh).
#include <cooperative_groups.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "kernels.cuh"
#include "megakernel.cuh"

namespace lb {
namespace k {
namespace {

constexpr int RG_CWARPS = 16;                      // consumer warps
constexpr int RG_CTHREADS = RG_CWARPS * 32;        // 512
constexpr int RG_THREADS = RG_CTHREADS + 32;       // + the producer warp
constexpr uint32_t RG_SLOT_FLOATS = 4096;          // one slot = one row (or a K chunk of a longer row) of <= 4096 weights: ONE bulk copy
template <typename WT> constexpr uint32_t RG_SLOT = RG_SLOT_FLOATS * sizeof(WT);   // 16 KB (FP32) / 8 KB (F16)
template <typename WT> constexpr int RG_MAX_SLOTS = sizeof(WT) == 4 ? 13 : 26;
constexpr int RG_GROUP = 32;                       // rows whose K-slice partials are combined per CTA barrier
constexpr int RG_MAX_PHASES = 4 * 160 + 1;        // MulMat phases of a launch: 4 per layer + lm_head
constexpr int RG_MAX_ITEMS = 2 * kNumSMs;
constexpr int RG_MAX_HEADS = 256;
// failed mbarrier polls before a trap: ~8 s at ~60 ns per poll, longer than any legitimate wait for a peer stage (p2p_wait
// traps after ~10 s)
constexpr uint32_t RG_MAX_SPINS = 1u << 27;

// 4 consecutive ring weights -> float4: FP32 (LDS.128) or binary16 (LDS.64, widened exactly)
template <typename WT>
__device__ __forceinline__ float4 lds_w4(uint32_t addr) {
    if constexpr (sizeof(WT) == 4) {
        return lds_f4(addr);
    } else {
        uint32_t a, b;
        asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "r"(addr));
        const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&a)), hi = __half22float2(*reinterpret_cast<const __half2 *>(&b));
        return make_float4(lo.x, lo.y, hi.x, hi.y);
    }
}
// a layer matrix of the element type the kernel streams
template <typename WT>
__device__ __forceinline__ const WT *wsel(const float *f32, const uint16_t *f16) {
    if constexpr (sizeof(WT) == 4) return f32;
    else return reinterpret_cast<const WT *>(f16);
}

struct RingParams {
    const MegaLayerHost *layers;
    uint32_t n_layers;
    const float *tok_embeddings;  // nullptr: the residual stream comes in through x
    const uint32_t *tokens;
    const uint32_t *state;        // {past, step}
    const float *final_norm, *output;  // nullptr: no lm_head on this stage
    const uint16_t *output_h;          // binary16 lm_head (F16 weights)
    float *x, *y, *qkv, *attn, *act, *logits;
    float *part_o, *part_ml;
    unsigned *barrier;
    uint32_t dim, ff, heads, vocab, ctx, splits, chunk_cap, n_slots;
    uint32_t spin_ns;             // consumers' back-off between polls of a slot's mbarrier (LB_RING_SPIN_NS)
    unsigned long long *trace;    // optional: 13 globaltimer stamps per layer written by consumer thread 0 of CTA 0 (+ per-CTA statistics of layer 5)
    // fused stage hand-off over NVLink peer memory (see MegaParamsHost)
    uint32_t *p2p_flags;          // local {in_flag, ack, seq}
    uint32_t p2p_wait_in;
    float *p2p_x_out;
    uint32_t *p2p_flag_out, *p2p_ack_out;
};

template <int NS>
struct RingShared {
    unsigned long long full[NS], empty[NS];
    unsigned jobrow[NS];  // the output row the slot's bytes belong to
    unsigned short done_jobs[RG_MAX_PHASES];   // jobs of MulMat phase i of this launch (0xFFFF: the producer has not finished it)
    float part[2][2][RG_GROUP][RG_CWARPS];     // [buffer][matrix (w1|w3)][row of the group][warp]
    unsigned grow[2][RG_GROUP];                // output rows of the group
    double red[RG_CWARPS];
    double rope_cs[64][2];
    float fred[2][RG_CWARPS / 2];
    float hbcast[2];
    float4 pv[RG_CTHREADS];
    float mrg_m[RG_MAX_ITEMS], mrg_l[RG_MAX_ITEMS], mrg_w[RG_MAX_ITEMS], mrg_inv[RG_MAX_HEADS];
};

// A row of K floats is streamed as NCH = ceil(K / 4096) chunks of CH floats (a multiple of 64: every warp's 1/16 slice of
// a chunk is whole float4s); the last chunk may be shorter.  Inside chunk c warp w owns floats [w * len_c / 16, (w + 1) * len_c / 16),
// lane l the float4s l and l + 32 of that slice (a slice is at most 256 floats).
__host__ __device__ __forceinline__ uint32_t ring_nch(uint32_t K) { return (K + RG_SLOT_FLOATS - 1) / RG_SLOT_FLOATS; }
__host__ __device__ __forceinline__ uint32_t ring_chunk(uint32_t K, uint32_t nch) { return (((K + nch - 1) / nch) + 63u) / 64u * 64u; }

// Work of a MulMat phase = "jobs", one per output row (its NCH chunks, both matrices of the SwiGLU pair).
// 4/5 of the rows are dealt out statically (CTA c: a contiguous block), the rest is a pool handed out a few rows per ticket
// (atomic counter per phase) — drawn by the PRODUCER as it runs ahead, two tickets in flight, the first two a few rows before
// the static block ends, so an SM that streams faster takes more rows and all CTAs reach the grid barrier within about a
// ticket of each other.  (r02k: drawing two tickets at the START of a phase handed the whole pool of a short phase to the
// first 128 CTAs to ask — wo and w2 ran as an UNBALANCED static split; r02o: one ticket at a time exposed the atomic's
// round trip, wo 13.6 us for 9.6 us of stream.)
// Every warp consumes every job, in issue order; the job's row number travels in sh.jobrow[]; the producer ends a phase by
// publishing its job count BEFORE it installs anything of the next phase.
constexpr unsigned RG_STATIC_NUM = 4, RG_STATIC_DEN = 5;
// rows per ticket: ~64 KB of stream (1.4 us of an SM's share; r02q: 4-row tickets of the w1|w3 pair = 128 KB left the CTAs up to
// 4.6 us apart at the barrier), at most 2 rows when a CTA has fewer than 48 rows in the phase
__device__ __forceinline__ uint32_t ticket_rows(uint32_t M, uint32_t K, uint32_t NM, uint32_t esz) {
    uint32_t t = 65536u / (K * esz * NM);
    t = t < 1u ? 1u : (t > 4u ? 4u : t);
    return (M / gridDim.x < 48u && t > 2u) ? 2u : t;
}

// ---------------------------------------------------------------------------------------------------------
// producer (one thread)
// ---------------------------------------------------------------------------------------------------------
template <typename WT, int NM, typename SH>
__device__ __forceinline__ void produce(const WT *W, const WT *W3, uint32_t K, uint32_t M, RingPos &q, uint32_t phidx, unsigned *ticket,
                                        uint32_t ring_base, SH &sh, uint32_t n_slots, unsigned long long *pstat = nullptr) {
    unsigned long long stall = 0;   // profiling aid (pstat != nullptr): ns this producer spent waiting for a free ring entry
    const uint32_t nch = ring_nch(K), CH = ring_chunk(K, nch);
    const uint32_t Q = (uint32_t)(((uint64_t)M * RG_STATIC_NUM) / (RG_STATIC_DEN * gridDim.x));   // static rows per CTA
    const uint32_t pool0 = Q * gridDim.x, TR = ticket_rows(M, K, NM, sizeof(WT));
    uint32_t njobs = 0;
    auto job = [&](uint32_t row) {
        for (uint32_t c = 0; c < nch; c++) {
            const uint32_t k0 = c * CH, len = min(CH, K - k0);
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const uint32_t slot = q.slot, ph = q.phase;
                const uint32_t fb = smem_u32(&sh.full[slot]);
                if (pstat) {
                    unsigned long long ta, tb;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ta));
                    mbar_wait<RG_MAX_SPINS, true>(smem_u32(&sh.empty[slot]), ph ^ 1);
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tb));
                    stall += tb - ta;
                } else {
                    mbar_wait<RG_MAX_SPINS, true>(smem_u32(&sh.empty[slot]), ph ^ 1);   // all 16 warps have read slot q - n_slots
                }
                *reinterpret_cast<volatile unsigned *>(&sh.jobrow[slot]) = row;
                __threadfence_block();
                mbar_expect_tx(fb, len * (uint32_t)sizeof(WT));
                bulk_g2s(ring_base + slot * RG_SLOT<WT>, (m == 0 ? W : W3) + (size_t)row * K + k0, len * (uint32_t)sizeof(WT), fb);
                q.next(n_slots);
            }
        }
        njobs++;
    };
    // (Measured and rejected, r02y: bringing the REST of the short wo phase — 16 of a CTA's 28 rows do not fit in the ring — into L2
    //  with cp.async.bulk.prefetch.L2 while the consumers are in the attention phase: 220.5 vs 223.1 tok/s, the wo phase no
    //  shorter (13.7 us), barrier 1 longer.  Third L2-prefetch experiment without a gain on this part: r02a, r02j, r02y.)
    // two tickets in flight (an L2 atomic round trip under load is ~1 us = 2-3 rows of stream), the first drawn ~8 rows and the
    // second ~4 rows before the static block ends — late enough that a CTA only takes tickets when it is about to need them
    const uint32_t r0 = blockIdx.x * Q, r1 = r0 + Q;
    const uint32_t e1 = Q > 8 ? r1 - 8 : r0, e2 = Q > 4 ? r1 - 4 : r0;
    unsigned ta = 0, tb = 0;
    if (Q == 0) { ta = atomicAdd(ticket, 1u); tb = atomicAdd(ticket, 1u); }
    for (uint32_t row = r0; row < r1; row++) {
        if (row == e1) ta = atomicAdd(ticket, 1u);
        if (row == e2) tb = atomicAdd(ticket, 1u);
        job(row);
    }
    while ((uint64_t)pool0 + (uint64_t)ta * TR < M) {
        const uint32_t rb = pool0 + ta * TR, re = min(M, rb + TR);
        ta = tb;
        tb = atomicAdd(ticket, 1u);                             // next ticket, overlapped with these rows' copies
        for (uint32_t row = rb; row < re; row++) job(row);
    }
    // end of phase: the job count for the consumers
    *reinterpret_cast<volatile unsigned short *>(&sh.done_jobs[phidx]) = (unsigned short)njobs;
    __threadfence_block();
    if (pstat) { pstat[blockIdx.x] = stall; pstat[4 * gridDim.x + blockIdx.x] = njobs; }
}

// ---------------------------------------------------------------------------------------------------------
// consumer: out[row] = epilogue(W[row] . x) for the rows this CTA's producer fetched; x: this warp's K-slices in registers
// (xs[c][v] = float4 (v * 32 + lane) of the warp's slice of chunk c).  EPI: 0 none, 1 + res[row];
// NM == 2: out[row] = silu(W1[row].x) * (W3[row].x)
// ---------------------------------------------------------------------------------------------------------
template <typename WT, int NM, int EPI, int NCH, typename SH>
__device__ __forceinline__ void consume(uint32_t K, const float4 (&xs)[NCH][2], float *out, const float *res, RingPos &q, uint32_t phidx,
                                        uint32_t ring_base, SH &sh, uint32_t n_slots, uint32_t spin_ns, bool peer_out = false) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t CH = ring_chunk(K, NCH);
    int buf = 0;
    uint32_t ingroup = 0, j = 0;
    auto combine = [&](uint32_t n) {
        csync<RG_CTHREADS>();
        if (threadIdx.x < n) {
            float s1 = 0.f, s3 = 0.f;
#pragma unroll
            for (int wv = 0; wv < RG_CWARPS; wv++) {
                s1 += sh.part[buf][0][threadIdx.x][wv];
                if (NM == 2) s3 += sh.part[buf][NM - 1][threadIdx.x][wv];
            }
            const uint32_t row = sh.grow[buf][threadIdx.x];
            float v;
            if (NM == 2) v = __fmul_rn(silu_ref(s1), s3);
            else if (EPI == 1) v = __fadd_rn(s1, __ldcg(res + row));
            else v = s1;
            out[row] = v;
            // out is the NEXT pipeline stage's buffer on another GPU: the WRITING thread orders its own store at system scope
            // (a fence by thread 0 after the CTA barrier does not cover other threads' stores still in flight over NVLink:
            //  r02r, logits 6e-3 off with the fence in the grid barrier only)
            if (peer_out) __threadfence_system();
        }
        buf ^= 1;   // the other buffer is written next; this one is reused only after the next csync
    };
    while (true) {
        // job j's first slot — or the end of the phase (the producer publishes the job count before it installs anything
        // of the next phase: a slot seen complete together with a published count <= j belongs to the NEXT phase)
        {
            const uint32_t fb = smem_u32(&sh.full[q.slot]);
            uint32_t spins = 0;
            bool over = false;
            while (true) {
                const bool got = mbar_try(fb, q.phase);
                const unsigned dj = *reinterpret_cast<volatile unsigned short *>(&sh.done_jobs[phidx]);
                if (dj != 0xFFFFu && j >= dj) { over = true; break; }
                if (got) break;
                if (spin_ns) __nanosleep(spin_ns);
                if (++spins > RG_MAX_SPINS) __trap();
            }
            if (over) break;
        }
        const uint32_t row = *reinterpret_cast<volatile unsigned *>(&sh.jobrow[q.slot]);
        float acc[NM];
#pragma unroll
        for (int m = 0; m < NM; m++) acc[m] = 0.f;
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            const uint32_t len = min(CH, K - (uint32_t)c * CH), sl16 = len / 16;   // floats of this warp's slice
            const bool v0 = (uint32_t)lane * 4 < sl16, v1 = (uint32_t)(lane + 32) * 4 < sl16;
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const uint32_t slot = q.slot;
                if (c | m) mbar_wait<RG_MAX_SPINS, true>(smem_u32(&sh.full[slot]), q.phase, spin_ns);
                const uint32_t base = ring_base + slot * RG_SLOT<WT> + ((uint32_t)warp * sl16 + (uint32_t)lane * 4) * (uint32_t)sizeof(WT);
                const float4 wa = v0 ? lds_w4<WT>(base) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float4 wb = v1 ? lds_w4<WT>(base + 128 * (uint32_t)sizeof(WT)) : make_float4(0.f, 0.f, 0.f, 0.f);
                float s = acc[m];
                s = fmaf(wa.x, xs[c][0].x, s); s = fmaf(wa.y, xs[c][0].y, s); s = fmaf(wa.z, xs[c][0].z, s); s = fmaf(wa.w, xs[c][0].w, s);
                s = fmaf(wb.x, xs[c][1].x, s); s = fmaf(wb.y, xs[c][1].y, s); s = fmaf(wb.z, xs[c][1].z, s); s = fmaf(wb.w, xs[c][1].w, s);
                acc[m] = s;
                __syncwarp();   // the FMAs above consumed every lane's loads: the slot may be refilled
                if (lane == 0) mbar_arrive(smem_u32(&sh.empty[slot]));
                q.next(n_slots);
            }
        }
#pragma unroll
        for (int m = 0; m < NM; m++) {
            const float a = warp_sum(acc[m]);
            if (lane == 0) sh.part[buf][m][ingroup][warp] = a;
        }
        if (threadIdx.x == 0) sh.grow[buf][ingroup] = row;
        j++;
        if (++ingroup == RG_GROUP) { combine(ingroup); ingroup = 0; }
    }
    if (ingroup) combine(ingroup);
}

// ---- this warp's K-slices of a phase's activation vector -> registers ------------------------------------------------
// element index of float4 (c, v) of this thread: c * CH + warp * len_c / 16 + (v * 32 + lane) * 4 (0xFFFFFFFF: past the slice)
template <int NCH>
__device__ __forceinline__ uint32_t slice_index(uint32_t K, uint32_t CH, int c, int v) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if ((uint32_t)c * CH >= K) return 0xFFFFFFFFu;
    const uint32_t len = min(CH, K - (uint32_t)c * CH), sl16 = len / 16, o = (uint32_t)(v * 32 + lane) * 4;
    return o < sl16 ? (uint32_t)c * CH + (uint32_t)warp * sl16 + o : 0xFFFFFFFFu;
}
// y = w * (x * f32(1/sqrt(mean_f64(x^2) + 1e-5)))   (ComputeForwardRMSNormFP32 + Mul, ml.go:1753-1812; llama.go:255-259)
// The 16 warps' slices tile x exactly once, so the slice a thread keeps is also its share of the sum of squares: one L2 round trip.
template <int NCH, typename SH>
__device__ __forceinline__ void fill_norm(float4 (&xs)[NCH][2], const float *x, const float *w, uint32_t K, SH &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t CH = ring_chunk(K, NCH);
    float4 ww[NCH][2];
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int v = 0; v < 2; v++) {
            const uint32_t e = slice_index<NCH>(K, CH, c, v);
            xs[c][v] = make_float4(0.f, 0.f, 0.f, 0.f);
            ww[c][v] = xs[c][v];
            if (e != 0xFFFFFFFFu) {
                xs[c][v] = ldcg4(x + e);
                ww[c][v] = __ldg(reinterpret_cast<const float4 *>(w + e));
            }
        }
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int v = 0; v < 2; v++) {
            acc += (double)__fmul_rn(xs[c][v].x, xs[c][v].x); acc += (double)__fmul_rn(xs[c][v].y, xs[c][v].y);
            acc += (double)__fmul_rn(xs[c][v].z, xs[c][v].z); acc += (double)__fmul_rn(xs[c][v].w, xs[c][v].w);
        }
    acc = warp_sum(acc);
    if (lane == 0) sh.red[warp] = acc;
    csync<RG_CTHREADS>();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < RG_CWARPS; i++) t += sh.red[i];
    const float sc = (float)(1.0 / sqrt(t / (double)K + 1e-5));
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int v = 0; v < 2; v++)
            xs[c][v] = make_float4(__fmul_rn(ww[c][v].x, __fmul_rn(xs[c][v].x, sc)), __fmul_rn(ww[c][v].y, __fmul_rn(xs[c][v].y, sc)),
                                   __fmul_rn(ww[c][v].z, __fmul_rn(xs[c][v].z, sc)), __fmul_rn(ww[c][v].w, __fmul_rn(xs[c][v].w, sc)));
    csync<RG_CTHREADS>();   // sh.red may be rewritten
}
template <int NCH>
__device__ __forceinline__ void fill_plain(float4 (&xs)[NCH][2], const float *x, uint32_t K) {
    const uint32_t CH = ring_chunk(K, NCH);
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int v = 0; v < 2; v++) {
            const uint32_t e = slice_index<NCH>(K, CH, c, v);
            xs[c][v] = e != 0xFFFFFFFFu ? ldcg4(x + e) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
}
// merge of the attention splits (see merge_stats, megakernel.cuh): out = (sum_s O_s w_s) * f32(1 / sum_s l_s w_s).
// The statistics are computed in line here, like the RoPE table in the kernel: through the shared functions this kernel's
// machine code changes (register allocation), while the other decode kernels compile to the same code either way.
template <int HD, int NCH, typename SH>
__device__ __forceinline__ void fill_merge(float4 (&xs)[NCH][2], const RingParams &p, SH &sh) {
    const uint32_t S = p.splits, items = p.heads * S, K = p.dim, CH = ring_chunk(K, NCH);
    for (uint32_t i = threadIdx.x; i < items; i += RG_CTHREADS) {
        const float2 ml = __ldcg(reinterpret_cast<const float2 *>(p.part_ml) + i);
        sh.mrg_m[i] = ml.x;
        sh.mrg_l[i] = ml.y;
    }
    csync<RG_CTHREADS>();
    for (uint32_t h = threadIdx.x; h < p.heads; h += RG_CTHREADS) {
        float M = -INFINITY;
        for (uint32_t s = 0; s < S; s++) M = fmaxf(M, sh.mrg_m[h * S + s]);
        float Lsum = 0.f;
        for (uint32_t s = 0; s < S; s++) {
            const float l = sh.mrg_l[h * S + s];
            float wgt = 0.f;
            if (l > 0.f) {
                wgt = expf(__fsub_rn(sh.mrg_m[h * S + s], M));
                Lsum = fmaf(l, wgt, Lsum);
            }
            sh.mrg_w[h * S + s] = wgt;
        }
        sh.mrg_inv[h] = __fdiv_rn(1.0f, Lsum);
    }
    csync<RG_CTHREADS>();
    constexpr int MB = 12;   // splits per batch of loads (a per-split loop of L2 reads costs one round trip per split)
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int v = 0; v < 2; v++) {
            const uint32_t e = slice_index<NCH>(K, CH, c, v);
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (e != 0xFFFFFFFFu) {
                const uint32_t h = e / HD, d = e % HD;
                const float *po = p.part_o + (size_t)h * S * HD + d;
                for (uint32_t s0 = 0; s0 < S; s0 += MB) {
                    float4 pv[MB];
#pragma unroll
                    for (int u = 0; u < MB; u++) pv[u] = s0 + u < S ? ldcg4(po + (size_t)(s0 + u) * HD) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int u = 0; u < MB; u++) {
                        if (s0 + u < S && sh.mrg_l[h * S + s0 + u] > 0.f) {
                            const float wgt = sh.mrg_w[h * S + s0 + u];
                            o.x = fmaf(pv[u].x, wgt, o.x); o.y = fmaf(pv[u].y, wgt, o.y);
                            o.z = fmaf(pv[u].z, wgt, o.z); o.w = fmaf(pv[u].w, wgt, o.w);
                        }
                    }
                }
                const float inv = sh.mrg_inv[h];
                o = make_float4(__fmul_rn(o.x, inv), __fmul_rn(o.y, inv), __fmul_rn(o.z, inv), __fmul_rn(o.w, inv));
            }
            xs[c][v] = o;
        }
}

// dynamic shared memory: [ring: n_slots x RG_SLOT][scores: 2 x chunk_cap floats][RingShared]
template <typename WT, int HD, int ND, int NF>
__global__ void __launch_bounds__(RG_THREADS, 1) decode_ring_kernel(const RingParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const uint32_t dim = p.dim, ff = p.ff, n_slots = p.n_slots;
    uint8_t *ring = smem_raw;
    float *scores = reinterpret_cast<float *>(smem_raw + (size_t)n_slots * RG_SLOT<WT>);
    RingShared<RG_MAX_SLOTS<WT>> &sh = *reinterpret_cast<RingShared<RG_MAX_SLOTS<WT>> *>(scores + 2 * (size_t)((p.chunk_cap + 3) & ~3u));
    const bool producer = threadIdx.x >= RG_CTHREADS;

    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < n_slots; s++) {
            mbar_init(smem_u32(&sh.full[s]), 1);
            mbar_init(smem_u32(&sh.empty[s]), RG_CWARPS);
        }
        for (int i = 0; i < RG_MAX_PHASES; i++) sh.done_jobs[i] = 0xFFFFu;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t past = p.state[0];
    if (threadIdx.x < HD / 2) {  // RoPE table of this token's position (f64 pow/cos/sin, ml.go:2307-2310)
        double sn, cs;
        sincos((double)past * pow(10000.0, ((double)(-(int)(2 * threadIdx.x))) / (double)HD), &sn, &cs);
        sh.rope_cs[threadIdx.x][0] = cs;
        sh.rope_cs[threadIdx.x][1] = sn;
    }
    __syncthreads();   // the only CTA-wide barrier: after it the producer warp and the consumers never meet again

    RingPos pos;        // the producer's next slot to fill / the consumers' next slot to read
    pos.slot = 0; pos.phase = 0;
    const uint32_t ring_base = smem_u32(ring);
    if (producer) {
        if (threadIdx.x != RG_CTHREADS) return;   // one thread drives the copy engine
        // ================= producer warp: the whole token's weights of this CTA, in schedule order =================
        unsigned *tk = p.barrier + 2;   // one ticket counter per MulMat phase of the launch (zeroed with the barrier)
        uint32_t phidx = 0;
        for (uint32_t li = 0; li < p.n_layers; li++) {
            const MegaLayerHost L = p.layers[li];
            // profiling aid: layer 5's producer wait time and job count per CTA and phase (after the 13 stamps per layer and the 5 x grid arrival stamps)
            unsigned long long *ps = (p.trace && li == 5 && p.n_layers > 6) ? p.trace + (size_t)p.n_layers * 13 + 5 * (size_t)gridDim.x : nullptr;
            produce<WT, 1>(wsel<WT>(L.wqkv, L.h_wqkv), (const WT *)nullptr, dim, 3 * dim, pos, phidx, tk + phidx, ring_base, sh, n_slots, ps); phidx++;
            produce<WT, 1>(wsel<WT>(L.wo, L.h_wo), (const WT *)nullptr, dim, dim, pos, phidx, tk + phidx, ring_base, sh, n_slots, ps ? ps + gridDim.x : nullptr); phidx++;
            produce<WT, 2>(wsel<WT>(L.w1, L.h_w1), wsel<WT>(L.w3, L.h_w3), dim, ff, pos, phidx, tk + phidx, ring_base, sh, n_slots, ps ? ps + 2 * gridDim.x : nullptr); phidx++;
            produce<WT, 1>(wsel<WT>(L.w2, L.h_w2), (const WT *)nullptr, ff, dim, pos, phidx, tk + phidx, ring_base, sh, n_slots, ps ? ps + 3 * gridDim.x : nullptr); phidx++;
        }
        if (p.final_norm) produce<WT, 1>(wsel<WT>(p.output, p.output_h), (const WT *)nullptr, dim, p.vocab, pos, phidx, tk + phidx, ring_base, sh, n_slots);
        return;
    }
    // ================= consumers =================
    unsigned target = 0;
    uint32_t phidx = 0;   // MulMat phase number (same sequence as the producer's)
    // Pipeline stage hand-off (multi-GPU layer sharding, SURVEY 8e) fused into this kernel: the upstream stage's kernel
    // stored the residual stream straight into this context's x over NVLink and then raised in_flag; the producer warp
    // above is already streaming this stage's weights while we wait.  Before this launch may overwrite the downstream
    // context's x (in its last phase) the downstream stage must have consumed the previous step: ack >= seq.
    unsigned p2p_seq = 0;
    if (p.p2p_flags) {
        p2p_seq = p.p2p_flags[2];
        if (threadIdx.x == 0) {
            if (p.p2p_wait_in) p2p_wait(p.p2p_flags + 0, p2p_seq + 1);
            if (p.p2p_x_out) p2p_wait(p.p2p_flags + 1, p2p_seq);
        }
        csync<RG_CTHREADS>();
    }
    const float *xin = p.x;
    if (p.tok_embeddings) xin = p.tok_embeddings + (size_t)p.tokens[p.state[1]] * dim;  // GetRows, llama.go:244
    unsigned long long *tr = (p.trace && blockIdx.x == 0 && threadIdx.x == 0) ? p.trace : nullptr;
    auto stamp = [&](uint32_t li, int i) {
        if (tr) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            tr[li * 13 + i] = t;
        }
    };
    auto arr = [&](uint32_t li, int b) -> unsigned long long * {   // profiling aid: arrival time of every CTA at each of layer 5's barriers
        return (p.trace && li == 5 && p.n_layers > 6) ? p.trace + (size_t)p.n_layers * 13 + (size_t)b * gridDim.x : nullptr;
    };
    for (uint32_t li = 0; li < p.n_layers; li++) {
        const MegaLayerHost L = p.layers[li];
        stamp(li, 0);
        {   // ---- P1: rmsnorm * attention_norm, [wq;wk;wv] (llama.go:255-265)
            float4 xs[ND][2];
            fill_norm<ND>(xs, xin, L.attention_norm, dim, sh);
            stamp(li, 1);
            consume<WT, 1, 0, ND>(dim, xs, p.qkv, nullptr, pos, phidx++, ring_base, sh, n_slots, p.spin_ns);
        }
        stamp(li, 2);
        grid_barrier<RG_CTHREADS>(p.barrier, target, gridDim.x, false, arr(li, 0));
        stamp(li, 3);
        // ---- P2: RoPE, KV store, split attention partials (llama.go:274-333)
        attention_phase<HD, RG_CTHREADS>(p, L, past, sh, scores);
        stamp(li, 4);
        grid_barrier<RG_CTHREADS>(p.barrier, target, gridDim.x, false, arr(li, 1));
        stamp(li, 5);
        {   // ---- P3: merge the attention splits, wo + residual (llama.go:336-340)
            float4 xs[ND][2];
            fill_merge<HD, ND>(xs, p, sh);
            consume<WT, 1, 1, ND>(dim, xs, p.y, xin, pos, phidx++, ring_base, sh, n_slots, p.spin_ns);
        }
        stamp(li, 6);
        grid_barrier<RG_CTHREADS>(p.barrier, target, gridDim.x, false, arr(li, 2));
        stamp(li, 7);
        {   // ---- P4: rmsnorm * ffn_norm, silu(w1.)*(w3.) (llama.go:346-361)
            float4 xs[ND][2];
            fill_norm<ND>(xs, p.y, L.ffn_norm, dim, sh);
            stamp(li, 8);
            consume<WT, 2, 0, ND>(dim, xs, p.act, nullptr, pos, phidx++, ring_base, sh, n_slots, p.spin_ns);
        }
        stamp(li, 9);
        grid_barrier<RG_CTHREADS>(p.barrier, target, gridDim.x, false, arr(li, 3));
        stamp(li, 10);
        {   // ---- P5: w2 + residual (llama.go:363-366); the stage's last layer writes the residual into the next stage's x
            float4 xf[NF][2];
            fill_plain<NF>(xf, p.act, ff);
            const bool to_peer = p.p2p_x_out != nullptr && li + 1 == p.n_layers;
            consume<WT, 1, 1, NF>(ff, xf, to_peer ? p.p2p_x_out : p.x, p.y, pos, phidx++, ring_base, sh, n_slots, p.spin_ns, to_peer);
        }
        stamp(li, 11);
        grid_barrier<RG_CTHREADS>(p.barrier, target, gridDim.x, p.p2p_x_out != nullptr && li + 1 == p.n_layers, arr(li, 4));
        stamp(li, 12);
        xin = p.x;
    }
    if (p.final_norm) {  // final norm + lm_head (llama.go:374-384)
        float4 xs[ND][2];
        fill_norm<ND>(xs, xin, p.final_norm, dim, sh);
        consume<WT, 1, 0, ND>(dim, xs, p.logits, nullptr, pos, phidx++, ring_base, sh, n_slots, p.spin_ns);
    }
    if (p.p2p_flags && blockIdx.x == 0 && threadIdx.x == 0) {
        // every CTA passed the last grid barrier (system-scope fences below) after storing its rows of the residual
        __threadfence_system();
        if (p.p2p_flag_out) st_release_sys_u32(p.p2p_flag_out + 0, p2p_seq + 1);   // downstream: your input for step seq+1 is there
        if (p.p2p_ack_out) st_release_sys_u32(p.p2p_ack_out + 1, p2p_seq + 1);     // upstream: I am done with what you sent for step seq+1
    }
}

template <typename WT, int HD, int ND, int NF>
static cudaError_t launch(const RingParams &p, size_t smem, cudaStream_t st) {
    static size_t attr[64] = {};  // function attributes are per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || attr[dev] < smem) {
        e = cudaFuncSetAttribute(decode_ring_kernel<WT, HD, ND, NF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = 227 * 1024;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs); cfg.blockDim = dim3(RG_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, decode_ring_kernel<WT, HD, ND, NF>, p);
}
// instantiated (chunks of dim, chunks of ff): (1,1) (1,2) test models — every head dim; (1,3) 7B, (2,4) 13B, (2,5) 30B, (2,6) 65B — head dim 128
static bool ring_variant(uint32_t dim, uint32_t ff, uint32_t hd) {
    const uint32_t nd = ring_nch(dim), nf = ring_nch(ff);
    if (nd == 1 && (nf == 1 || nf == 2)) return true;
    if (hd != 128) return false;
    return (nd == 1 && nf == 3) || (nd == 2 && (nf == 4 || nf == 5 || nf == 6));
}
template <typename WT, int HD>
static cudaError_t launch_small(const RingParams &p, uint32_t nf, size_t smem, cudaStream_t st) {
    return nf == 1 ? launch<WT, HD, 1, 1>(p, smem, st) : launch<WT, HD, 1, 2>(p, smem, st);
}
template <typename WT>
static cudaError_t launch_shape(const RingParams &p, uint32_t hd, uint32_t nd, uint32_t nf, size_t smem, cudaStream_t st) {
    if (nd == 1 && nf <= 2) return hd == 128 ? launch_small<WT, 128>(p, nf, smem, st) : hd == 64 ? launch_small<WT, 64>(p, nf, smem, st) : launch_small<WT, 32>(p, nf, smem, st);
    if (nd == 1) return launch<WT, 128, 1, 3>(p, smem, st);
    if (nf == 4) return launch<WT, 128, 2, 4>(p, smem, st);
    if (nf == 5) return launch<WT, 128, 2, 5>(p, smem, st);
    return launch<WT, 128, 2, 6>(p, smem, st);
}

static uint32_t ring_splits(uint32_t heads) {
    uint32_t s = (2 * kNumSMs) / heads;
    return s < 1 ? 1 : (s > 32 ? 32 : s);
}
// shared-memory plan: returns the number of ring slots (0 = does not fit)
template <typename WT>
static uint32_t ring_plan(uint32_t heads, uint32_t ctx, size_t *smem_out) {
    const uint32_t S = ring_splits(heads), chunk_cap = (ctx + S - 1) / S;
    const size_t fixed = 2 * (size_t)((chunk_cap + 3) & ~3u) * 4 + sizeof(RingShared<RG_MAX_SLOTS<WT>>) + 128;
    const size_t cap = 227 * 1024;
    if (fixed + 4 * (size_t)RG_SLOT<WT> > cap) return 0;
    uint32_t n = (uint32_t)((cap - fixed) / RG_SLOT<WT>);
    if (n > (uint32_t)RG_MAX_SLOTS<WT>) n = RG_MAX_SLOTS<WT>;
    if (smem_out) *smem_out = fixed - 128 + (size_t)n * RG_SLOT<WT>;
    return n;
}

}  // namespace

// layout query for the CPU tests: K -> out {chunks per row, floats per chunk}
void ring_layout_query(uint32_t K, uint32_t *out) {
    out[0] = ring_nch(K);
    out[1] = ring_chunk(K, out[0]);
}

bool decode_ring_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx) {
    if (heads == 0 || dim % heads || heads > (uint32_t)RG_MAX_HEADS) return false;
    if (((uint64_t)(ff > vocab ? ff : vocab) > 3ull * dim ? (ff > vocab ? ff : vocab) : 3ull * dim) >= 65535ull * kNumSMs / 2) return false;   // job counts are 16-bit
    const uint32_t hd = dim / heads;
    if (hd != 128 && hd != 64 && hd != 32) return false;
    if (dim % 64 || ff % 64) return false;             // every warp's 1/16 slice of a chunk is whole float4s; 16-byte bulk copies
    if (!ring_variant(dim, ff, hd)) return false;
    return ring_plan<float>(heads, ctx, nullptr) >= 4;   // (an F16 ring has slots of half the size: it fits wherever this does)
}

void decode_ring(const MegaParamsHost &h, cudaStream_t st) {
    LB_CHECK(decode_ring_supported(h.dim, h.ff, h.heads, h.vocab, h.ctx), "decode_ring: unsupported shape");
    RingParams p;
    p.layers = h.layers_dev;
    p.n_layers = h.n_layers;
    p.tok_embeddings = h.tok_embeddings; p.tokens = h.tokens; p.state = h.state;
    p.final_norm = h.final_norm; p.output = h.output; p.output_h = h.h_output;
    p.x = h.x; p.y = h.y; p.qkv = h.qkv; p.attn = h.attn; p.act = h.act; p.logits = h.logits;
    p.part_o = h.part_o; p.part_ml = h.part_ml; p.barrier = h.barrier;
    p.dim = h.dim; p.ff = h.ff; p.heads = h.heads; p.vocab = h.vocab; p.ctx = h.ctx;
    p.splits = ring_splits(h.heads);
    p.chunk_cap = (h.ctx + p.splits - 1) / p.splits;
    size_t smem = 0;
    p.n_slots = h.f16 ? ring_plan<__half>(h.heads, h.ctx, &smem) : ring_plan<float>(h.heads, h.ctx, &smem);
    if (const char *e = getenv("LB_RING_SLOTS")) {   // profiling aid: a shallower ring
        const uint32_t n = (uint32_t)atoi(e);
        if (n >= 2 && n < p.n_slots) { smem -= (size_t)(p.n_slots - n) * (h.f16 ? RG_SLOT<__half> : RG_SLOT<float>); p.n_slots = n; }
    }
    p.trace = reinterpret_cast<unsigned long long *>(h.trace);
    static const uint32_t spin_ns = getenv("LB_RING_SPIN_NS") ? (uint32_t)atoi(getenv("LB_RING_SPIN_NS")) : 50u;   // no effect on an un-capped box (r02q); fewer polls = less power under the 1 kW cap
    p.spin_ns = spin_ns;
    p.p2p_flags = h.p2p_flags; p.p2p_wait_in = h.p2p_wait_in ? 1u : 0u;
    p.p2p_x_out = h.p2p_x_out; p.p2p_flag_out = h.p2p_flag_out; p.p2p_ack_out = h.p2p_ack_out;
    LB_CUDA(cudaMemsetAsync(h.barrier, 0, sizeof(unsigned) * (3 + 4 * (size_t)h.n_layers), st));   // grid barrier + per-phase row tickets
    const uint32_t hd = h.dim / h.heads, nd = ring_nch(h.dim), nf = ring_nch(h.ff);
    LB_CUDA(h.f16 ? launch_shape<__half>(p, hd, nd, nf, smem, st) : launch_shape<float>(p, hd, nd, nf, smem, st));
    count_launch();
}

}  // namespace k
}  // namespace lb
