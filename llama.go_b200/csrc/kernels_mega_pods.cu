// kernels_mega_pods.cu — pod batching (SURVEY §8f-1, pkg/server/server.go:84-106, 151-175): ONE decode step
// of B <= 8 independent sequences ("pods": own KV cache, own position) as ONE persistent cooperative kernel
// that streams every weight exactly once for all B tokens.
//
// Same phase schedule as the single-sequence megakernel (kernels_mega.cu): per layer
//   P1 rmsnorm + [wq;wk;wv] | P2 RoPE + KV store + attention per (pod, head, split) | P3 wo + residual
//   P4 rmsnorm + w1,w3 + SiLU*mul | P5 w2 + residual         then final rmsnorm + lm_head,
// 148 CTAs x 12 warps, grid barriers between phases.  What changes is the MulMat: with B activation columns a
// CUDA-core GEMV needs 8 FMAs per weight plus a cross-lane reduction per (row, column) — the per-op B-column
// GEMV of round 1 reached 0.37 of the HBM roofline.  Here the B x 16-row x 16-k products run on the tensor
// cores, fed STRAIGHT FROM THE LOAD REGISTERS:
//   * mma.sync.m16n8k8 (tf32 in, f32 out): A = 16 weight rows x 8 k, B = 8 k x 8 pods.  Lane (g, t) of a warp
//     loads ONE float4 W[row g][16c + 4t .. +3] (and one of row g + 8) — 64 contiguous bytes per row and
//     instruction, 512 B per row per 8-deep ring — and uses its four values as the A fragments of two k-steps
//     (the k index inside a 16-float chunk is permuted identically for A and B, which a dot product does not
//     see).  No shared-memory staging of the weights, no transposition, no reduction shuffles.
//   * FP32 semantics by the 3xTF32 split in registers: hardware truncates the raw FP32 operand to TF32 (= hi);
//     lo = v - trunc(v) is exact; D += Whi*Xhi, Wlo*Xhi, Whi*Xlo in three separate accumulators (short chains,
//     small terms never meet the big sum inside the tensor core, whose accumulate truncates), added in FP32 RN.
//   * the B activation columns live in shared memory in fragment order ([chunk][pod][t] float4: one
//     conflict-free LDS.128 per chunk and lane); K-slices of a row are split over the CTA's 12 warps and
//     combined through shared memory in a fixed order (deterministic).
//   * weights are prefetched through a register ring that runs ahead across tile (and K-pass) boundaries, so
//     the HBM stream does not stop at the per-tile combine.
// K > 5632 (w2: K = ff) does not fit the 176 KB activation stage: its K axis is walked in passes with the
// next pass's columns arriving by cp.async behind the current pass's MMAs.
// Numerics of everything else (RMSNorm f64 sums, f64 RoPE, f64 exp softmax terms, FP32 sequential-order
// independent sums) are those of kernels_mega.cu / kernels_attn.cu.  The attention phase (attention_pods), merge
// statistics, grid barrier and PTX wrappers are shared with the other decode kernels (megakernel.cuh).
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"
#include "kernels.cuh"
#include "megakernel.cuh"

namespace lb {
namespace k {
namespace {

constexpr int PM_WARPS = 12;   // 384 threads -> 168 registers per thread: room for a 10-chunk weight ring per warp
constexpr int PM_THREADS = PM_WARPS * 32;
constexpr int PM_MAXB = 8;
#ifndef PM_U1
#define PM_U1 10  // ring depth (chunks in flight per warp) of the one-matrix phases
#endif
#ifndef PM_U2
#define PM_U2 5   // ... of the two-matrix (w1, w3) phase
#endif
constexpr uint32_t PM_XS_CHUNKS = 352;                 // chunks of 16 floats (x 8 pods) resident: K <= 5632
constexpr uint32_t PM_XS_F4 = PM_XS_CHUNKS * 32;       // float4 slots of the activation stage (176 KB)
constexpr uint32_t PM_PASS_CHUNKS = PM_XS_CHUNKS / 2;  // streamed phases: two buffers of 176 chunks
constexpr int PM_MAX_ITEMS = 2 * kNumSMs + 64;         // (pod, head, split) items whose statistics are merged
constexpr int PM_MAX_TILES = 8;                        // 16-row tiles of a CTA in a streamed (multi-pass) phase

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

using PodsLayer = MegaLayerHost;  // Kc/Vc unused here: every pod has its own cache (PodsParams::Kb/Vb + layer_off)
struct PodsParams {
    const PodsLayer *layers;
    uint32_t n_layers, B;
    const float *tok_embeddings;
    const uint32_t *tokens;   // [B][tok_stride]
    uint32_t tok_stride;
    const uint32_t *state;    // {unused, step}
    const uint32_t *pasts;    // [B] position of each pod's new token
    float *const *Kb;         // [B] base of pod b's K cache
    float *const *Vb;
    const float *final_norm, *output;
    float *x, *y, *qkv, *attn, *act, *logits;  // [B][dim] [B][dim] [B][3 dim] [B][dim] [B][ff] [B][vocab]
    float *part_o, *part_ml;                   // [B][H][S][hd], [B][H][S][2]
    unsigned *barrier;
    uint32_t dim, ff, heads, vocab, ctx, splits, chunk_cap;
};

struct PodsShared {
    union {
        float part[2][PM_WARPS][128];   // GEMV: per-warp partial 16 rows x 8 pods tiles (double-buffered; the
                                        // two-matrix SwiGLU phase uses [0] = w1, [1] = w3 with two barriers)
        float4 pv[PM_THREADS];          // attention: P·V partials per half
    };
    double rope_cs[PM_MAXB][64][2];     // cos, sin(past_b * 10000^(-2j/hd))
    double red[PM_WARPS][PM_MAXB];
    float acc[PM_MAX_TILES][128];       // streamed phases: running sums of the CTA's tiles across K passes
    float scale[PM_MAXB];               // RMSNorm scale per pod
    const float *xrow[PM_MAXB];         // residual-stream row of each pod entering the layer
    float fred[2][PM_WARPS / 2];
    float hbcast[2];
    float mrg_m[PM_MAX_ITEMS], mrg_l[PM_MAX_ITEMS], mrg_w[PM_MAX_ITEMS], mrg_inv[PM_MAX_ITEMS];
};

// ---------------------------------------------------------------------------------------------------------
// activation stage fills: xs[(chunk * 8 + pod) * 4 + t] = X[pod][16 chunk + 4 t .. + 3]   (pods >= B: zeros)
// ---------------------------------------------------------------------------------------------------------
// RMSNorm * w of B rows (ComputeForwardRMSNormFP32 + Mul, ml.go:1753-1812; llama.go:255-259): each thread owns
// the float4 slots f = tid, tid + 512, ... which all belong to pod (lane >> 2): raw values go to the stage,
// the f64 sums of squares are reduced (4 lanes, then the warps in fixed order), then the thread scales its
// own slots in place.
__device__ __forceinline__ void fill_norm(float4 *xs, const float *w, uint32_t K, uint32_t B, PodsShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, pod = lane >> 2, t = lane & 3;
    const uint32_t nf4 = K * 2;  // K/16 chunks x 32 slots
    const float *xr = pod < (int)B ? sh.xrow[pod] : nullptr;
    double acc = 0.0;
    for (uint32_t f = threadIdx.x; f < nf4; f += PM_THREADS) {
        const uint32_t kk = (f >> 5) * 16 + t * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (xr) v = ldcg4(xr + kk);
        xs[f] = v;
        acc += (double)__fmul_rn(v.x, v.x); acc += (double)__fmul_rn(v.y, v.y);
        acc += (double)__fmul_rn(v.z, v.z); acc += (double)__fmul_rn(v.w, v.w);
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (t == 0) sh.red[warp][pod] = acc;
    csync<PM_THREADS>();
    if (threadIdx.x < PM_MAXB) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < PM_WARPS; i++) s += sh.red[i][threadIdx.x];
        sh.scale[threadIdx.x] = (float)(1.0 / sqrt(s / (double)K + 1e-5));
    }
    csync<PM_THREADS>();
    const float sc = sh.scale[pod];
    for (uint32_t f = threadIdx.x; f < nf4; f += PM_THREADS) {
        const uint32_t kk = (f >> 5) * 16 + t * 4;
        const float4 v = xs[f];
        const float4 ww = __ldg(reinterpret_cast<const float4 *>(w + kk));
        xs[f] = make_float4(__fmul_rn(ww.x, __fmul_rn(v.x, sc)), __fmul_rn(ww.y, __fmul_rn(v.y, sc)),
                            __fmul_rn(ww.z, __fmul_rn(v.z, sc)), __fmul_rn(ww.w, __fmul_rn(v.w, sc)));
    }
    csync<PM_THREADS>();
}

// plain rows X[pod] = src + pod * ld (written earlier in this launch by other CTAs -> L2 loads)
__device__ __forceinline__ void fill_rows(float4 *xs, const float *src, uint32_t ld, uint32_t K, uint32_t B) {
    const int lane = threadIdx.x & 31, pod = lane >> 2, t = lane & 3;
    const uint32_t nf4 = K * 2;
    for (uint32_t f = threadIdx.x; f < nf4; f += PM_THREADS) {
        const uint32_t kk = (f >> 5) * 16 + t * 4;
        xs[f] = pod < (int)B ? ldcg4(src + (size_t)pod * ld + kk) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    csync<PM_THREADS>();
}

// merge of the attention splits straight into the stage (S > 1): out = (sum_s O_s w_s) * f32(1 / sum_s l_s w_s),
// w_s = expf(m_s - max_s m_s) — the same reassociation of the single-pass softmax as kernels_mega.cu.
template <int HD>
__device__ __forceinline__ void fill_merge(float4 *xs, const PodsParams &p, PodsShared &sh) {
    const uint32_t S = p.splits;
    merge_stats<PM_THREADS>(p, p.B * p.heads, sh);
    const int lane = threadIdx.x & 31, pod = lane >> 2, t = lane & 3;
    const uint32_t nf4 = p.dim * 2;
    for (uint32_t f = threadIdx.x; f < nf4; f += PM_THREADS) {
        const uint32_t kk = (f >> 5) * 16 + t * 4;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (pod < (int)p.B) {
            const uint32_t h = kk / HD, d = kk % HD, bh = pod * p.heads + h;
            const float *po = p.part_o + (size_t)bh * S * HD + d;
            for (uint32_t s = 0; s < S; s++) {
                if (sh.mrg_l[bh * S + s] > 0.f) {
                    const float4 pv = ldcg4(po + (size_t)s * HD);
                    const float wgt = sh.mrg_w[bh * S + s];
                    o.x = fmaf(pv.x, wgt, o.x); o.y = fmaf(pv.y, wgt, o.y);
                    o.z = fmaf(pv.z, wgt, o.z); o.w = fmaf(pv.w, wgt, o.w);
                }
            }
            const float inv = sh.mrg_inv[bh];
            o.x = __fmul_rn(o.x, inv); o.y = __fmul_rn(o.y, inv); o.z = __fmul_rn(o.z, inv); o.w = __fmul_rn(o.w, inv);
        }
        xs[f] = o;
    }
    csync<PM_THREADS>();
}

// one K pass of a streamed phase: chunks [c0, c1) of src rows -> buffer `dst` by cp.async (16 B per slot)
__device__ __forceinline__ void stream_pass(float4 *dst, const float *src, uint32_t ld, uint32_t c0, uint32_t c1, uint32_t B) {
    const int lane = threadIdx.x & 31, pod = lane >> 2, t = lane & 3;
    const uint32_t nf4 = (c1 - c0) * 32;
    for (uint32_t f = threadIdx.x; f < nf4; f += PM_THREADS) {
        const uint32_t kk = (c0 + (f >> 5)) * 16 + t * 4;
        if (pod < (int)B) cp_async16(dst + f, src + (size_t)pod * ld + kk);
        else dst[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---------------------------------------------------------------------------------------------------------
// The MulMat phase.  out[pod][r] = epilogue( sum_k W[r][k] X[pod][k] ) for the CTA's rows [r_begin, r_end),
// NM = 2: out = silu(W1·x) * (W3·x).  EPI: 0 none, 1 + residual rows (res + pod * ldr, or sh.xrow when res == 0).
//   npass == 1: the activation stage already holds all K columns (filled by the caller).
//   npass  > 1: columns come from `xsrc` ([B][K] in global memory) pass by pass through the two half buffers.
// Work of one warp: for pass, for tile (16 rows), for its chunk sub-range of the pass — walked by two cursors,
// the load cursor U chunks ahead of the MMA cursor (register ring), across tile and pass boundaries.
// ---------------------------------------------------------------------------------------------------------
template <int NM, int U, int EPI>
__device__ __forceinline__ void gemv_pods(const float *__restrict__ W1, const float *__restrict__ W3, uint32_t K,
                                          uint32_t r_begin, uint32_t r_end, uint32_t npass, const float *xsrc, uint32_t ldx,
                                          float *out, uint32_t ldo, const float *res, uint32_t ldr, uint32_t B,
                                          float4 *xs, PodsShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const uint32_t CT = K / 16;                                // chunks along K
    const uint32_t NT = (r_end - r_begin + 15) / 16;           // 16-row tiles of this CTA
    auto pass_c0 = [&](uint32_t p) { return (uint32_t)(((uint64_t)CT * p) / npass); };
    if (npass > 1) {  // first two passes on their way before anything else
        stream_pass(xs, xsrc, ldx, pass_c0(0), pass_c0(1), B);
        cp_async_wait_all();
        csync<PM_THREADS>();
        stream_pass(xs + PM_XS_F4 / 2, xsrc, ldx, pass_c0(1), pass_c0(2), B);
    }
    if (NT == 0) {  // (cannot happen for M >= gridDim.x; keeps the barrier counts consistent if it does)
        for (uint32_t p = 0; p + 1 < npass; p++) {
            cp_async_wait_all();
            csync<PM_THREADS>();
            if (p + 2 < npass) stream_pass(xs + (p & 1) * (PM_XS_F4 / 2), xsrc, ldx, pass_c0(p + 2), pass_c0(p + 3), B);
        }
        return;
    }
    const ptrdiff_t d13 = NM == 2 ? W3 - W1 : 0;

    // ---- the two cursors over (pass, tile, chunk): `cb`/`cn` = first chunk / chunk count of this warp in the pass
    struct Cur { uint32_t p, j, left, cb, cn; };
    auto enter_pass = [&](Cur &cu) {      // cu.p set: this warp's chunk sub-range of the pass
        const uint32_t a = pass_c0(cu.p), b = pass_c0(cu.p + 1);
        cu.cb = a + (uint32_t)(((uint64_t)(b - a) * warp) / PM_WARPS);
        cu.cn = a + (uint32_t)(((uint64_t)(b - a) * (warp + 1)) / PM_WARPS) - cu.cb;
    };
    // load cursor
    Cur lc;
    lc.p = 0; lc.j = 0;
    enter_pass(lc);
    lc.left = lc.cn;
    const float *lpa, *lpb;   // rows (tile base + g) and (+ 8) of W1 at this warp's next chunk
    bool lva, lvb;
    auto load_tile = [&]() {
        const uint32_t ra = r_begin + lc.j * 16 + g, rb = ra + 8;
        lva = lc.p < npass && ra < r_end;
        lvb = lc.p < npass && rb < r_end;
        lpa = W1 + (size_t)ra * K + (size_t)lc.cb * 16 + t * 4;
        lpb = lpa + (size_t)8 * K;
    };
    load_tile();
    float4 ring[U][NM][2];
    auto load = [&](float4 (&dst)[NM][2]) {
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        dst[0][0] = lva ? ld_stream_f4(lpa) : z;
        dst[0][1] = lvb ? ld_stream_f4(lpb) : z;
        if (NM == 2) {
            dst[NM - 1][0] = lva ? ld_stream_f4(lpa + d13) : z;
            dst[NM - 1][1] = lvb ? ld_stream_f4(lpb + d13) : z;
        }
        lpa += 16; lpb += 16;
        if (--lc.left == 0 && lc.p < npass) {
            if (++lc.j == NT) {
                lc.j = 0;
                if (++lc.p < npass) enter_pass(lc);
            }
            lc.left = lc.cn;
            load_tile();
        }
    };
#pragma unroll
    for (int u = 0; u < U; u++) load(ring[u]);

    // MMA cursor
    Cur mc;
    mc.p = 0; mc.j = 0;
    enter_pass(mc);
    mc.left = mc.cn;
    uint32_t xi = (mc.cb - pass_c0(0)) * 32 + lane;   // slot of this lane's activation float4 for the next chunk
    float hh[NM][4], lh[NM][4], hl[NM][4];
#pragma unroll
    for (int m = 0; m < NM; m++)
#pragma unroll
        for (int i = 0; i < 4; i++) hh[m][i] = lh[m][i] = hl[m][i] = 0.f;
    int buf = 0;

    while (mc.p < npass) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            if (mc.p < npass) {
                // ---- MMAs of one chunk: 16 rows x 16 k x 8 pods, 3xTF32
                asm volatile("" ::: "memory");  // keep the chunks in program order: hoisted LDS/splits of later chunks only cost registers
                const float4 xv = xs[xi];
                xi += 32;
                const float4 xl = tf32_lo4(xv);
#pragma unroll
                for (int m = 0; m < NM; m++) {
                    const float4 wa = ring[u][m][0], wb = ring[u][m][1];
                    const float4 wal = tf32_lo4(wa), wbl = tf32_lo4(wb);
                    mma_tf32(hh[m], wa.x, wb.x, wa.y, wb.y, xv.x, xv.y);
                    mma_tf32(lh[m], wal.x, wbl.x, wal.y, wbl.y, xv.x, xv.y);
                    mma_tf32(hl[m], wa.x, wb.x, wa.y, wb.y, xl.x, xl.y);
                    mma_tf32(hh[m], wa.z, wb.z, wa.w, wb.w, xv.z, xv.w);
                    mma_tf32(lh[m], wal.z, wbl.z, wal.w, wbl.w, xv.z, xv.w);
                    mma_tf32(hl[m], wa.z, wb.z, wa.w, wb.w, xl.z, xl.w);
                }
                load(ring[u]);  // refill this ring slot U chunks ahead
                if (--mc.left == 0) {
                    // ---- this warp's K-slice of tile (mc.p, mc.j) is complete: publish, combine across the warps
                    const uint32_t tj = mc.j, tp = mc.p;
                    const bool last_tile_of_pass = tj + 1 == NT;
                    const bool last_pass = tp + 1 == npass;
#pragma unroll
                    for (int m = 0; m < NM; m++) {
                        float *pw = sh.part[NM == 2 ? m : buf][warp];
                        const float d0 = __fadd_rn(hh[m][0], __fadd_rn(lh[m][0], hl[m][0])), d1 = __fadd_rn(hh[m][1], __fadd_rn(lh[m][1], hl[m][1]));
                        const float d2 = __fadd_rn(hh[m][2], __fadd_rn(lh[m][2], hl[m][2])), d3 = __fadd_rn(hh[m][3], __fadd_rn(lh[m][3], hl[m][3]));
                        *reinterpret_cast<float2 *>(pw + g * 8 + 2 * t) = make_float2(d0, d1);         // (row g,     pods 2t, 2t+1)
                        *reinterpret_cast<float2 *>(pw + (g + 8) * 8 + 2 * t) = make_float2(d2, d3);   // (row g + 8, pods 2t, 2t+1)
#pragma unroll
                        for (int i = 0; i < 4; i++) hh[m][i] = lh[m][i] = hl[m][i] = 0.f;
                    }
                    if (npass > 1 && last_tile_of_pass && !last_pass) cp_async_wait_all();  // next pass's columns (this thread's share)
                    csync<PM_THREADS>();
                    if (threadIdx.x < 128) {
                        const uint32_t row = r_begin + tj * 16 + (threadIdx.x >> 3), pod = threadIdx.x & 7;
                        float s1 = 0.f, s3 = 0.f;
#pragma unroll
                        for (int wv = 0; wv < PM_WARPS; wv++) {
                            s1 += sh.part[NM == 2 ? 0 : buf][wv][threadIdx.x];
                            if (NM == 2) s3 += sh.part[1][wv][threadIdx.x];
                        }
                        if (npass > 1) {
                            if (tp > 0) s1 = __fadd_rn(sh.acc[tj][threadIdx.x], s1);
                            if (!last_pass) sh.acc[tj][threadIdx.x] = s1;
                        }
                        if (last_pass && row < r_end && pod < B) {
                            float v;
                            if (NM == 2) v = __fmul_rn(silu_ref(s1), s3);
                            else if (EPI == 1) v = __fadd_rn(s1, __ldcg((res ? res + (size_t)pod * ldr : sh.xrow[pod]) + row));
                            else v = s1;
                            out[(size_t)pod * ldo + row] = v;
                        }
                    }
                    if (NM == 2) csync<PM_THREADS>();   // single-buffered partials in the two-matrix phase
                    else buf ^= 1;
                    if (npass > 1 && last_tile_of_pass && tp + 2 < npass)  // buffer (tp & 1) is free now: stream pass tp + 2 into it
                        stream_pass(xs + (tp & 1) * (PM_XS_F4 / 2), xsrc, ldx, pass_c0(tp + 2), pass_c0(tp + 3), B);
                    // next tile / pass of the MMA cursor
                    if (++mc.j == NT) {
                        mc.j = 0;
                        if (++mc.p < npass) enter_pass(mc);
                    }
                    mc.left = mc.cn;
                    if (mc.p < npass) xi = (npass > 1 ? (mc.p & 1) * (PM_XS_F4 / 2) : 0) + (mc.cb - pass_c0(mc.p)) * 32 + lane;
                }
            }
        }
    }
}

__device__ __forceinline__ void cta_rows(uint32_t M, uint32_t &r0, uint32_t &r1) {
    r0 = (uint32_t)(((uint64_t)M * blockIdx.x) / gridDim.x);
    r1 = (uint32_t)(((uint64_t)M * (blockIdx.x + 1)) / gridDim.x);
}

template <int HD>
__global__ void __launch_bounds__(PM_THREADS, 1) decode_mega_pods_kernel(const PodsParams p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float4 *xs = reinterpret_cast<float4 *>(smem_raw);                                   // activation stage (176 KB)
    PodsShared &sh = *reinterpret_cast<PodsShared *>(smem_raw + (size_t)PM_XS_F4 * 16);
    float *scores = reinterpret_cast<float *>(smem_raw);                                 // attention overlays the stage
    const uint32_t dim = p.dim, ff = p.ff, B = p.B;
    unsigned target = 0;
    // RoPE tables of the B positions (ComputeForwardRopeFP32's pow/cos/sin in f64, ml.go:2307-2310)
    for (uint32_t i = threadIdx.x; i < B * 64; i += PM_THREADS) {
        const uint32_t b = i / 64, j = i % 64;
        if (j < HD / 2) {
            double sn, cs;
            sincos((double)p.pasts[b] * pow(10000.0, ((double)(-(int)(2 * j))) / (double)HD), &sn, &cs);
            sh.rope_cs[b][j][0] = cs;
            sh.rope_cs[b][j][1] = sn;
        }
    }
    if (threadIdx.x < PM_MAXB)
        sh.xrow[threadIdx.x] = threadIdx.x < B ? p.tok_embeddings + (size_t)p.tokens[(size_t)threadIdx.x * p.tok_stride + p.state[1]] * dim
                                                 : nullptr;  // GetRows, llama.go:244
    csync<PM_THREADS>();
    const uint32_t np_ff = (ff / 16 + PM_PASS_CHUNKS - 1) / PM_PASS_CHUNKS;  // K passes of the w2 phase
    uint32_t r0, r1;
    for (uint32_t li = 0; li < p.n_layers; li++) {
        const PodsLayer L = p.layers[li];
        const size_t layer_off = (size_t)li * p.ctx * dim;
        // ---- P1: rmsnorm * attention_norm, [wq;wk;wv] (llama.go:255-265)
        fill_norm(xs, L.attention_norm, dim, B, sh);
        cta_rows(3 * dim, r0, r1);
        gemv_pods<1, PM_U1, 0>(L.wqkv, nullptr, dim, r0, r1, 1, nullptr, 0, p.qkv, 3 * dim, nullptr, 0, B, xs, sh);
        grid_barrier<PM_THREADS>(p.barrier, target, gridDim.x);
        // ---- P2: RoPE, KV store, attention (llama.go:274-333)
        attention_pods<HD, PM_THREADS>(p, layer_off, sh, scores);
        grid_barrier<PM_THREADS>(p.barrier, target, gridDim.x);
        // ---- P3: wo + residual (llama.go:336-340)
        if (p.splits > 1) fill_merge<HD>(xs, p, sh);
        else fill_rows(xs, p.attn, dim, dim, B);
        cta_rows(dim, r0, r1);
        gemv_pods<1, PM_U1, 1>(L.wo, nullptr, dim, r0, r1, 1, nullptr, 0, p.y, dim, nullptr, 0, B, xs, sh);
        grid_barrier<PM_THREADS>(p.barrier, target, gridDim.x);
        // ---- P4: rmsnorm * ffn_norm, silu(w1·)·(w3·) (llama.go:346-361)
        if (threadIdx.x < PM_MAXB) sh.xrow[threadIdx.x] = threadIdx.x < B ? p.y + (size_t)threadIdx.x * dim : nullptr;
        csync<PM_THREADS>();
        fill_norm(xs, L.ffn_norm, dim, B, sh);
        cta_rows(ff, r0, r1);
        gemv_pods<2, PM_U2, 0>(L.w1, L.w3, dim, r0, r1, 1, nullptr, 0, p.act, ff, nullptr, 0, B, xs, sh);
        grid_barrier<PM_THREADS>(p.barrier, target, gridDim.x);
        // ---- P5: w2 + residual (llama.go:363-366)
        cta_rows(dim, r0, r1);
        if (np_ff > 1) {
            gemv_pods<1, PM_U1, 1>(L.w2, nullptr, ff, r0, r1, np_ff, p.act, ff, p.x, dim, p.y, dim, B, xs, sh);
        } else {
            fill_rows(xs, p.act, ff, ff, B);
            gemv_pods<1, PM_U1, 1>(L.w2, nullptr, ff, r0, r1, 1, nullptr, 0, p.x, dim, p.y, dim, B, xs, sh);
        }
        grid_barrier<PM_THREADS>(p.barrier, target, gridDim.x);
        if (threadIdx.x < PM_MAXB) sh.xrow[threadIdx.x] = threadIdx.x < B ? p.x + (size_t)threadIdx.x * dim : nullptr;
        csync<PM_THREADS>();
    }
    if (p.final_norm) {  // final norm + lm_head (llama.go:374-384)
        fill_norm(xs, p.final_norm, dim, B, sh);
        cta_rows(p.vocab, r0, r1);
        gemv_pods<1, PM_U1, 0>(p.output, nullptr, dim, r0, r1, 1, nullptr, 0, p.logits, p.vocab, nullptr, 0, B, xs, sh);
    }
}

constexpr size_t PM_SMEM_BYTES = (size_t)PM_XS_F4 * 16 + sizeof(PodsShared);
static_assert(PM_SMEM_BYTES <= 227 * 1024, "pods megakernel: shared memory over the 227 KB limit");

template <int HD>
static cudaError_t launch(const PodsParams &p, cudaStream_t st) {
    static bool attr[64] = {};  // function attributes are per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        e = cudaFuncSetAttribute(decode_mega_pods_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PM_SMEM_BYTES);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs); cfg.blockDim = dim3(PM_THREADS); cfg.dynamicSmemBytes = PM_SMEM_BYTES; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, decode_mega_pods_kernel<HD>, p);
}

}  // namespace

uint32_t decode_mega_pods_splits(uint32_t B, uint32_t heads) {
    uint32_t s = (2 * kNumSMs) / (B * heads);  // <= 2 attention items per CTA, run concurrently
    return s < 1 ? 1 : (s > 32 ? 32 : s);
}

bool decode_mega_pods_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx) {
    if (heads == 0 || dim % heads) return false;
    const uint32_t hd = dim / heads;
    if (hd != 128 && hd != 64 && hd != 32) return false;
    if (dim % 16 || ff % 16 || dim < 256 || ff < 256) return false;           // >= one chunk per warp and K pass
    if (dim / 16 > PM_XS_CHUNKS) return false;                                // the dim-wide phases keep all columns resident
    if (vocab < (uint32_t)kNumSMs || dim < (uint32_t)kNumSMs) return false;   // every CTA owns rows in every phase
    if ((dim + kNumSMs - 1) / kNumSMs + 15 > 16u * PM_MAX_TILES) return false; // tiles of a streamed phase (acc[] rows)
    if ((size_t)2 * ctx * sizeof(float) > (size_t)PM_XS_F4 * 16) return false;  // attention scores overlay the stage
    return true;
}

void decode_mega_pods(const MegaPodsParamsHost &h, cudaStream_t st) {
    LB_CHECK(h.B >= 1 && h.B <= PM_MAXB, "decode_mega_pods: 1..8 pods");
    LB_CHECK(decode_mega_pods_supported(h.dim, h.ff, h.heads, h.vocab, h.ctx), "decode_mega_pods: unsupported shape");
    PodsParams p;
    p.layers = reinterpret_cast<const PodsLayer *>(h.layers_dev);
    p.n_layers = h.n_layers; p.B = h.B;
    p.tok_embeddings = h.tok_embeddings; p.tokens = h.tokens; p.tok_stride = h.tok_stride; p.state = h.state; p.pasts = h.pasts;
    p.Kb = h.Kb; p.Vb = h.Vb;
    p.final_norm = h.final_norm; p.output = h.output;
    p.x = h.x; p.y = h.y; p.qkv = h.qkv; p.attn = h.attn; p.act = h.act; p.logits = h.logits;
    p.part_o = h.part_o; p.part_ml = h.part_ml; p.barrier = h.barrier;
    p.dim = h.dim; p.ff = h.ff; p.heads = h.heads; p.vocab = h.vocab; p.ctx = h.ctx;
    p.splits = decode_mega_pods_splits(h.B, h.heads);
    LB_CHECK(h.B * h.heads * p.splits <= (uint32_t)PM_MAX_ITEMS, "decode_mega_pods: too many attention items");
    p.chunk_cap = (h.ctx + p.splits - 1) / p.splits;
    LB_CUDA(cudaMemsetAsync(h.barrier, 0, sizeof(unsigned) * 2, st));
    const uint32_t hd = h.dim / h.heads;
    cudaError_t e = hd == 128 ? launch<128>(p, st) : hd == 64 ? launch<64>(p, st) : launch<32>(p, st);
    LB_CUDA(e);
    count_launch();
}

}  // namespace k
}  // namespace lb
