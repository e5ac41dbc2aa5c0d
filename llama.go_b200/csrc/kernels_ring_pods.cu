// kernels_ring_pods.cu — pod batching (SURVEY §8f-1, pkg/server/server.go:84-106, 151-175) on the TMA ring:
// ONE decode step of B <= 8 independent sequences ("pods") as one persistent cooperative kernel that streams
// every weight exactly once for all B tokens.
//
// Round-2 history (profiles/README.md): the first pod megakernel (kernels_mega_pods.cu) fed mma.sync straight
// from LDG registers through a 10-deep register ring.  It was correct (2.8e-6 vs the single-sequence path) but
// slow — 612 tok/s at B = 8, below the per-op path: ncu showed the warps on `long_scoreboard` (register spills
// of loop invariants land in L2 because the 211 KB shared-memory carve-out leaves no L1; one LDG.128 touching
// 8 rows costs 8 L1 wavefronts; 24.8 K instructions of unrolled code miss the instruction cache).  This
// version keeps its verified MMA formulation and takes the weights off the LSU path entirely:
//   * a producer warp streams the CTA's rows of every matrix, in schedule order, into a shared-memory ring
//     with cp.async.bulk (TMA engine, mbarrier completion): slot = 16 rows x 256 floats (16 copies of 1 KB),
//     running ahead across tiles, K passes, phases and grid barriers (see kernels_ring.cu);
//   * 16 consumer warps share every slot: warp w takes the 16-float chunk w of the slot's 256 k for all 16 rows —
//     A fragments (rows g, g + 8; 16 bytes at chunk w) by two conflict-free LDS.128 (row pitch 1 KB + 64 B),
//     B fragment (8 pods x 16 k, fragment-ordered activation stage) by one LDS.128, six mma.sync.m16n8k8 tf32
//     (3xTF32: Whi*Xhi, Wlo*Xhi, Whi*Xlo in separate accumulators; the tensor core truncates raw FP32 to TF32);
//   * the K axis is walked in passes of 8 segments (2048 columns x 8 pods = 64 KB of activations in shared
//     memory, refilled synchronously by the consumers while the ring keeps the HBM stream going); per (tile,
//     pass) the 16 warps' partial 16 x 8 tiles are combined through shared memory in a fixed order
//     (deterministic) and accumulated across passes.
// Attention / RMSNorm / RoPE numerics: kernels_mega.cu; the attention phase (attention_pods), merge statistics, grid
// barrier and PTX wrappers are shared with the other decode kernels (megakernel.cuh).
#include <cooperative_groups.h>
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.cuh"
#include "megakernel.cuh"

namespace lb {
namespace k {
namespace {

constexpr int RP_CWARPS = 16;
constexpr int RP_CTHREADS = RP_CWARPS * 32;
constexpr int RP_ALL_THREADS = RP_CTHREADS + 32;   // + the producer warp
constexpr int RP_MAXB = 8;
constexpr int RP_SEG = 256;                        // floats of K per slot row
constexpr int RP_ROWS = 16;
constexpr uint32_t RP_PITCH = RP_SEG * 4;          // dense rows (one 3-D tensor-map box per slot): fragment-order LDS.128 is 2-way conflicted
constexpr uint32_t RP_SLOT = RP_ROWS * RP_PITCH;
constexpr int RP_MAX_SLOTS = 8;
constexpr uint32_t RP_PASS_SEGS = 8;               // segments per K pass
constexpr uint32_t RP_XS_F4 = RP_PASS_SEGS * 16 * 32;   // float4 slots of the activation stage (64 KB): [chunk][pod][t]
constexpr int RP_MAX_ITEMS = 2 * kNumSMs + 64;
constexpr int RP_MAX_TILES = 16;                   // 16-row tiles of a CTA per matrix (x2 for the w1/w3 pair)

// 3-D tiled load (k, row, layer) -> dense [16][256] floats in shared memory, ONE instruction per slot: 1-D bulk copies
// of 1 KB per row were measured copy-engine bound (~75 clk per copy instruction, 4 TB/s; profiles/README.md)
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// two maps per weight kind:
//   m[]  dims {K, rows, layers} with the model's layer stride, box {256, 16, 1} — bounded by the matrix: rows past M are zero-filled;
//   mc[] dims {K, R, nfull, layers}: the matrix seen as nfull chunks of R = ceil(M / 148) consecutive rows, box {256, 16, 1, 1} —
//        bounded by the CHUNK: a box that hangs over the end of a CTA's chunk fetches only the chunk's rows (the copy engine
//        zero-fills the rest without reading it), so a CTA can own a row range that is not a multiple of 16.
enum { RPK_WQKV = 0, RPK_WO, RPK_W1, RPK_W3, RPK_W2, RPK_OUT, RPK_KINDS };
struct RPMaps {
    CUtensorMap m[RPK_KINDS];
    CUtensorMap mc[RPK_KINDS];
};
// Rows of an M-row matrix owned by this CTA in MulMat phase number `ph`.
// Round-2 history (profiles/README.md): (1) contiguous balanced row ranges through the matrix-bounded map wasted ~11 % of the
// stream on ragged last tiles (a box fetches all 16 rows); (2) whole 16-row tiles dealt out evenly fetch nothing twice, but
// ceil vs mean is a whole tile per CTA and phase — 256 KB .. 700 KB, more than the ring can run ahead — and showed up as
// 5-12 us of barrier wait per phase (r02i trace: 36 of 198 us per layer); (3) 16 + 8 + 4 + 2 + 1-row boxes: every box costs a
// full slot cycle, 941 vs 1239 tok/s.  Now: every CTA owns R = ceil(M / grid) consecutive rows (balanced to one row), fetched
// as 16-row boxes through the chunk-bounded map: the last box of a chunk reads only the rows that exist in the chunk.
// The chunk -> CTA assignment rotates with the phase number (the one or two short chunks at the end move around).
// Matrices with fewer than 16 rows per CTA (test models) keep the whole-tile split.
struct RowPlan {
    uint32_t r0, r1;      // rows [r0, r1)
    uint32_t chunk;       // >= 0: index into the chunked map; 0xFFFFFFFF: use the matrix-bounded map with absolute rows
};
__host__ __device__ __forceinline__ RowPlan rp_rows_plan(uint32_t M, uint32_t c, uint32_t grid) {   // work slot c of `grid` (host: CPU layout test)
    RowPlan rp;
    if (M >= RP_ROWS * grid) {
        const uint32_t R = (M + grid - 1) / grid, nfull = M / R;
        rp.r0 = M < c * R ? M : c * R;
        rp.r1 = M < rp.r0 + R ? M : rp.r0 + R;
        rp.chunk = c < nfull ? c : 0xFFFFFFFFu;
    } else {
        const uint32_t ntiles = (M + RP_ROWS - 1) / RP_ROWS;
        const uint32_t a = (uint32_t)(((uint64_t)ntiles * c) / grid) * RP_ROWS, b = (uint32_t)(((uint64_t)ntiles * (c + 1)) / grid) * RP_ROWS;
        rp.r0 = M < a ? M : a;
        rp.r1 = M < b ? M : b;
        rp.chunk = 0xFFFFFFFFu;
    }
    return rp;
}
__device__ __forceinline__ RowPlan cta_rows_plan(uint32_t M, uint32_t ph) {
    return rp_rows_plan(M, (blockIdx.x + ph * 37u) % gridDim.x, gridDim.x);
}

struct RPParams {
    const MegaLayerHost *layers;   // Kc/Vc unused: every pod has its own cache (Kb/Vb + layer_off)
    uint32_t n_layers, B;
    const float *tok_embeddings;
    const uint32_t *tokens;   // [B][tok_stride]
    uint32_t tok_stride;
    const uint32_t *state;    // {unused, step}
    const uint32_t *pasts;    // [B]
    float *const *Kb;
    float *const *Vb;
    const float *final_norm, *output;
    float *x, *y, *qkv, *attn, *act, *logits;
    float *part_o, *part_ml;
    unsigned *barrier;
    uint32_t dim, ff, heads, vocab, ctx, splits, chunk_cap, n_slots;
    unsigned long long *trace;   // optional: 13 globaltimer stamps per layer by consumer thread 0 of CTA 0 (profiling aid)
};

struct RPShared {
    unsigned long long full[RP_MAX_SLOTS], empty[RP_MAX_SLOTS];
    union {
        float part[2][RP_CWARPS][128];   // per-warp partial 16 rows x 8 pods tiles ([buffer] or, for the w1/w3 pair, [matrix])
        float4 pv[RP_CTHREADS];          // attention: P.V partials per half
    };
    double rope_cs[RP_MAXB][64][2];
    double red[RP_CWARPS][RP_MAXB];
    float acc[2 * RP_MAX_TILES][128];    // running sums of the CTA's tiles across K passes
    float scale[RP_MAXB];
    const float *xrow[RP_MAXB];
    float fred[2][RP_CWARPS / 2];
    float hbcast[2];
    float mrg_m[RP_MAX_ITEMS], mrg_l[RP_MAX_ITEMS], mrg_w[RP_MAX_ITEMS], mrg_inv[RP_MAX_ITEMS];
};

// ---------------------------------------------------------------------------------------------------------
// producer: for K pass, for tile, for segment of the pass (, for matrix): one slot
// ---------------------------------------------------------------------------------------------------------
template <int NM>
__device__ __forceinline__ void produce(const CUtensorMap *mapA, const CUtensorMap *mapB, const CUtensorMap *chunkA, const CUtensorMap *chunkB,
                                        int layer, uint32_t K, uint32_t M, uint32_t &ph,
                                        RingPos &pos, uint32_t ring_base, RPShared &sh, uint32_t n_slots) {
    const RowPlan rp = cta_rows_plan(M, ph++);
    const uint32_t r0 = rp.r0, r1 = rp.r1;
    const uint32_t nseg = K / RP_SEG;
    for (uint32_t s0 = 0; s0 < nseg; s0 += RP_PASS_SEGS) {
        const uint32_t s1 = min(s0 + RP_PASS_SEGS, nseg);
        for (uint32_t tile = r0; tile < r1; tile += RP_ROWS) {
            for (uint32_t seg = s0; seg < s1; seg++) {
#pragma unroll
                for (int m = 0; m < NM; m++) {
                    const uint32_t fb = smem_u32(&sh.full[pos.slot]);
                    mbar_wait<(1u << 24)>(smem_u32(&sh.empty[pos.slot]), pos.phase ^ 1);
                    mbar_expect_tx(fb, RP_SLOT);   // rows past the matrix end are zero-filled by the copy engine and still counted
                    if (rp.chunk != 0xFFFFFFFFu)
                        tma_load_4d(ring_base + pos.slot * RP_SLOT, m == 0 ? chunkA : chunkB, fb, (int)(seg * RP_SEG), (int)(tile - r0), (int)rp.chunk, layer);
                    else
                        tma_load_3d(ring_base + pos.slot * RP_SLOT, m == 0 ? mapA : mapB, fb, (int)(seg * RP_SEG), (int)tile, layer);
                    pos.next(n_slots);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// activation stage of one K pass: xs[(chunk * 8 + pod) * 4 + t] = X[pod][k0 + 16 chunk + 4 t .. + 3]  (pods >= B: zeros)
// MODE 0: plain rows src + pod * ld;  1: rows sh.xrow[pod], times sh.scale[pod] * w[k] (RMSNorm * weight);
// MODE 2: rows of the merged attention output (splits > 1)
// ---------------------------------------------------------------------------------------------------------
template <int MODE, int HD>
__device__ __forceinline__ void fill_pass(float4 *xs, const float *src, uint32_t ld, const float *w, uint32_t k0, uint32_t nchunks,
                                          const RPParams &p, RPShared &sh) {
    const int lane = threadIdx.x & 31, pod = lane >> 2, t = lane & 3;
    const uint32_t nf4 = nchunks * 32, B = p.B;
    const float sc = MODE == 1 ? sh.scale[pod] : 1.f;
    if (MODE == 2) {
        for (uint32_t f = threadIdx.x; f < nf4; f += RP_CTHREADS) {
            const uint32_t kk = k0 + (f >> 5) * 16 + t * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pod < (int)B) {
                const uint32_t S = p.splits, h = kk / HD, d = kk % HD, bh = pod * p.heads + h;
                const float *po = p.part_o + (size_t)bh * S * HD + d;
                for (uint32_t s = 0; s < S; s++) {
                    if (sh.mrg_l[bh * S + s] > 0.f) {
                        const float4 pv = ldcg4(po + (size_t)s * HD);
                        const float wgt = sh.mrg_w[bh * S + s];
                        v.x = fmaf(pv.x, wgt, v.x); v.y = fmaf(pv.y, wgt, v.y);
                        v.z = fmaf(pv.z, wgt, v.z); v.w = fmaf(pv.w, wgt, v.w);
                    }
                }
                const float inv = sh.mrg_inv[bh];
                v = make_float4(__fmul_rn(v.x, inv), __fmul_rn(v.y, inv), __fmul_rn(v.z, inv), __fmul_rn(v.w, inv));
            }
            xs[f] = v;
        }
    } else {
        // a pass is 8 float4 per thread: all of a batch's L2 loads are issued before the first use (a load -> store loop pays one
        // L2 round trip per iteration: ncu r02n, 24 % of the kernel's warp samples on long_scoreboard)
        constexpr int U = 8;
        for (uint32_t f0 = threadIdx.x; f0 < nf4; f0 += U * RP_CTHREADS) {
            float4 xv[U], ww[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t f = f0 + u * RP_CTHREADS, kk = k0 + (f >> 5) * 16 + t * 4;
                xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                ww[u] = xv[u];
                if (f < nf4 && pod < (int)B) {
                    if (MODE == 0) xv[u] = ldcg4(src + (size_t)pod * ld + kk);
                    else {
                        xv[u] = ldcg4(sh.xrow[pod] + kk);
                        ww[u] = __ldg(reinterpret_cast<const float4 *>(w + kk));
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t f = f0 + u * RP_CTHREADS;
                if (f < nf4) {
                    float4 v = xv[u];
                    if (MODE == 1)
                        v = make_float4(__fmul_rn(ww[u].x, __fmul_rn(v.x, sc)), __fmul_rn(ww[u].y, __fmul_rn(v.y, sc)),
                                        __fmul_rn(ww[u].z, __fmul_rn(v.z, sc)), __fmul_rn(ww[u].w, __fmul_rn(v.w, sc)));
                    xs[f] = v;
                }
            }
        }
    }
    csync<RP_CTHREADS>();
}

// RMSNorm scales of the B rows sh.xrow[] (f64 sums of squares of FP32 products, ml.go:1788-1808)
__device__ __forceinline__ void rms_scales(uint32_t K, uint32_t B, RPShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, pod = lane >> 2, t = lane & 3;
    const float *xr = pod < (int)B ? sh.xrow[pod] : nullptr;
    double acc = 0.0;
    if (xr) {
        constexpr int U = 8;   // loads per batch: one L2 round trip per 128 chunks instead of one per chunk
        for (uint32_t f0 = threadIdx.x >> 5; f0 < K / 16; f0 += U * RP_CWARPS) {   // warp-strided chunks; lane (pod, t) takes 4 floats
            float4 v[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t f = f0 + u * RP_CWARPS;
                v[u] = f < K / 16 ? ldcg4(xr + (size_t)f * 16 + t * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                acc += (double)__fmul_rn(v[u].x, v[u].x); acc += (double)__fmul_rn(v[u].y, v[u].y);
                acc += (double)__fmul_rn(v[u].z, v[u].z); acc += (double)__fmul_rn(v[u].w, v[u].w);
            }
        }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (t == 0) sh.red[warp][pod] = acc;
    csync<RP_CTHREADS>();
    if (threadIdx.x < RP_MAXB) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < RP_CWARPS; i++) s += sh.red[i][threadIdx.x];
        sh.scale[threadIdx.x] = (float)(1.0 / sqrt(s / (double)K + 1e-5));
    }
    csync<RP_CTHREADS>();
}

// ---------------------------------------------------------------------------------------------------------
// consumer side of one MulMat phase.  XMODE: how the activation stage of a pass is produced (fill_pass MODE).
// EPI: 0 none, 1 + residual rows (res + pod * ldr, or sh.xrow[pod] when res == nullptr).  NM == 2: SwiGLU pair.
// ---------------------------------------------------------------------------------------------------------
template <int NM, int EPI, int XMODE, int HD>
__device__ __forceinline__ void consume(uint32_t K, uint32_t M, const float *xsrc, uint32_t ldx, const float *wnorm,
                                        float *out, uint32_t ldo, const float *res, uint32_t ldr, uint32_t &ph, RingPos &pos,
                                        const uint8_t *ring, float4 *xs, const RPParams &p, RPShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const uint32_t n_slots = p.n_slots, B = p.B;
    const RowPlan rp = cta_rows_plan(M, ph++);
    const uint32_t r0 = rp.r0, r1 = rp.r1;
    const uint32_t nseg = K / RP_SEG;
    const uint32_t npass = (nseg + RP_PASS_SEGS - 1) / RP_PASS_SEGS;
    const uint32_t wofs = (uint32_t)g * RP_PITCH + (uint32_t)warp * 64 + (uint32_t)t * 16;   // this lane's 16 B of row g inside a slot
    int buf = 0;
    for (uint32_t ps = 0; ps < npass; ps++) {
        const uint32_t s0 = ps * RP_PASS_SEGS, s1 = min(s0 + RP_PASS_SEGS, nseg);
        fill_pass<XMODE, HD>(xs, xsrc, ldx, wnorm, s0 * RP_SEG, (s1 - s0) * 16, p, sh);
        uint32_t tj = 0;
        for (uint32_t tile = r0; tile < r1; tile += RP_ROWS, tj++) {
            float hh[NM][4], lh[NM][4], hl[NM][4];
#pragma unroll
            for (int m = 0; m < NM; m++)
#pragma unroll
                for (int i = 0; i < 4; i++) hh[m][i] = lh[m][i] = hl[m][i] = 0.f;
            for (uint32_t seg = s0; seg < s1; seg++) {
                const float4 xv = xs[((seg - s0) * 16 + warp) * 32 + lane];
                const float4 xl = tf32_lo4(xv);
#pragma unroll
                for (int m = 0; m < NM; m++) {
                    mbar_wait<(1u << 24)>(smem_u32(&sh.full[pos.slot]), pos.phase);
                    const uint8_t *sl = ring + (size_t)pos.slot * RP_SLOT + wofs;
                    const float4 wa = *reinterpret_cast<const float4 *>(sl);
                    const float4 wb = *reinterpret_cast<const float4 *>(sl + 8 * RP_PITCH);
                    const float4 wal = tf32_lo4(wa), wbl = tf32_lo4(wb);
                    mma_tf32(hh[m], wa.x, wb.x, wa.y, wb.y, xv.x, xv.y);
                    mma_tf32(lh[m], wal.x, wbl.x, wal.y, wbl.y, xv.x, xv.y);
                    __syncwarp();   // the MMAs above issued, so every lane's operands have landed in registers: release the slot
                    if (lane == 0) mbar_arrive(smem_u32(&sh.empty[pos.slot]));
                    pos.next(n_slots);
                    mma_tf32(hl[m], wa.x, wb.x, wa.y, wb.y, xl.x, xl.y);
                    mma_tf32(hh[m], wa.z, wb.z, wa.w, wb.w, xv.z, xv.w);
                    mma_tf32(lh[m], wal.z, wbl.z, wal.w, wbl.w, xv.z, xv.w);
                    mma_tf32(hl[m], wa.z, wb.z, wa.w, wb.w, xl.z, xl.w);
                }
            }
            // ---- publish this warp's K-slice of (pass, tile); combine the 16 warps in fixed order
#pragma unroll
            for (int m = 0; m < NM; m++) {
                float *pw = sh.part[NM == 2 ? m : buf][warp];
                const float d0 = __fadd_rn(hh[m][0], __fadd_rn(lh[m][0], hl[m][0])), d1 = __fadd_rn(hh[m][1], __fadd_rn(lh[m][1], hl[m][1]));
                const float d2 = __fadd_rn(hh[m][2], __fadd_rn(lh[m][2], hl[m][2])), d3 = __fadd_rn(hh[m][3], __fadd_rn(lh[m][3], hl[m][3]));
                *reinterpret_cast<float2 *>(pw + g * 8 + 2 * t) = make_float2(d0, d1);         // (row g,     pods 2t, 2t+1)
                *reinterpret_cast<float2 *>(pw + (g + 8) * 8 + 2 * t) = make_float2(d2, d3);   // (row g + 8, pods 2t, 2t+1)
            }
            csync<RP_CTHREADS>();
            if (threadIdx.x < 128) {
                const uint32_t row = tile + (threadIdx.x >> 3), pod = threadIdx.x & 7;
                float s1v = 0.f, s3v = 0.f;
#pragma unroll
                for (int wv = 0; wv < RP_CWARPS; wv++) {
                    s1v += sh.part[NM == 2 ? 0 : buf][wv][threadIdx.x];
                    if (NM == 2) s3v += sh.part[1][wv][threadIdx.x];
                }
                if (npass > 1) {
                    if (ps > 0) {
                        s1v = __fadd_rn(sh.acc[tj][threadIdx.x], s1v);
                        if (NM == 2) s3v = __fadd_rn(sh.acc[RP_MAX_TILES + tj][threadIdx.x], s3v);
                    }
                    if (ps + 1 < npass) {
                        sh.acc[tj][threadIdx.x] = s1v;
                        if (NM == 2) sh.acc[RP_MAX_TILES + tj][threadIdx.x] = s3v;
                    }
                }
                if (ps + 1 == npass && row < r1 && pod < B) {
                    float v;
                    if (NM == 2) v = __fmul_rn(silu_ref(s1v), s3v);
                    else if (EPI == 1) v = __fadd_rn(s1v, __ldcg((res ? res + (size_t)pod * ldr : sh.xrow[pod]) + row));
                    else v = s1v;
                    out[(size_t)pod * ldo + row] = v;
                }
            }
            if (NM == 2) csync<RP_CTHREADS>();   // single-buffered partials in the two-matrix phase
            else buf ^= 1;
        }
        if (ps + 1 < npass) csync<RP_CTHREADS>();   // every warp is done with this pass's activation stage before it is refilled
    }
}

// dynamic shared memory: [ring: n_slots x RP_SLOT][xs: 64 KB (attention scores overlay it)][RPShared]
template <int HD>
__global__ void __launch_bounds__(RP_ALL_THREADS, 1) decode_ring_pods_kernel(const RPParams p, const __grid_constant__ RPMaps maps) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const uint32_t dim = p.dim, ff = p.ff, n_slots = p.n_slots, B = p.B;
    uint8_t *ring = smem_raw;
    float4 *xs = reinterpret_cast<float4 *>(smem_raw + (size_t)n_slots * RP_SLOT);
    float *scores = reinterpret_cast<float *>(xs);
    RPShared &sh = *reinterpret_cast<RPShared *>(smem_raw + (size_t)n_slots * RP_SLOT + (size_t)RP_XS_F4 * 16);
    const bool producer = threadIdx.x >= RP_CTHREADS;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < n_slots; s++) {
            mbar_init(smem_u32(&sh.full[s]), 1);
            mbar_init(smem_u32(&sh.empty[s]), RP_CWARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t i = threadIdx.x; i < B * 64; i += RP_ALL_THREADS) {   // RoPE tables of the B positions (f64, ml.go:2307-2310)
        const uint32_t b = i / 64, j = i % 64;
        if (j < HD / 2) {
            double sn, cs;
            sincos((double)p.pasts[b] * pow(10000.0, ((double)(-(int)(2 * j))) / (double)HD), &sn, &cs);
            sh.rope_cs[b][j][0] = cs;
            sh.rope_cs[b][j][1] = sn;
        }
    }
    if (threadIdx.x < RP_MAXB)
        sh.xrow[threadIdx.x] = threadIdx.x < B ? p.tok_embeddings + (size_t)p.tokens[(size_t)threadIdx.x * p.tok_stride + p.state[1]] * dim
                                                 : nullptr;  // GetRows, llama.go:244
    __syncthreads();   // the only CTA-wide barrier

    RingPos pos;
    pos.slot = 0; pos.phase = 0;
    uint32_t ph = 0;   // MulMat phase counter (rotates the tile assignment; identical on both sides)
    if (producer) {
        if (threadIdx.x != RP_CTHREADS) return;   // one thread drives the copy engine
        const uint32_t ring_base = smem_u32(ring);
        for (uint32_t li = 0; li < p.n_layers; li++) {
            produce<1>(&maps.m[RPK_WQKV], nullptr, &maps.mc[RPK_WQKV], nullptr, (int)li, dim, 3 * dim, ph, pos, ring_base, sh, n_slots);
            produce<1>(&maps.m[RPK_WO], nullptr, &maps.mc[RPK_WO], nullptr, (int)li, dim, dim, ph, pos, ring_base, sh, n_slots);
            produce<2>(&maps.m[RPK_W1], &maps.m[RPK_W3], &maps.mc[RPK_W1], &maps.mc[RPK_W3], (int)li, dim, ff, ph, pos, ring_base, sh, n_slots);
            produce<1>(&maps.m[RPK_W2], nullptr, &maps.mc[RPK_W2], nullptr, (int)li, ff, dim, ph, pos, ring_base, sh, n_slots);
        }
        if (p.final_norm) produce<1>(&maps.m[RPK_OUT], nullptr, &maps.mc[RPK_OUT], nullptr, 0, dim, p.vocab, ph, pos, ring_base, sh, n_slots);
        return;
    }
    unsigned target = 0;
    unsigned long long *tr = (p.trace && blockIdx.x == 0 && threadIdx.x == 0) ? p.trace : nullptr;
    auto stamp = [&](uint32_t li, int i) {
        if (tr) {
            unsigned long long tt;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt));
            tr[li * 13 + i] = tt;
        }
    };
    for (uint32_t li = 0; li < p.n_layers; li++) {
        const MegaLayerHost L = p.layers[li];
        const size_t layer_off = (size_t)li * p.ctx * dim;
        stamp(li, 0);
        // ---- P1: rmsnorm * attention_norm, [wq;wk;wv] (llama.go:255-265)
        rms_scales(dim, B, sh);
        stamp(li, 1);
        consume<1, 0, 1, HD>(dim, 3 * dim, nullptr, 0, L.attention_norm, p.qkv, 3 * dim, nullptr, 0, ph, pos, ring, xs, p, sh);
        stamp(li, 2);
        grid_barrier<RP_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 3);
        // ---- P2: RoPE, KV store, attention (llama.go:274-333)
        attention_pods<HD, RP_CTHREADS>(p, layer_off, sh, scores);
        stamp(li, 4);
        grid_barrier<RP_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 5);
        // ---- P3: wo + residual (llama.go:336-340)
        if (p.splits > 1) {
            merge_stats<RP_CTHREADS>(p, p.B * p.heads, sh);
            consume<1, 1, 2, HD>(dim, dim, nullptr, 0, nullptr, p.y, dim, nullptr, 0, ph, pos, ring, xs, p, sh);
        } else {
            consume<1, 1, 0, HD>(dim, dim, p.attn, dim, nullptr, p.y, dim, nullptr, 0, ph, pos, ring, xs, p, sh);
        }
        stamp(li, 6);
        grid_barrier<RP_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 7);
        // ---- P4: rmsnorm * ffn_norm, silu(w1.)*(w3.) (llama.go:346-361)
        if (threadIdx.x < RP_MAXB) sh.xrow[threadIdx.x] = threadIdx.x < B ? p.y + (size_t)threadIdx.x * dim : nullptr;
        csync<RP_CTHREADS>();
        rms_scales(dim, B, sh);
        stamp(li, 8);
        consume<2, 0, 1, HD>(dim, ff, nullptr, 0, L.ffn_norm, p.act, ff, nullptr, 0, ph, pos, ring, xs, p, sh);
        stamp(li, 9);
        grid_barrier<RP_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 10);
        // ---- P5: w2 + residual (llama.go:363-366)
        consume<1, 1, 0, HD>(ff, dim, p.act, ff, nullptr, p.x, dim, p.y, dim, ph, pos, ring, xs, p, sh);
        stamp(li, 11);
        grid_barrier<RP_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 12);
        if (threadIdx.x < RP_MAXB) sh.xrow[threadIdx.x] = threadIdx.x < B ? p.x + (size_t)threadIdx.x * dim : nullptr;
        csync<RP_CTHREADS>();
    }
    if (p.final_norm) {  // final norm + lm_head (llama.go:374-384)
        rms_scales(dim, B, sh);
        consume<1, 0, 1, HD>(dim, p.vocab, nullptr, 0, p.final_norm, p.logits, p.vocab, nullptr, 0, ph, pos, ring, xs, p, sh);
    }
}

static uint32_t pods_splits(uint32_t B, uint32_t heads) {
    uint32_t s = (2 * kNumSMs) / (B * heads);
    return s < 1 ? 1 : (s > 32 ? 32 : s);
}
static uint32_t pods_plan(size_t *smem_out) {
    const size_t fixed = (size_t)RP_XS_F4 * 16 + sizeof(RPShared);
    const size_t cap = 227 * 1024;
    uint32_t n = (uint32_t)((cap - fixed) / RP_SLOT);
    if (n > RP_MAX_SLOTS) n = RP_MAX_SLOTS;
    if (smem_out) *smem_out = fixed + (size_t)n * RP_SLOT;
    return n;
}

template <int HD>
static cudaError_t launch(const RPParams &p, const RPMaps &maps, size_t smem, cudaStream_t st) {
    static bool attr[64] = {};  // function attributes are per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        e = cudaFuncSetAttribute(decode_ring_pods_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs); cfg.blockDim = dim3(RP_ALL_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, decode_ring_pods_kernel<HD>, p, maps);
}

}  // namespace

// layout query for the CPU tests: rows and chunk index of work slot `idx` -> out {r0, r1, chunk}
void ring_pods_layout_query(uint32_t M, uint32_t idx, uint32_t *out) {
    const RowPlan rp = rp_rows_plan(M, idx, kNumSMs);
    out[0] = rp.r0; out[1] = rp.r1; out[2] = rp.chunk;
}

bool decode_ring_pods_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx) {
    if (heads == 0 || dim % heads) return false;
    const uint32_t hd = dim / heads;
    if (hd != 128 && hd != 64 && hd != 32) return false;
    if (dim % RP_SEG || ff % RP_SEG) return false;
    const uint32_t max_m = (ff > vocab ? ff : vocab) > 3 * dim ? (ff > vocab ? ff : vocab) : 3 * dim;
    if (((max_m + RP_ROWS - 1) / RP_ROWS + kNumSMs - 1) / kNumSMs > (uint32_t)RP_MAX_TILES ||
        ((max_m + kNumSMs - 1) / kNumSMs + RP_ROWS - 1) / RP_ROWS > (uint32_t)RP_MAX_TILES) return false;   // acc[] rows (either row split)
    if ((size_t)2 * ctx * sizeof(float) > (size_t)RP_XS_F4 * 16) return false;             // attention scores overlay the stage
    return pods_plan(nullptr) >= 3;
}

void decode_ring_pods(const MegaPodsParamsHost &h, cudaStream_t st) {
    LB_CHECK(h.B >= 1 && h.B <= RP_MAXB, "decode_ring_pods: 1..8 pods");
    LB_CHECK(decode_ring_pods_supported(h.dim, h.ff, h.heads, h.vocab, h.ctx), "decode_ring_pods: unsupported shape");
    RPParams p;
    p.layers = h.layers_dev;
    p.n_layers = h.n_layers; p.B = h.B;
    p.tok_embeddings = h.tok_embeddings; p.tokens = h.tokens; p.tok_stride = h.tok_stride; p.state = h.state; p.pasts = h.pasts;
    p.Kb = h.Kb; p.Vb = h.Vb;
    p.final_norm = h.final_norm; p.output = h.output;
    p.x = h.x; p.y = h.y; p.qkv = h.qkv; p.attn = h.attn; p.act = h.act; p.logits = h.logits;
    p.part_o = h.part_o; p.part_ml = h.part_ml; p.barrier = h.barrier;
    p.dim = h.dim; p.ff = h.ff; p.heads = h.heads; p.vocab = h.vocab; p.ctx = h.ctx;
    p.splits = pods_splits(h.B, h.heads);
    LB_CHECK(h.B * h.heads * p.splits <= (uint32_t)RP_MAX_ITEMS, "decode_ring_pods: too many attention items");
    p.chunk_cap = (h.ctx + p.splits - 1) / p.splits;
    p.trace = reinterpret_cast<unsigned long long *>(h.trace);
    size_t smem = 0;
    p.n_slots = pods_plan(&smem);
    LB_CUDA(cudaMemsetAsync(h.barrier, 0, sizeof(unsigned) * 2, st));
    const uint32_t hd = h.dim / h.heads;
    LB_CHECK(h.tmaps != nullptr, "decode_ring_pods: tensor maps missing (ring_pods_make_maps)");
    const RPMaps &maps = *static_cast<const RPMaps *>(h.tmaps);
    cudaError_t e = hd == 128 ? launch<128>(p, maps, smem, st) : hd == 64 ? launch<64>(p, maps, smem, st) : launch<32>(p, maps, smem, st);
    LB_CUDA(e);
    count_launch();
}

// ---- tensor maps -------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled_rp)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                       const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled_rp rp_encode_fn() {
    static PFN_encodeTiled_rp fn = nullptr;
    if (!fn) {
        void *pfn = nullptr;
        cudaDriverEntryPointQueryResult q;
        LB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &pfn, cudaEnableDefault, &q));
        LB_CHECK(pfn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled is not available in this driver");
        fn = reinterpret_cast<PFN_encodeTiled_rp>(pfn);
    }
    return fn;
}
// the matrix as nfull chunks of R = ceil(rows / 148) rows (cta_rows_plan): dims {K, R, nfull, layers}, box {256, 16, 1, 1}
static CUtensorMap rp_map_chunked(const float *base, uint64_t K, uint64_t rows, uint64_t layers, uint64_t layer_stride_floats) {
    PFN_encodeTiled_rp fn = rp_encode_fn();
    const uint64_t R = (rows + kNumSMs - 1) / kNumSMs, nfull = rows / R;
    CUtensorMap m;
    memset(&m, 0, sizeof(m));
    if (rows < (uint64_t)RP_ROWS * kNumSMs) return m;   // never used: such a matrix keeps the whole-tile split (cta_rows_plan)
    cuuint64_t dims[4] = {K, R, nfull ? nfull : 1, layers};
    cuuint64_t strides[3] = {K * 4, R * K * 4, (layers > 1 ? layer_stride_floats : K * rows) * 4};
    cuuint32_t box[4] = {RP_SEG, RP_ROWS, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LB_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (chunked) failed (" + std::to_string((int)r) + ")");
    return m;
}
static CUtensorMap rp_map(const float *base, uint64_t K, uint64_t rows, uint64_t layers, uint64_t layer_stride_floats) {
    PFN_encodeTiled_rp fn = rp_encode_fn();
    CUtensorMap m;
    cuuint64_t dims[3] = {K, rows, layers};
    cuuint64_t strides[2] = {K * 4, (layers > 1 ? layer_stride_floats : K * rows) * 4};
    cuuint32_t box[3] = {RP_SEG, RP_ROWS, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LB_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return m;
}

size_t ring_pods_maps_bytes() { return sizeof(RPMaps); }

// layers_host = the host copy of the MegaLayerHost array: every layer must sit at the same stride in one slab
void ring_pods_make_maps(const MegaLayerHost *L, uint32_t n_layers, uint32_t dim, uint32_t ff, uint32_t vocab, const float *output,
                         void *maps_out) {
    LB_CHECK(L && n_layers >= 1 && maps_out, "ring_pods_make_maps: nil argument");
    ptrdiff_t stride = n_layers > 1 ? L[1].wqkv - L[0].wqkv : 0;
    for (uint32_t i = 1; i < n_layers; i++) {
        LB_CHECK(L[i].wqkv - L[i - 1].wqkv == stride && L[i].wo - L[i - 1].wo == stride && L[i].w1 - L[i - 1].w1 == stride &&
                     L[i].w3 - L[i - 1].w3 == stride && L[i].w2 - L[i - 1].w2 == stride,
                 "ring_pods_make_maps: layers are not equally spaced in one slab");
    }
    LB_CHECK(stride >= 0 && (stride % 4) == 0, "ring_pods_make_maps: bad layer stride");
    RPMaps m;
    m.m[RPK_WQKV] = rp_map(L[0].wqkv, dim, 3ull * dim, n_layers, (uint64_t)stride);
    m.m[RPK_WO] = rp_map(L[0].wo, dim, dim, n_layers, (uint64_t)stride);
    m.m[RPK_W1] = rp_map(L[0].w1, dim, ff, n_layers, (uint64_t)stride);
    m.m[RPK_W3] = rp_map(L[0].w3, dim, ff, n_layers, (uint64_t)stride);
    m.m[RPK_W2] = rp_map(L[0].w2, ff, dim, n_layers, (uint64_t)stride);
    m.m[RPK_OUT] = output ? rp_map(output, dim, vocab, 1, 0) : m.m[RPK_WO];
    m.mc[RPK_WQKV] = rp_map_chunked(L[0].wqkv, dim, 3ull * dim, n_layers, (uint64_t)stride);
    m.mc[RPK_WO] = rp_map_chunked(L[0].wo, dim, dim, n_layers, (uint64_t)stride);
    m.mc[RPK_W1] = rp_map_chunked(L[0].w1, dim, ff, n_layers, (uint64_t)stride);
    m.mc[RPK_W3] = rp_map_chunked(L[0].w3, dim, ff, n_layers, (uint64_t)stride);
    m.mc[RPK_W2] = rp_map_chunked(L[0].w2, ff, dim, n_layers, (uint64_t)stride);
    m.mc[RPK_OUT] = output ? rp_map_chunked(output, dim, vocab, 1, 0) : m.mc[RPK_WO];
    memcpy(maps_out, &m, sizeof(RPMaps));
}

}  // namespace k
}  // namespace lb
