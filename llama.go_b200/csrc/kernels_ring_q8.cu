// kernels_ring_q8.cu — single-token decode with Q8_0 block-quantised weights (BASELINE config 3; format DESIGN.md §6)
// as ONE persistent cooperative kernel on the TMA ring, with the MulMat on the INT8 tensor cores.
//
// Round-1/2 history (profiles/README.md): the per-op Q8 path is a latency chain per kernel (0.50 of its roofline:
// a Q8 matrix is 4x smaller than its FP32 twin, so every kernel is one wave of resident warps, and the PRMT/FADD
// dequantisation costs ~3.5 CUDA-core instructions per weight); a register-fed Q8 megakernel (173 / 290 tok/s) and an
// int8-mma per-op GEMV (382 tok/s) were measured slower.  Here
//   * the weight stream is decoupled from the consumers: a producer thread feeds a shared-memory ring with ONE bulk
//     copy per slot (cp.async.bulk, 18 KB), running ahead across tiles, phases and grid barriers (kernels_ring.cu).
//     The matrices are kept in a TILE-MAJOR "decode plane" (q8_to_tile_major): for every 16-row tile and every
//     1024-column segment one contiguous record [32 blocks][16 rows][32 int8] + [32 blocks][16 rows] f32 scales —
//     exactly the order a CTA streams them, and a shared-memory image in which the mma fragment reads are
//     bank-conflict free (the first version streamed row-major planes through 3-D tensor maps: 4-way conflicts on
//     the fragment loads and 8-way on the scales capped it below the per-op path, profiles/README.md);
//   * the int8 weights are consumed AS STORED by mma.sync.m16n8k32.s8 (A = 16 rows x 32 k = one Q8 block per row);
//     the FP32 activation block (32 values) enters as four balanced base-128 digit planes relative to the block's
//     power-of-two scale s (x = s * (d0/2^6 + d1/2^13 + d2/2^20 + d3/2^27) +- s * 2^-28), four of the eight B columns;
//     the s32 products are exact, one FMA per (row, block) applies d_w * s.  No dequantisation instruction per weight:
//     ~24 instructions per 512 weights instead of ~1800.
// The result differs from "the FP32 path on the dequantised weights d*q" (the parity target, tests/test_gpu_q8.py)
// only by summation order and the 2^-28 digit truncation.
// Attention / RMSNorm / RoPE numerics: kernels_mega.cu; the attention phase, grid barrier and PTX wrappers are shared
// with the other decode kernels (megakernel.cuh).
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.cuh"
#include "megakernel.cuh"

namespace lb {
namespace k {
namespace {

constexpr int RQ_CWARPS = 16;
constexpr int RQ_CTHREADS = RQ_CWARPS * 32;
constexpr int RQ_THREADS = RQ_CTHREADS + 32;       // + the producer warp
constexpr uint32_t RQ_SEGK = 1024;                 // k per slot row
constexpr uint32_t RQ_ROWS = 16;
constexpr uint32_t RQ_BLKQ = RQ_ROWS * 32;                     // int8 bytes of one 32-column block of a tile: [16 rows][32]
constexpr uint32_t RQ_BLKD = RQ_ROWS * 4;                      // its scales: [16 rows] f32
constexpr uint32_t RQ_BLK = RQ_BLKQ + RQ_BLKD;                 // 576 bytes per (tile, block)
constexpr uint32_t RQ_SLOT = (RQ_SEGK / 32) * RQ_BLK;          // 18432: a full segment record = [32][16][32] int8 | [32][16] f32
constexpr int RQ_MAX_SLOTS = 10;
constexpr int RQ_MAX_ITEMS = 2 * kNumSMs;
constexpr int RQ_MAX_HEADS = 256;

// D(16x8, s32) = A(16x32, s8, row) * B(32x8, s8, col)
__device__ __forceinline__ void mma_s8(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(0));
}

// explicit shared-space loads from 32-bit shared addresses: a generic pointer into the ring costs an S2R of the cluster CTA id
// and an address-space conversion per load (SASS of the first version of this loop)
__device__ __forceinline__ uint2 lds_u2(uint32_t addr) {
    uint2 r;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr));
    return r;
}
__device__ __forceinline__ float lds_f(uint32_t addr) {
    float r;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(addr));
    return r;
}

struct RQParams {
    const MegaLayerHost *layers;      // norm vectors and the KV slabs
    const RingQ8Layer *planes;        // [n_layers] tile-major decode planes of the layer's matrices
    const uint8_t *out_plane;         // lm_head plane (nullptr: no lm_head on this stage)
    uint32_t n_layers;
    const float *tok_embeddings;
    const uint32_t *tokens;
    const uint32_t *state;            // {past, step}
    const float *final_norm;          // nullptr: no lm_head on this stage
    float *x, *y, *qkv, *attn, *act, *logits;
    float *part_o, *part_ml;
    unsigned *barrier;
    uint32_t dim, ff, heads, vocab, ctx, splits, chunk_cap, n_slots, kpad;   // kpad = max(dim, ff) rounded up to 1024
    uint32_t spin_ns;   // consumers' back-off between polls of a slot's mbarrier (LB_Q8_SPIN_NS)
    unsigned long long *trace;
};

struct RQShared {
    unsigned long long full[RQ_MAX_SLOTS], empty[RQ_MAX_SLOTS];
    double red[RQ_CWARPS];
    double rope_cs[64][2];
    float fred[2][RQ_CWARPS / 2];
    float hbcast[2];
    float part[2][2][RQ_CWARPS][16];  // [buffer][matrix][warp][row of the tile]
    float4 pv[RQ_CTHREADS];
    float mrg_m[RQ_MAX_ITEMS], mrg_l[RQ_MAX_ITEMS], mrg_w[RQ_MAX_ITEMS], mrg_inv[RQ_MAX_HEADS];
};

// Rows of an M-row matrix owned by this CTA in MulMat phase number `ph`: whole 16-row tiles (a TMA box never fetches
// rows the CTA does not use), ceil(M/16) tiles dealt out evenly; WHICH CTAs get the extra tile rotates with the phase
// number, and the run-ahead of the ring lets a CTA that is short one tile in this phase start on the next phase's
// weights while the others finish — the per-phase imbalance averages out over a layer.
// Row grouping of an M-row matrix — shared by the decode plane's layout (q8_to_tile_major) and the work split:
//   M >= 16 rows per CTA: the matrix is cut into grid-many chunks of R = ceil(M / grid) consecutive rows (balanced to one row; a
//   whole-tile split left ceil-vs-mean = one 16-row tile per CTA and phase, 72 .. 200 KB, as barrier wait: r02k trace, 21 of 67 us
//   per layer); inside a chunk: 16-row tiles and one short last tile.  Smaller matrices (test models): plain 16-row tiles.
// A tile of rt rows starting at row g0 is stored compactly: record(g0, seg) at (g0 * K/32 + seg * 32 * rt) * 36 bytes =
// [nb blocks][rt rows][32 int8] | [nb][rt] f32 scales — one contiguous bulk copy per slot, whatever rt is.
__host__ __device__ __forceinline__ uint32_t rq_chunk_rows(uint32_t M, uint32_t grid) {   // 0: plain 16-row tiles
    return M >= RQ_ROWS * grid ? (M + grid - 1) / grid : 0u;
}
// rows [r0, r1) of work slot c of `grid` (host + device: the same function drives the producer, the consumers and the CPU layout test)
__host__ __device__ __forceinline__ void rq_rows_of(uint32_t M, uint32_t c, uint32_t grid, uint32_t &r0, uint32_t &r1) {
    const uint32_t R = rq_chunk_rows(M, grid);
    if (R) {
        r0 = M < c * R ? M : c * R;
        r1 = M < r0 + R ? M : r0 + R;
    } else {
        const uint32_t ntiles = (M + RQ_ROWS - 1) / RQ_ROWS;
        const uint32_t a = (uint32_t)(((uint64_t)ntiles * c) / grid) * RQ_ROWS, b = (uint32_t)(((uint64_t)ntiles * (c + 1)) / grid) * RQ_ROWS;
        r0 = M < a ? M : a;
        r1 = M < b ? M : b;
    }
}
// the tile of the decode plane that holds `row`: first row g0, height rt (<= 16)
__host__ __device__ __forceinline__ void rq_group_of(uint32_t M, uint32_t row, uint32_t grid, uint32_t &g0, uint32_t &rt) {
    const uint32_t R = rq_chunk_rows(M, grid);
    if (R) {
        const uint32_t c = row / R, cend = M < (c + 1) * R ? M : (c + 1) * R;
        g0 = c * R + ((row - c * R) / RQ_ROWS) * RQ_ROWS;
        rt = cend - g0 < RQ_ROWS ? cend - g0 : RQ_ROWS;
    } else {
        g0 = (row / RQ_ROWS) * RQ_ROWS;
        rt = M - g0 < RQ_ROWS ? M - g0 : RQ_ROWS;
    }
}
__device__ __forceinline__ void cta_rows(uint32_t M, uint32_t ph, uint32_t &r0, uint32_t &r1) {
    rq_rows_of(M, (blockIdx.x + ph * 37u) % gridDim.x, gridDim.x, r0, r1);
}

// ---------------------------------------------------------------------------------------------------------
// producer (one thread): for tile, for segment (, for matrix): one contiguous record of the tile-major plane per slot
// ---------------------------------------------------------------------------------------------------------
template <int NM>
__device__ __forceinline__ void produce(const uint8_t *PA, const uint8_t *PB, uint32_t K, uint32_t M, uint32_t &ph, RingPos &pos,
                                        uint32_t ring_base, RQShared &sh, uint32_t n_slots) {
    uint32_t r0, r1;
    cta_rows(M, ph++, r0, r1);
    const uint32_t nblk = K / 32, nseg = (K + RQ_SEGK - 1) / RQ_SEGK;
    for (uint32_t tile = r0; tile < r1; tile += RQ_ROWS) {
        const uint32_t rt = min((uint32_t)RQ_ROWS, r1 - tile);
        const size_t tbase = (size_t)tile * nblk * 36u;
        for (uint32_t seg = 0; seg < nseg; seg++) {
            const uint32_t nb = min(RQ_SEGK / 32, nblk - seg * (RQ_SEGK / 32));
            const uint32_t bytes = nb * rt * 36u;
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const uint32_t fb = smem_u32(&sh.full[pos.slot]);
                mbar_wait<(1u << 24)>(smem_u32(&sh.empty[pos.slot]), pos.phase ^ 1);
                mbar_expect_tx(fb, bytes);
                bulk_g2s(ring_base + pos.slot * RQ_SLOT, (m == 0 ? PA : PB) + tbase + (size_t)seg * (RQ_SEGK / 32) * rt * 36u, bytes, fb);
                pos.next(n_slots);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Activation vector -> digit planes.  A 32-value block of x becomes four int8 planes relative to the block's power-of-two
// scale s = 2^e (max|x| / s in [0.5, 1)):  x = s * (d0/2^6 + d1/2^13 + d2/2^20 + d3/2^27) +- s * 2^-28, |d_i| <= 64.
// dig[(b * 4 + plane) * 32 + k % 32], xsc[b] = s.  One warp per block, one lane per element, everything in registers
// (the first version staged the FP32 vector in shared memory and converted it in a second sweep: ~4 us per phase).
// ---------------------------------------------------------------------------------------------------------
// Lane layout: a thread holds 4 consecutive elements (one float4) of block f / 8, f = the float4's index in the vector;
// the 8 lanes of a block sit next to each other in the warp (f = threadIdx.x + i * 512 keeps f % 8 == lane % 8).
__device__ __forceinline__ uint32_t pack4(int a, int b, int c, int d) {
    return ((uint32_t)a & 0xFFu) | (((uint32_t)b & 0xFFu) << 8) | (((uint32_t)c & 0xFFu) << 16) | ((uint32_t)d << 24);
}
__device__ __forceinline__ void emit4(uint32_t f, float4 v, int8_t *dig, float *xsc) {
    float m = fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));
    const uint32_t grp = 0xFFu << (threadIdx.x & 24u);   // the block's 8 lanes (a warp's other blocks may be past the end of the vector)
    m = fmaxf(m, __shfl_xor_sync(grp, m, 1));
    m = fmaxf(m, __shfl_xor_sync(grp, m, 2));
    m = fmaxf(m, __shfl_xor_sync(grp, m, 4));
    // exponent arithmetic on the bits; a block whose maximum is zero or denormal is sent as zeros (|v| < 1.2e-38)
    const uint32_t E = (__float_as_uint(m) >> 23) & 0xFFu;
    const float s = E ? __uint_as_float((E + 1u) << 23) : 1.0f, inv = E ? __uint_as_float((253u - E) << 23) : 0.0f;
    const float in[4] = {v.x, v.y, v.z, v.w};
    int d[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float r = __fmul_rn(__fmul_rn(in[i], inv), 64.0f);   // exact (powers of two)
        d[0][i] = __float2int_rn(r); r = __fsub_rn(r, (float)d[0][i]);
        r = __fmul_rn(r, 128.0f);
        d[1][i] = __float2int_rn(r); r = __fsub_rn(r, (float)d[1][i]);
        r = __fmul_rn(r, 128.0f);
        d[2][i] = __float2int_rn(r); r = __fsub_rn(r, (float)d[2][i]);
        r = __fmul_rn(r, 128.0f);
        d[3][i] = __float2int_rn(r);
    }
    const uint32_t b = f >> 3, sub = f & 7u;
    uint32_t *o = reinterpret_cast<uint32_t *>(dig + (size_t)b * 128) + sub;
#pragma unroll
    for (int pl = 0; pl < 4; pl++) o[pl * 8] = pack4(d[pl][0], d[pl][1], d[pl][2], d[pl][3]);
    if (sub == 0) xsc[b] = s;
}
__device__ __forceinline__ void zero_blocks(uint32_t b0, uint32_t b1, int8_t *dig, float *xsc) {   // padding columns of the last segment
    for (uint32_t i = b0 * 32 + threadIdx.x; i < b1 * 32; i += RQ_CTHREADS) {
        reinterpret_cast<uint32_t *>(dig)[i] = 0u;
        if ((i & 31) == 0) xsc[i >> 5] = 1.0f;
    }
}
// digits of  w * (x * f32(1/sqrt(mean_f64(x^2) + 1e-5)))   (ComputeForwardRMSNormFP32 + Mul, ml.go:1753-1812; llama.go:255-259)
// One L2/HBM round trip: the residual stream and the norm weights are requested together, as float4 per thread.
__device__ __forceinline__ void norm_digits(const float *x, const float *w, uint32_t K, uint32_t kp, int8_t *dig, float *xsc, RQShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int R = 4;   // float4 per thread kept in registers (K <= 8192); the rest is re-read
    float4 v[R], g[R];
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < R; i++) {
        const uint32_t f = threadIdx.x + i * RQ_CTHREADS;
        v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        g[i] = v[i];
        if (f < K / 4) {
            v[i] = ldcg4(x + (size_t)f * 4);
            g[i] = __ldg(reinterpret_cast<const float4 *>(w) + f);
        }
    }
#pragma unroll
    for (int i = 0; i < R; i++) {
        acc += (double)__fmul_rn(v[i].x, v[i].x); acc += (double)__fmul_rn(v[i].y, v[i].y);
        acc += (double)__fmul_rn(v[i].z, v[i].z); acc += (double)__fmul_rn(v[i].w, v[i].w);
    }
    for (uint32_t f = threadIdx.x + R * RQ_CTHREADS; f < K / 4; f += RQ_CTHREADS) {
        const float4 u = ldcg4(x + (size_t)f * 4);
        acc += (double)__fmul_rn(u.x, u.x); acc += (double)__fmul_rn(u.y, u.y);
        acc += (double)__fmul_rn(u.z, u.z); acc += (double)__fmul_rn(u.w, u.w);
    }
    acc = warp_sum(acc);
    if (lane == 0) sh.red[warp] = acc;
    csync<RQ_CTHREADS>();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < RQ_CWARPS; i++) t += sh.red[i];
    const float sc = (float)(1.0 / sqrt(t / (double)K + 1e-5));
    auto nrm = [&](float4 u, float4 q) {
        return make_float4(__fmul_rn(q.x, __fmul_rn(u.x, sc)), __fmul_rn(q.y, __fmul_rn(u.y, sc)),
                           __fmul_rn(q.z, __fmul_rn(u.z, sc)), __fmul_rn(q.w, __fmul_rn(u.w, sc)));
    };
#pragma unroll
    for (int i = 0; i < R; i++) {
        const uint32_t f = threadIdx.x + i * RQ_CTHREADS;
        if (f < K / 4) emit4(f, nrm(v[i], g[i]), dig, xsc);   // (f < K/4 is uniform over the 8 lanes of a block: K % 32 == 0)
    }
    for (uint32_t f = threadIdx.x + R * RQ_CTHREADS; f < K / 4; f += RQ_CTHREADS)
        emit4(f, nrm(ldcg4(x + (size_t)f * 4), __ldg(reinterpret_cast<const float4 *>(w) + f)), dig, xsc);
    zero_blocks(K / 32, kp / 32, dig, xsc);
    csync<RQ_CTHREADS>();   // also orders sh.red against its next use
}
__device__ __forceinline__ void plain_digits(const float *x, uint32_t K, uint32_t kp, int8_t *dig, float *xsc) {
    constexpr int PB = 6;   // float4 per thread per batch of loads: one L2 round trip per 12288 elements
    for (uint32_t f0 = threadIdx.x; f0 < K / 4; f0 += PB * RQ_CTHREADS) {
        float4 v[PB];
#pragma unroll
        for (int i = 0; i < PB; i++) {
            const uint32_t f = f0 + i * RQ_CTHREADS;
            v[i] = f < K / 4 ? ldcg4(x + (size_t)f * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < PB; i++) {
            const uint32_t f = f0 + i * RQ_CTHREADS;
            if (f < K / 4) emit4(f, v[i], dig, xsc);
        }
    }
    zero_blocks(K / 32, kp / 32, dig, xsc);
    csync<RQ_CTHREADS>();
}
// digits of the merged attention output (statistics: merge_stats, megakernel.cuh): out = (sum_s O_s w_s) * f32(1 / sum_s l_s w_s)
template <int HD>
__device__ __forceinline__ void merge_digits(const RQParams &p, uint32_t kp, int8_t *dig, float *xsc, RQShared &sh) {
    const uint32_t S = p.splits;
    merge_stats<RQ_CTHREADS>(p, p.heads, sh);
    constexpr int MB = 12;   // splits per batch of loads (a per-split loop of L2 reads costs one round trip per split)
    for (uint32_t f = threadIdx.x; f < p.dim / 4; f += RQ_CTHREADS) {
        const uint32_t e = f * 4, h = e / HD, d = e % HD;
        const float *po = p.part_o + (size_t)h * S * HD + d;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
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
        emit4(f, make_float4(__fmul_rn(o.x, inv), __fmul_rn(o.y, inv), __fmul_rn(o.z, inv), __fmul_rn(o.w, inv)), dig, xsc);
    }
    zero_blocks(p.dim / 32, kp / 32, dig, xsc);
    csync<RQ_CTHREADS>();
}

// ---------------------------------------------------------------------------------------------------------
// consumer: out[row] = epilogue(sum_k d[row][k/32] q[row][k] x[k]) for this CTA's rows; NM == 2: silu(W1.x) * (W3.x)
// Warp w takes blocks 2w and 2w + 1 of every slot (64 of its 1024 k) for all 16 rows; K-slices are combined
// across the 16 warps per tile in a fixed order.
// ---------------------------------------------------------------------------------------------------------
// KREG: number of 1024-column segments whose B fragments (activation digits + block scales) stay in registers for the whole
// phase (K <= KREG * 1024; 0: reloaded from shared memory for every segment — what the kernel uses: with 17 warps per CTA the
// register file allows 96 registers per thread, and 24 more live registers spill inside the slot loop).  Instruction diet of round 2 (ncu r02n: an HBM-bound
// kernel with 49 % of its issue slots busy): full 16-row tiles and full 32-block records take a path without predicates whose
// eight loads are immediates off two per-warp base registers; K-slice partials are double-buffered (one CTA barrier per tile).
template <int NM, int EPI, int KREG>
__device__ __forceinline__ void consume(uint32_t K, uint32_t M, const int8_t *dig, const float *xsc, float *out, const float *res,
                                        uint32_t &ph, RingPos &pos, const uint8_t *ring, RQShared &sh, uint32_t n_slots, uint32_t spin_ns) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const uint32_t ring_s = smem_u32(ring), dig_s = smem_u32(dig), xsc_s = smem_u32(xsc);
    uint32_t r0, r1;
    cta_rows(M, ph++, r0, r1);
    const uint32_t nblk = K / 32, nseg = (K + RQ_SEGK - 1) / RQ_SEGK;
    // digit weights of this lane's two D columns (2t, 2t + 1): digits 0..3 live in columns 0..3, columns 4..7 are zero planes
    const float w0 = t == 0 ? 0.015625f : (t == 1 ? 9.5367431640625e-07f : 0.f);            // 2^-6, 2^-20
    const float w1 = t == 0 ? 1.220703125e-04f : (t == 1 ? 7.450580596923828e-09f : 0.f);   // 2^-13, 2^-27
    auto bfrag = [&](uint32_t b, uint2 &bd, float &sx) {   // B fragment (digits) of block b: plane g (g < 4), 8 bytes at 8t
        const bool ok = b < nblk;
        bd = (g < 4 && ok) ? lds_u2(dig_s + (b * 4 + g) * 32 + t * 8) : make_uint2(0u, 0u);
        sx = ok ? lds_f(xsc_s + b * 4) : 0.f;
    };
    constexpr int NR = KREG ? KREG : 1;
    uint2 bdr[NR][2];
    float sxr[NR][2];
    if (KREG) {
#pragma unroll
        for (int sg = 0; sg < NR; sg++)
#pragma unroll
            for (int j = 0; j < 2; j++) bfrag((uint32_t)sg * (RQ_SEGK / 32) + warp * 2 + j, bdr[sg][j], sxr[sg][j]);
    }
    // offsets inside a FULL record (16 rows, 32 blocks): int8 rows g / g + 8 of blocks 2w, 2w + 1; their scales
    const uint32_t cA = ((uint32_t)warp * 2 * RQ_ROWS + g) * 32 + t * 8;
    const uint32_t cD = (RQ_SEGK / 32) * RQ_BLKQ + ((uint32_t)warp * 2 * RQ_ROWS + g) * 4;
    int buf = 0;
    for (uint32_t tile = r0; tile < r1; tile += RQ_ROWS) {
        const uint32_t rt = min((uint32_t)RQ_ROWS, r1 - tile);   // rows of this tile (the chunk's last tile may be short)
        const bool full_tile = rt == RQ_ROWS;
        const bool lo_row = (uint32_t)g < rt, hi_row = (uint32_t)g + 8 < rt;
        float acc[NM][2];
#pragma unroll
        for (int m = 0; m < NM; m++) acc[m][0] = acc[m][1] = 0.f;
        auto slot_math = [&](int m, const uint2 (&qa)[2], const uint2 (&qb)[2], const float (&da)[2], const float (&db)[2],
                             const uint2 (&bd)[2], const float (&sx)[2]) {
#pragma unroll
            for (int j = 0; j < 2; j++) {
                int c[4];
                mma_s8(c, qa[j].x, qb[j].x, qa[j].y, qb[j].y, bd[j].x, bd[j].y);
                // (the s32 -> f32 conversions stay on the I2F pipe, which is otherwise idle: the bit-pattern trick — 2 IADD + the
                //  offset folded into the FMA — moved them onto the ALU pipe, the busiest one: 437 vs 451 tok/s, r02o/r02q)
                const float va = fmaf((float)c[1], w1, __fmul_rn((float)c[0], w0));   // row g:     this lane's two digit columns
                const float vb = fmaf((float)c[3], w1, __fmul_rn((float)c[2], w0));   // row g + 8
                acc[m][0] = fmaf(va, __fmul_rn(da[j], sx[j]), acc[m][0]);
                acc[m][1] = fmaf(vb, __fmul_rn(db[j], sx[j]), acc[m][1]);
            }
        };
        auto do_seg = [&](uint32_t seg, const uint2 (&bd)[2], const float (&sx)[2]) {
            const uint32_t nb = min(RQ_SEGK / 32, nblk - seg * (RQ_SEGK / 32));   // blocks in this record (the last segment may be short)
            const bool fast = full_tile && nb == RQ_SEGK / 32;
#pragma unroll
            for (int m = 0; m < NM; m++) {
                mbar_wait<(1u << 24)>(smem_u32(&sh.full[pos.slot]), pos.phase, spin_ns);
                const uint32_t sl = ring_s + pos.slot * RQ_SLOT;
                uint2 qa[2], qb[2];
                float da[2], db[2];
                if (fast) {
                    const uint32_t pa = sl + cA, pd = sl + cD;
                    qa[0] = lds_u2(pa);                        // block 2w,     row g
                    qb[0] = lds_u2(pa + 8 * 32);               //               row g + 8
                    qa[1] = lds_u2(pa + RQ_BLKQ);              // block 2w + 1
                    qb[1] = lds_u2(pa + RQ_BLKQ + 8 * 32);
                    da[0] = lds_f(pd);
                    db[0] = lds_f(pd + 8 * 4);
                    da[1] = lds_f(pd + RQ_ROWS * 4);
                    db[1] = lds_f(pd + RQ_ROWS * 4 + 8 * 4);
                } else {
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        const uint32_t bl = warp * 2 + j;   // block inside the record: [bl][row < rt][32 int8], scales [bl][row] after the nb int8 blocks
                        const bool live = bl < nb;
                        qa[j] = live && lo_row ? lds_u2(sl + (bl * rt + g) * 32 + t * 8) : make_uint2(0u, 0u);        // row g, 8 int8
                        qb[j] = live && hi_row ? lds_u2(sl + (bl * rt + g + 8) * 32 + t * 8) : make_uint2(0u, 0u);    // row g + 8
                        da[j] = live && lo_row ? lds_f(sl + nb * rt * 32 + (bl * rt + g) * 4) : 0.f;
                        db[j] = live && hi_row ? lds_f(sl + nb * rt * 32 + (bl * rt + g + 8) * 4) : 0.f;
                    }
                }
                slot_math(m, qa, qb, da, db, bd, sx);
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(&sh.empty[pos.slot]));
                pos.next(n_slots);
            }
        };
        if (KREG) {
#pragma unroll
            for (int sg = 0; sg < NR; sg++)
                if ((uint32_t)sg < nseg) do_seg((uint32_t)sg, bdr[sg], sxr[sg]);
        } else {
#pragma unroll 1
            for (uint32_t seg = 0; seg < nseg; seg++) {
                uint2 bd[2];
                float sx[2];
#pragma unroll
                for (int j = 0; j < 2; j++) bfrag(seg * (RQ_SEGK / 32) + warp * 2 + j, bd[j], sx[j]);
                do_seg(seg, bd, sx);
            }
        }
        // digits 0,1 (lanes t = 0) + digits 2,3 (t = 1): the block scale d_w * s is common to both, so the two lanes' sums
        // are added once per tile instead of once per block
#pragma unroll
        for (int m = 0; m < NM; m++) {
            acc[m][0] += __shfl_xor_sync(0xffffffffu, acc[m][0], 1);
            acc[m][1] += __shfl_xor_sync(0xffffffffu, acc[m][1], 1);
        }
        // ---- combine the 16 warps' K-slices of this tile (lanes t == 0 hold rows g and g + 8); double-buffered partials:
        //      a buffer is rewritten two tiles later, after the next tile's barrier
        if (t == 0) {
#pragma unroll
            for (int m = 0; m < NM; m++) {
                sh.part[buf][m][warp][g] = acc[m][0];
                sh.part[buf][m][warp][g + 8] = acc[m][1];
            }
        }
        csync<RQ_CTHREADS>();
        if (threadIdx.x < RQ_ROWS) {
            const uint32_t row = tile + threadIdx.x;
            float s1 = 0.f, s3 = 0.f;
#pragma unroll
            for (int wv = 0; wv < RQ_CWARPS; wv++) {
                s1 += sh.part[buf][0][wv][threadIdx.x];
                if (NM == 2) s3 += sh.part[buf][NM - 1][wv][threadIdx.x];
            }
            if (row < r1) {
                float v;
                if (NM == 2) v = __fmul_rn(silu_ref(s1), s3);
                else if (EPI == 1) v = __fadd_rn(s1, __ldcg(res + row));
                else v = s1;
                out[row] = v;
            }
        }
        buf ^= 1;
    }
    csync<RQ_CTHREADS>();   // the last tile's partials are read before the next phase's prologue reuses shared memory
}

// dynamic shared memory: [ring: n_slots x RQ_SLOT][xs: kpad floats, digit planes in place][xsc: kpad/32 floats][scores][RQShared]
template <int HD>
__global__ void __launch_bounds__(RQ_THREADS, 1) decode_ring_q8_kernel(const RQParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const uint32_t dim = p.dim, ff = p.ff, n_slots = p.n_slots, kpad = p.kpad;
    uint8_t *ring = smem_raw;
    float *xs = reinterpret_cast<float *>(smem_raw + (size_t)n_slots * RQ_SLOT);
    int8_t *dig = reinterpret_cast<int8_t *>(xs);   // digit planes: 4 bytes per column, [block][plane][32]
    float *xsc = xs + kpad;
    const uint32_t kp_dim = (dim + RQ_SEGK - 1) / RQ_SEGK * RQ_SEGK, kp_ff = (ff + RQ_SEGK - 1) / RQ_SEGK * RQ_SEGK;
    float *scores = xsc + kpad / 32;
    RQShared &sh = *reinterpret_cast<RQShared *>(scores + 2 * (size_t)((p.chunk_cap + 3) & ~3u));
    const bool producer = threadIdx.x >= RQ_CTHREADS;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < n_slots; s++) {
            mbar_init(smem_u32(&sh.full[s]), 1);
            mbar_init(smem_u32(&sh.empty[s]), RQ_CWARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t past = p.state[0];
    rope_table<HD>(sh, past);
    __syncthreads();   // the only CTA-wide barrier

    RingPos pos;
    pos.slot = 0; pos.phase = 0;
    uint32_t ph = 0;   // MulMat phase counter (rotates the tile assignment; identical on both sides)
    if (producer) {
        if (threadIdx.x != RQ_CTHREADS) return;   // one thread drives the copy engine
        const uint32_t ring_base = smem_u32(ring);
        for (uint32_t li = 0; li < p.n_layers; li++) {
            const RingQ8Layer P = p.planes[li];
            produce<1>(P.wqkv, nullptr, dim, 3 * dim, ph, pos, ring_base, sh, n_slots);
            produce<1>(P.wo, nullptr, dim, dim, ph, pos, ring_base, sh, n_slots);
            produce<2>(P.w1, P.w3, dim, ff, ph, pos, ring_base, sh, n_slots);
            produce<1>(P.w2, nullptr, ff, dim, ph, pos, ring_base, sh, n_slots);
        }
        if (p.final_norm) produce<1>(p.out_plane, nullptr, dim, p.vocab, ph, pos, ring_base, sh, n_slots);
        return;
    }
    unsigned target = 0;
    const float *xin = p.x;
    if (p.tok_embeddings) xin = p.tok_embeddings + (size_t)p.tokens[p.state[1]] * dim;  // GetRows, llama.go:244
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
        stamp(li, 0);
        // ---- P1: rmsnorm * attention_norm, [wq;wk;wv] (llama.go:255-265)
        norm_digits(xin, L.attention_norm, dim, kp_dim, dig, xsc, sh);
        stamp(li, 1);
        consume<1, 0, 0>(dim, 3 * dim, dig, xsc, p.qkv, nullptr, ph, pos, ring, sh, n_slots, p.spin_ns);
        stamp(li, 2);
        grid_barrier<RQ_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 3);
        // ---- P2: RoPE, KV store, split attention partials (llama.go:274-333)
        attention_phase<HD, RQ_CTHREADS>(p, L, past, sh, scores);
        stamp(li, 4);
        grid_barrier<RQ_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 5);
        // ---- P3: merge the attention splits, wo + residual (llama.go:336-340)
        merge_digits<HD>(p, kp_dim, dig, xsc, sh);
        consume<1, 1, 0>(dim, dim, dig, xsc, p.y, xin, ph, pos, ring, sh, n_slots, p.spin_ns);
        stamp(li, 6);
        grid_barrier<RQ_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 7);
        // ---- P4: rmsnorm * ffn_norm, silu(w1.)*(w3.) (llama.go:346-361)
        norm_digits(p.y, L.ffn_norm, dim, kp_dim, dig, xsc, sh);
        stamp(li, 8);
        consume<2, 0, 0>(dim, ff, dig, xsc, p.act, nullptr, ph, pos, ring, sh, n_slots, p.spin_ns);
        stamp(li, 9);
        grid_barrier<RQ_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 10);
        // ---- P5: w2 + residual (llama.go:363-366)
        plain_digits(p.act, ff, kp_ff, dig, xsc);
        consume<1, 1, 0>(ff, dim, dig, xsc, p.x, p.y, ph, pos, ring, sh, n_slots, p.spin_ns);
        stamp(li, 11);
        grid_barrier<RQ_CTHREADS>(p.barrier, target, gridDim.x);
        stamp(li, 12);
        xin = p.x;
    }
    if (p.final_norm) {  // final norm + lm_head (llama.go:374-384)
        norm_digits(xin, p.final_norm, dim, kp_dim, dig, xsc, sh);
        consume<1, 0, 0>(dim, p.vocab, dig, xsc, p.logits, nullptr, ph, pos, ring, sh, n_slots, p.spin_ns);
    }
}

template <int HD>
static cudaError_t launch(const RQParams &p, size_t smem, cudaStream_t st) {
    static bool attr[64] = {};  // function attributes are per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !attr[dev]) {
        e = cudaFuncSetAttribute(decode_ring_q8_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs); cfg.blockDim = dim3(RQ_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, decode_ring_q8_kernel<HD>, p);
}

static uint32_t q8_splits(uint32_t heads) {
    uint32_t s = (2 * kNumSMs) / heads;
    return s < 1 ? 1 : (s > 32 ? 32 : s);
}
static uint32_t q8_plan(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t ctx, uint32_t *kpad_out, size_t *smem_out) {
    const uint32_t S = q8_splits(heads), chunk_cap = (ctx + S - 1) / S;
    const uint32_t kmax = dim > ff ? dim : ff, kpad = (kmax + RQ_SEGK - 1) / RQ_SEGK * RQ_SEGK;
    const size_t fixed = (size_t)kpad * 4 + (size_t)kpad / 32 * 4 + 2 * (size_t)((chunk_cap + 3) & ~3u) * 4 + sizeof(RQShared) + 128;
    const size_t cap = 227 * 1024;
    if (kpad_out) *kpad_out = kpad;
    if (fixed + 3 * (size_t)RQ_SLOT > cap) return 0;
    uint32_t n = (uint32_t)((cap - fixed) / RQ_SLOT);
    if (n > RQ_MAX_SLOTS) n = RQ_MAX_SLOTS;
    if (smem_out) *smem_out = fixed - 128 + (size_t)n * RQ_SLOT;
    return n;
}

// ---- interleaved planes (kernels_q8.cu) -> the tile-major decode plane this kernel streams ------------------------------
// plane = for tile (16 rows), for block b (32 columns): [16 rows][32 int8]; then per (tile, segment of 32 blocks) the
// scales [blocks of the segment][16 rows] f32 FOLLOW the segment's int8 blocks:  record(tile, seg) at
// (tile * K/32 + seg * 32) * 576 bytes = [nb][16][32] int8 | [nb][16] f32.  Rows >= `rows` of the last tile are zero.
__global__ void q8_to_tile_major_kernel(const int8_t *__restrict__ q, const float *__restrict__ d, uint8_t *__restrict__ plane,
                                        uint32_t M, uint32_t row0, uint32_t nrows, uint32_t K, uint32_t grid) {
    const uint32_t nblk = K / 32;
    const size_t n = (size_t)nrows * nblk * 8, stride = (size_t)gridDim.x * blockDim.x;   // one thread per (row, block, 4-byte group)
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t k4 = (uint32_t)(i & 7);
        const size_t rb = i >> 3;
        const uint32_t b = (uint32_t)(rb % nblk), lr = (uint32_t)(rb / nblk);   // lr: row inside q/d (the tensor's own planes)
        const uint32_t row = row0 + lr;                                           // row inside the whole matrix
        // the tile this row belongs to: first row g0, height rt
        uint32_t g0, rt;
        rq_group_of(M, row, grid, g0, rt);
        const uint32_t r = row - g0, seg = b / (RQ_SEGK / 32), bl = b % (RQ_SEGK / 32);
        const uint32_t nb = min(RQ_SEGK / 32, nblk - seg * (RQ_SEGK / 32));
        uint8_t *rec = plane + ((size_t)g0 * nblk + (size_t)seg * (RQ_SEGK / 32) * rt) * 36u;
        const uint32_t kcol = b * 32 + k4 * 4;
        const uint32_t w = *reinterpret_cast<const uint32_t *>(q + ((size_t)(lr >> 2) * (K >> 2) + (kcol >> 2)) * 16 + (lr & 3) * 4);
        *reinterpret_cast<uint32_t *>(rec + (bl * rt + r) * 32 + k4 * 4) = w;
        if (k4 == 0) *reinterpret_cast<float *>(rec + nb * rt * 32 + (bl * rt + r) * 4) = d[((size_t)(lr >> 2) * (K >> 5) + b) * 4 + (lr & 3)];
    }
}

}  // namespace

size_t q8_tile_major_bytes(uint32_t rows, uint32_t K) { return (size_t)rows * (K / 32) * 36u; }

// every record must start on and span a multiple of 16 bytes (bulk copy): K % 128 == 0 makes that true for any tile height;
// matrices that keep plain 16-row tiles only need whole tiles
static bool rq_layout_ok(uint32_t M, uint32_t K) {
    if (K % 32 || M % 4) return false;
    return rq_chunk_rows(M, kNumSMs) ? K % 128 == 0 : M % RQ_ROWS == 0;
}

void q8_to_tile_major(const int8_t *q, const float *d, uint8_t *plane, uint32_t M, uint32_t row0, uint32_t nrows, uint32_t K, cudaStream_t st) {
    if (!rq_layout_ok(M, K)) return;   // shapes the ring megakernel does not take (decode_ring_q8_supported): no decode plane
    LB_CHECK(row0 % 4 == 0 && nrows % 4 == 0 && row0 + nrows <= M, "q8_to_tile_major: bad row range");
    if (!nrows) return;
    q8_to_tile_major_kernel<<<148 * 8, 256, 0, st>>>(q, d, plane, M, row0, nrows, K, (uint32_t)kNumSMs);
    LB_LAUNCH_CHECK();
}

// layout queries for the CPU tests (tests/test_layouts.py): what=0 rows of work slot `idx` -> out {r0, r1};
// what=1 tile of row `idx` -> out {g0, rt, byte offset of the tile's segment-0 record (low, high 32 bits)}
bool ring_q8_layout_query(uint32_t what, uint32_t M, uint32_t K, uint32_t idx, uint32_t *out) {
    if (!rq_layout_ok(M, K)) return false;
    if (what == 0) {
        rq_rows_of(M, idx, kNumSMs, out[0], out[1]);
    } else {
        rq_group_of(M, idx, kNumSMs, out[0], out[1]);
        const uint64_t off = (uint64_t)out[0] * (K / 32) * 36u;
        out[2] = (uint32_t)off; out[3] = (uint32_t)(off >> 32);
    }
    return true;
}

bool decode_ring_q8_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx) {
    if (heads == 0 || dim % heads || heads > (uint32_t)RQ_MAX_HEADS) return false;
    const uint32_t hd = dim / heads;
    if (hd != 128 && hd != 64 && hd != 32) return false;
    if (dim % 32 || ff % 32 || dim < 256) return false;
    if (!rq_layout_ok(3 * dim, dim) || !rq_layout_ok(dim, dim) || !rq_layout_ok(ff, dim) || !rq_layout_ok(dim, ff) || !rq_layout_ok(vocab, dim)) return false;
    return q8_plan(dim, ff, heads, ctx, nullptr, nullptr) >= 3;
}

void decode_ring_q8(const MegaParamsHost &h, const RingQ8Layer *planes_dev, const uint8_t *out_plane, cudaStream_t st) {
    LB_CHECK(decode_ring_q8_supported(h.dim, h.ff, h.heads, h.vocab, h.ctx), "decode_ring_q8: unsupported shape");
    LB_CHECK(planes_dev != nullptr, "decode_ring_q8: decode planes missing");
    RQParams p;
    p.layers = h.layers_dev;
    p.planes = planes_dev;
    p.out_plane = out_plane;
    p.n_layers = h.n_layers;
    p.tok_embeddings = h.tok_embeddings; p.tokens = h.tokens; p.state = h.state;
    p.final_norm = h.final_norm;
    p.x = h.x; p.y = h.y; p.qkv = h.qkv; p.attn = h.attn; p.act = h.act; p.logits = h.logits;
    p.part_o = h.part_o; p.part_ml = h.part_ml; p.barrier = h.barrier;
    p.dim = h.dim; p.ff = h.ff; p.heads = h.heads; p.vocab = h.vocab; p.ctx = h.ctx;
    p.splits = q8_splits(h.heads);
    p.chunk_cap = (h.ctx + p.splits - 1) / p.splits;
    size_t smem = 0;
    p.n_slots = q8_plan(h.dim, h.ff, h.heads, h.ctx, &p.kpad, &smem);
    p.trace = reinterpret_cast<unsigned long long *>(h.trace);
    static const uint32_t spin_ns = getenv("LB_Q8_SPIN_NS") ? (uint32_t)atoi(getenv("LB_Q8_SPIN_NS")) : 0u;
    p.spin_ns = spin_ns;
    LB_CUDA(cudaMemsetAsync(h.barrier, 0, sizeof(unsigned) * 2, st));
    const uint32_t hd = h.dim / h.heads;
    cudaError_t e = hd == 128 ? launch<128>(p, smem, st) : hd == 64 ? launch<64>(p, smem, st) : launch<32>(p, smem, st);
    LB_CUDA(e);
    count_launch();
}

}  // namespace k
}  // namespace lb
