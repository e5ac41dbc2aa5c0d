// kernels_mega.cu — the whole single-token forward pass (llama.Eval with N = 1,
// pkg/llama/llama.go:211-426) of a range of layers as ONE persistent cooperative kernel.
//
// Why: decode is HBM-bound (0.5 flop/byte) and a layer is only ~115 us of weight streaming; split
// into 7-8 kernels per layer, each kernel's ramp-up and tail leave HBM idle (measured: 162 us per
// layer with per-op kernels + PDL = 78 % of the measured-peak roofline).  Here 148 CTAs (one per
// SM, 16 warps) stay resident for the whole token and walk a static schedule of phases separated by
// grid barriers:
//   per layer:  P1 rmsnorm + [wq;wk;wv] GEMV | P2 RoPE + KV store + split-T attention (+ merge)
//               P3 wo GEMV + residual        | P4 rmsnorm + w1,w3 GEMV + SiLU*mul | P5 w2 GEMV + residual
//   then:       final rmsnorm + lm_head GEMV
// Work split of a GEMV phase: CTA c owns a contiguous block of ~M/148 output rows (balanced to one
// row); inside the CTA every warp owns a fixed 1/16 slice of K, so its slice of the activation vector
// lives in REGISTERS for the whole phase (no activation re-reads at all) and a weight row is read by
// 16 warps x 512-byte coalesced requests.  Row partials are combined through shared memory in a fixed
// order (deterministic).
// Measured and rejected (profiles/README.md): cp.async.bulk.prefetch.L2 of the next phase's rows before a
// barrier (no gain), a decoupled 17th prefetch warp with a progress window (544 threads cap the kernel at
// 96 registers, the GEMV loop spills: 142 tok/s), loading the next phase's first weight batch into
// registers across the barrier (no gain), 1-2-row dynamic blocks (too little in flight).
// Numerics are those of the per-op kernels (see kernels_elementwise.cu / kernels_attn.cu); only the
// association order of the FP32 dot-product sums differs.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"
#include "kernels.cuh"

#include <cstdlib>
#include <type_traits>

namespace lb {
namespace k {

constexpr int MG_WARPS = 16;
constexpr int MG_THREADS = MG_WARPS * 32;
constexpr int MG_HALF = MG_THREADS / 2;      // attention runs two items at a time, 8 warps each
constexpr int MG_ROWBLK = 32;          // rows whose partials are combined per __syncthreads
constexpr int MG_DYN_ROWS = 4;          // rows per dynamically scheduled block of a GEMV phase
constexpr int MG_MAX_ITEMS = 2 * kNumSMs;  // attention items (head, split) per layer: <= 2 per CTA (decode_mega_splits)
constexpr int MG_MAX_HEADS = 256;          // dim <= 8192 (largest K-slice variant), head dim >= 32
// CTA-wide and half-CTA named barriers
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, %0;" ::"n"(MG_THREADS) : "memory"); }
__device__ __forceinline__ void hsync(int half) { asm volatile("bar.sync %0, %1;" ::"r"(2 + half), "n"(MG_HALF) : "memory"); }

__device__ __forceinline__ float4 ldcg4(const float *p) { return __ldcg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct MegaShared {
    float part[2][2][MG_ROWBLK][MG_WARPS];  // [buffer][matrix (w1|w3)][row][warp]
    double red[MG_WARPS];
    float fred[2][MG_WARPS / 2];            // per attention half
    float bcast;
    float hbcast[2];
    unsigned ticket_slot[2];                // dynamic row-block tickets of the current GEMV phase
    float4 pv[MG_THREADS];                  // P·V partials: per half [key group][float4 lane of the head]
    double rope_cs[64][2];  // cos,sin(past * 10000^(-2j/hd)) for this token, j < hd/2 (once per launch)
    // merge of the attention splits (P3 prologue): per (head, split) m, l, weight; per head 1/L
    float mrg_m[MG_MAX_ITEMS], mrg_l[MG_MAX_ITEMS], mrg_w[MG_MAX_ITEMS], mrg_inv[MG_MAX_HEADS];
};

// ---- shared-memory head start of the NEXT MulMat phase (round 2) ---------------------------------------------
// HBM idles while the grid synchronises (~2 us per barrier + the RMSNorm prologue, ~8 us around the attention phase):
// nothing the CTA has in flight survives a phase boundary.  Weights do not depend on anything computed in the
// launch, so when a CTA has finished a phase, one thread issues cp.async.bulk copies (TMA engine, completion on an
// mbarrier) of the first rows of the CTA's static block of the NEXT phase into the otherwise unused shared memory
// (~190 KB: 12 rows of a 7B wq/wk/wv/wo, 2 x 6 rows of w1|w3, 4 rows of w2).  The copies are in flight during the
// barrier, the attention phase and the prologue; the next phase consumes those rows from shared memory (same
// K-slices, same arithmetic, LDS instead of LDG) at the END of its static part, so it never waits for them.
// (L2 prefetch hints at the same place measured no gain, profiles/README.md r02a: the async proxy is not held up by
// the polling thread's fences, and the bytes land where the consumer reads them at shared-memory speed.)
struct MegaPre {
    uint32_t buf;      // shared-memory address of the buffer (0: feature off)
    uint32_t bar;      // shared-memory address of its mbarrier
    uint32_t cap;      // bytes
};
__device__ __forceinline__ uint32_t mg_static_rows(uint32_t M) {   // static rows per CTA of a phase (see gemv_phase)
    return ((uint32_t)(((uint64_t)M * 4) / (5 * gridDim.x)) / MG_DYN_ROWS) * MG_DYN_ROWS;
}
__device__ __forceinline__ uint32_t mg_pre_rows(const MegaPre &pre, uint32_t M, uint32_t K, uint32_t NM) {
    if (!pre.buf) return 0;
    uint32_t n = pre.cap / (K * 4u * NM);
    const uint32_t Q = mg_static_rows(M);
    if (n > Q) n = Q;
    return n > (uint32_t)MG_ROWBLK ? (uint32_t)MG_ROWBLK : n;
}
// one thread: start the copies of the next phase's head rows (rows are adjacent in HBM: one copy per matrix row keeps
// every copy <= 88 KB; >= 8 KB copies run at the full HBM rate from a single issuing thread, profiles/README.md r02f)
__device__ __forceinline__ void mg_pre_issue(const MegaPre &pre, const float *W, const float *W3, uint32_t M, uint32_t K) {
    const uint32_t NM = W3 ? 2u : 1u, n = mg_pre_rows(pre, M, K, NM);
    if (!n) return;
    const uint32_t r0 = blockIdx.x * mg_static_rows(M), rb = K * 4u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pre.bar), "r"(n * rb * NM) : "memory");
    for (uint32_t m = 0; m < NM; m++) {
        const float *src = (m ? W3 : W) + (size_t)r0 * K;
        for (uint32_t r = 0; r < n; r++)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(pre.buf + (m * n + r) * rb), "l"(src + (size_t)r * K), "r"(rb), "r"(pre.bar) : "memory");
    }
}
__device__ __forceinline__ void mg_pre_wait(const MegaPre &pre, uint32_t parity) {
    const long long t0 = clock64();
    while (true) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(pre.bar), "r"(parity) : "memory");
        if (done) return;
        if (clock64() - t0 > 4000000000LL) __trap();  // ~2 s: never hang the GPU
    }
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}

// ---- fused pipeline-stage hand-off (multi-GPU layer sharding, SURVEY 8e; same protocol as kernels_ring.cu) ----
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

// ---- grid barrier: monotonically increasing counter, reset to 0 by a memset node before each launch
__device__ __forceinline__ void grid_barrier(unsigned *bar, unsigned &target, unsigned nctas, unsigned long long *arrive = nullptr, bool sys = false) {
    target += nctas;
    csync();
    if (threadIdx.x == 0) {
        if (arrive) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            arrive[blockIdx.x] = t;
        }
        if (sys) __threadfence_system();   // this CTA's stores to the peer GPU are ordered before the hand-off flag
        else __threadfence();
        atomicAdd(bar, 1u);
    }
    if (threadIdx.x == 0) {
        const long long t0 = clock64();
        while (ld_acquire_u32(bar) < target) {
            if (clock64() - t0 > 4000000000LL) __trap();  // never hang the GPU on a scheduling bug
        }
        __threadfence();
    }
    csync();
}

// this CTA's contiguous row range of an M-row matrix
__device__ __forceinline__ void cta_rows(uint32_t M, uint32_t &r0, uint32_t &r1) {
    r0 = (uint32_t)(((uint64_t)M * blockIdx.x) / gridDim.x);
    r1 = (uint32_t)(((uint64_t)M * (blockIdx.x + 1)) / gridDim.x);
}

// y = x * f32(1/sqrt(mean_f64(x^2)+1e-5)) * w, only this warp's K-slice, into registers
// (ComputeForwardRMSNormFP32 + Mul, ml.go:1753-1812, llama.go:255-259).  x may have been written by
// other CTAs during this launch -> L2 loads (ld.global.cg).
template <int V>
__device__ __forceinline__ void rms_slice(const float *x, const float *w, uint32_t K, float4 (&xs)[V], MegaShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t KS = K / MG_WARPS;
    // The 16 warps' K-slices tile x exactly once, so the slice this thread keeps is also its share of the sum
    // of squares: one L2 round trip instead of two.  f64 accumulation: per thread, per warp, then warps 0..15.
    float4 v[V], ww[V];
#pragma unroll
    for (int j = 0; j < V; j++) {
        const uint32_t e = (j * 32 + lane) * 4;
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        ww[j] = v[j];
        if (e < KS) {
            v[j] = ldcg4(x + (size_t)warp * KS + e);
            ww[j] = __ldg(reinterpret_cast<const float4 *>(w + (size_t)warp * KS + e));
        }
    }
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < V; j++) {
        acc += (double)__fmul_rn(v[j].x, v[j].x); acc += (double)__fmul_rn(v[j].y, v[j].y);
        acc += (double)__fmul_rn(v[j].z, v[j].z); acc += (double)__fmul_rn(v[j].w, v[j].w);
    }
    acc = warp_sum(acc);
    if (lane == 0) sh.red[warp] = acc;  // (a grid barrier separates this from the previous use of sh.red)
    csync();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < MG_WARPS; i++) t += sh.red[i];
    const float sc = (float)(1.0 / sqrt(t / (double)K + 1e-5));
#pragma unroll
    for (int j = 0; j < V; j++) {
        xs[j].x = __fmul_rn(ww[j].x, __fmul_rn(v[j].x, sc)); xs[j].y = __fmul_rn(ww[j].y, __fmul_rn(v[j].y, sc));
        xs[j].z = __fmul_rn(ww[j].z, __fmul_rn(v[j].z, sc)); xs[j].w = __fmul_rn(ww[j].w, __fmul_rn(v[j].w, sc));
    }
}

template <int V>
__device__ __forceinline__ void load_slice(const float *x, uint32_t K, float4 (&xs)[V]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t KS = K / MG_WARPS;
#pragma unroll
    for (int j = 0; j < V; j++) {
        const uint32_t e = (j * 32 + lane) * 4;
        xs[j] = e < KS ? ldcg4(x + (size_t)warp * KS + e) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// rows per load batch of a phase with V float4 per lane and NM matrices
__host__ __device__ constexpr int mg_rb(int V, int NM) { return (V * NM >= 10) ? 1 : (V * NM >= 6) ? 2 : (V * NM >= 3) ? 4 : 8; }

// One GEMV phase.  SWIGLU = false: out[r] = W[r]·xs (+ res[r]).  SWIGLU = true: out[r] = silu(W[r]·xs) * (W3[r]·xs).
// Scheduling: ~80 % of the rows are assigned statically (CTA c owns a contiguous block, processed
// 32 rows per shared-memory combine); the rest is a pool handed out 4 rows at a time through an
// atomic ticket (`ctr`, zeroed per launch), so SMs that stream faster take more rows and all CTAs
// reach the next grid barrier within one small block of each other (measured skew with a purely
// static split: 3-4 us per phase).  The next ticket is fetched while the current block streams.
template <int V, bool SWIGLU>
__device__ __forceinline__ void gemv_phase(const float *__restrict__ W, const float *__restrict__ W3, uint32_t M, uint32_t K,
                                           const float4 (&xs)[V], float *out, const float *res, MegaShared &sh, unsigned *ctr,
                                           const MegaPre &pre, uint32_t &pre_parity, bool peer_out = false) {
    constexpr int NM = SWIGLU ? 2 : 1;
    constexpr int RB = mg_rb(V, NM);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t KS = K / MG_WARPS;
    const float *w1 = W + (size_t)warp * KS + lane * 4;
    const float *w3 = SWIGLU ? W3 + (size_t)warp * KS + lane * 4 : nullptr;
    const uint32_t Q = mg_static_rows(M);  // static rows per CTA
    const uint32_t pool0 = Q * gridDim.x;
    const uint32_t npre = mg_pre_rows(pre, M, K, NM);   // the first npre static rows are (on their way) in shared memory
    if (threadIdx.x == 0) sh.ticket_slot[0] = atomicAdd(ctr, 1u);  // latency hidden behind the static part
    int buf = 0;
    // rows [rb, rb+nrb) -> partials -> combine -> out;  SM: the rows come from the head-start buffer (row rb = its row 0)
    auto do_block = [&](auto from_smem, uint32_t rb, uint32_t nrb) {
        constexpr bool SM = decltype(from_smem)::value;
        const uint32_t s1 = pre.buf + ((uint32_t)warp * KS + lane * 4) * 4u, s3 = s1 + npre * K * 4u;
        for (uint32_t r = 0; r < nrb; r += RB) {
            float4 a[RB][NM][V];
#pragma unroll
            for (int i = 0; i < RB; i++) {
                const bool rok = r + i < nrb;
                const size_t off = (size_t)(rb + r + i) * K;
                const uint32_t soff = (r + i) * K * 4u;
#pragma unroll
                for (int j = 0; j < V; j++) {
                    const bool ok = rok && (uint32_t)((j * 32 + lane) * 4) < KS;
                    if (SM) {
                        a[i][0][j] = ok ? lds_f4(s1 + soff + j * 512) : make_float4(0.f, 0.f, 0.f, 0.f);
                        if (SWIGLU) a[i][NM - 1][j] = ok ? lds_f4(s3 + soff + j * 512) : make_float4(0.f, 0.f, 0.f, 0.f);
                    } else {
                        a[i][0][j] = ok ? ld_stream_f4(w1 + off + j * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
                        if (SWIGLU) a[i][NM - 1][j] = ok ? ld_stream_f4(w3 + off + j * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < RB; i++) {
#pragma unroll
                for (int mtx = 0; mtx < NM; mtx++) {
                    float acc = 0.f;
#pragma unroll
                    for (int j = 0; j < V; j++) {
                        acc = fmaf(a[i][mtx][j].x, xs[j].x, acc); acc = fmaf(a[i][mtx][j].y, xs[j].y, acc);
                        acc = fmaf(a[i][mtx][j].z, xs[j].z, acc); acc = fmaf(a[i][mtx][j].w, xs[j].w, acc);
                    }
                    acc = warp_sum(acc);
                    if (lane == 0 && r + i < nrb) sh.part[buf][mtx][r + i][warp] = acc;
                }
            }
        }
        csync();
        if (threadIdx.x < nrb) {
            float s1 = 0.f, s3 = 0.f;
#pragma unroll
            for (int wv = 0; wv < MG_WARPS; wv++) {
                s1 += sh.part[buf][0][threadIdx.x][wv];
                if (SWIGLU) s3 += sh.part[buf][NM - 1][threadIdx.x][wv];
            }
            const uint32_t row = rb + threadIdx.x;
            float v;
            if (SWIGLU) v = __fmul_rn(silu_ref(s1), s3);
            else v = res ? __fadd_rn(s1, __ldcg(res + row)) : s1;
            out[row] = v;
            // out is the NEXT pipeline stage's buffer on another GPU: the WRITING thread orders its own store at system scope
            // (a fence by thread 0 after the CTA barrier does not cover other threads' stores still in flight over NVLink)
            if (peer_out) __threadfence_system();
        }
        buf ^= 1;  // the other partial buffer is used next; this one is reused only after the next csync
    };
    // static part: the rows that stream from HBM first, the head-start rows last (their copies have had the whole
    // barrier + prologue + this loop to land)
    const uint32_t r0 = blockIdx.x * Q, r1 = r0 + Q;
    for (uint32_t rb = r0 + npre; rb < r1; rb += MG_ROWBLK) do_block(std::false_type{}, rb, min((uint32_t)MG_ROWBLK, r1 - rb));
    if (npre) {
        mg_pre_wait(pre, pre_parity);
        pre_parity ^= 1u;
        do_block(std::true_type{}, r0, npre);   // its csync: every warp is done reading the buffer -> it may be refilled
    }
    // dynamic pool
    int slot = 0;
    csync();  // ticket_slot[0] written by thread 0 is visible
    uint32_t t = sh.ticket_slot[0];
    while ((uint64_t)pool0 + (uint64_t)t * MG_DYN_ROWS < M) {
        const uint32_t rb = pool0 + t * MG_DYN_ROWS;
        if (threadIdx.x == 0) sh.ticket_slot[slot ^ 1] = atomicAdd(ctr, 1u);  // next ticket, overlapped with this block
        do_block(std::false_type{}, rb, min((uint32_t)MG_DYN_ROWS, M - rb));  // contains a csync after the loads: the slot write is visible after it
        slot ^= 1;
        t = sh.ticket_slot[slot];
    }
}

struct MegaLayer {
    const float *attention_norm, *wqkv, *wo, *ffn_norm, *w1, *w3, *w2;
    float *Kc, *Vc;
    const int8_t *q_wqkv, *q_wo, *q_w1, *q_w3, *q_w2;  // Q8_0 planes (Q8 megakernel)
    const float *d_wqkv, *d_wo, *d_w1, *d_w3, *d_w2;
    const uint16_t *h_wqkv, *h_wo, *h_w1, *h_w3, *h_w2;  // F16 matrices (read by the TMA-ring kernel only)
};
struct MegaParams {
    const MegaLayer *layers;
    uint32_t n_layers;
    const float *tok_embeddings;  // nullptr: the residual stream comes in through x
    const uint32_t *tokens;
    const uint32_t *state;        // {past, step}
    const float *final_norm, *output;  // nullptr: no lm_head on this stage
    const int8_t *q_output;            // Q8 megakernel: lm_head planes
    const float *d_output;
    float *x, *y, *qkv, *attn, *act, *logits;
    float *part_o, *part_ml;
    unsigned *tickets, *barrier;
    uint32_t dim, ff, heads, vocab, ctx, splits, chunk_cap;
    unsigned long long *trace;  // optional: 13 globaltimer stamps per layer written by CTA 0 (profiling aid)
    uint32_t pre_bytes;         // shared-memory head start of the next MulMat phase: buffer size (0: off; LB_MEGA_PRE_KB)
    // fused stage hand-off over NVLink peer memory (see MegaParamsHost)
    uint32_t *p2p_flags;        // local {in_flag, ack, seq}
    uint32_t p2p_wait_in;
    float *p2p_x_out;
    uint32_t *p2p_flag_out, *p2p_ack_out;
};

// ---- attention phase: items (head, split); each CTA runs up to two items CONCURRENTLY, one per half
// (8 warps, own named barrier), so the latency chain of an item is paid once per layer.
template <int HD>
__device__ __forceinline__ void attention_phase(const MegaParams &p, const MegaLayer &L, uint32_t past, MegaShared &sh, float *scores_all) {
    constexpr int LANES = HD / 4;
    constexpr int HW = MG_WARPS / 2;     // warps per half
    constexpr int KG = MG_HALF / LANES;  // P·V key groups per half: thread (kg, dl) takes keys kg, kg + KG, ... for 4 dims
    constexpr int AU = 8;                // K rows per warp / V rows per thread in flight
    const int half = threadIdx.x / MG_HALF, ht = threadIdx.x % MG_HALF;
    const int hwarp = ht >> 5, lane = threadIdx.x & 31;
    const uint32_t dim = p.dim, S = p.splits, Tn = past + 1;
    const float scale = (float)(1.0 / sqrt((double)HD));  // f32(1/sqrt(dim/heads)), llama.go:306
    const uint32_t chunk = min((Tn + S - 1) / S, p.chunk_cap);
    const uint32_t items = p.heads * S;
    float *scores = scores_all + (size_t)half * p.chunk_cap;
    float4 *pv = sh.pv + half * MG_HALF;
    const uint32_t kg = ht / LANES, dl = ht % LANES;
    for (uint32_t item = blockIdx.x * 2 + half; item < items; item += gridDim.x * 2) {
        const uint32_t h = item / S, sp = item % S;
        const uint32_t t0 = min(sp * chunk, Tn), t1 = min(t0 + chunk, Tn), nk = t1 - t0;
        float *Kh = L.Kc + (size_t)h * HD;
        float *Vh = L.Vc + (size_t)h * HD;
        // RoPE of q (every warp, its own copy) and, in the item that owns position `past`, of k; store k,v
        // (ComputeForwardRopeFP32 ml.go:2253-2328; llama.go:274-297 — K is cached rotated)
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
        hsync(half);  // the freshly stored K/V row is visible to this half (read back through L2)
        // scores (MulMat K·Q, Scale): warp w takes keys w, w+HW, ... (AU keys in flight: one HBM round trip for
        // the 7B chunk of <= 57 keys)
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
        hsync(half);
        // local softmax statistics (SoftMax, ml.go:2472-2499, per split)
        float m = -INFINITY;
        for (uint32_t i = ht; i < nk; i += MG_HALF) m = fmaxf(m, scores[i]);
        m = warp_max(m);
        if (lane == 0) sh.fred[half][hwarp] = m;
        hsync(half);
        if (ht == 0) {
            float t = sh.fred[half][0];
            for (int i = 1; i < HW; i++) t = fmaxf(t, sh.fred[half][i]);
            sh.hbcast[half] = t;
        }
        hsync(half);
        m = sh.hbcast[half];
        float l = 0.f;
        for (uint32_t i = ht; i < nk; i += MG_HALF) {
            float e = (float)exp((double)__fsub_rn(scores[i], m));
            scores[i] = e;
            l += e;
        }
        l = warp_sum(l);
        hsync(half);
        if (lane == 0) sh.fred[half][hwarp] = l;
        hsync(half);
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
        hsync(half);
        if (ht < HD) {
            const float *pvf = reinterpret_cast<const float *>(pv);
            float r = 0.f;
            for (int i = 0; i < KG; i++) r += pvf[i * HD + ht];
            p.part_o[((size_t)h * S + sp) * HD + ht] = r;
        }
        hsync(half);  // scores / pv buffers are reused by the next item of this half
    }
}

// P3 prologue: merge the S split partials of the heads this warp's K-slice covers, straight into the
// register-resident activation slice:  out = (sum_s O_s * w_s) * f32(1 / sum_s l_s * w_s),
// w_s = expf(m_s - M), M = max_s m_s.  (The split/merge is this engine's reassociation of the
// reference's single-pass softmax; the merge weights use the FP32 expf — an f64 exp per lane and split
// measured 8 us per layer here — while the softmax terms themselves keep the reference's f64 exp.)
template <int V, int HD>
__device__ __forceinline__ void merged_attention_slice(const MegaParams &p, float4 (&xs)[V], MegaShared &sh) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t KS = p.dim / MG_WARPS, S = p.splits, items = p.heads * S;
    // Statistics first, by one thread per (head, split) and then per head, through shared memory; the partial
    // outputs are then fetched 12 splits at a time.  (A per-lane loop "read m,l -> if l > 0 read O_s"
    // is a chain of 2 dependent L2 round trips per split: 9 splits cost ~5 us per layer.)  The accumulation
    // order over the splits is unchanged, so are the bits.
    for (uint32_t i = threadIdx.x; i < items; i += MG_THREADS) {
        const float2 ml = __ldcg(reinterpret_cast<const float2 *>(p.part_ml) + i);
        sh.mrg_m[i] = ml.x;
        sh.mrg_l[i] = ml.y;
    }
    csync();
    for (uint32_t h = threadIdx.x; h < p.heads; h += MG_THREADS) {
        float M = -INFINITY;
        for (uint32_t s2 = 0; s2 < S; s2++) M = fmaxf(M, sh.mrg_m[h * S + s2]);
        float Lsum = 0.f;
        for (uint32_t s2 = 0; s2 < S; s2++) {
            const float l = sh.mrg_l[h * S + s2];
            float wgt = 0.f;
            if (l > 0.f) {
                wgt = expf(__fsub_rn(sh.mrg_m[h * S + s2], M));
                Lsum = fmaf(l, wgt, Lsum);
            }
            sh.mrg_w[h * S + s2] = wgt;
        }
        sh.mrg_inv[h] = __fdiv_rn(1.0f, Lsum);
    }
    csync();
    constexpr int MB = 12;  // splits per batch of loads: 7B has 9 splits, 13B 7, 30B 5, 65B 4
#pragma unroll
    for (int j = 0; j < V; j++) {
        const uint32_t e = (j * 32 + lane) * 4;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (e < KS) {
            const uint32_t g = warp * KS + e, h = g / HD, d = g % HD;
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
            o.x = __fmul_rn(o.x, inv); o.y = __fmul_rn(o.y, inv); o.z = __fmul_rn(o.z, inv); o.w = __fmul_rn(o.w, inv);
        }
        xs[j] = o;
    }
}

// dynamic shared memory: [scores: 2 x chunk_cap floats, padded to 128 B][head-start buffer: pre_bytes]
template <int VD, int VF, int HD>
__global__ void __launch_bounds__(MG_THREADS, 1) decode_mega_kernel(const MegaParams p) {
    extern __shared__ __align__(128) float scores[];  // [2][chunk_cap]
    __shared__ MegaShared sh;
    __shared__ __align__(8) unsigned long long pre_bar;
    const uint32_t dim = p.dim, ff = p.ff;
    unsigned target = 0;
    const uint32_t past = p.state[0];
    const float *xin = p.x;
    if (p.tok_embeddings) xin = p.tok_embeddings + (size_t)p.tokens[p.state[1]] * dim;  // GetRows, llama.go:244

    unsigned long long *tr = (p.trace && blockIdx.x == 0 && threadIdx.x == 0) ? p.trace : nullptr;
    // profiling aid: arrival time of every CTA at each of layer 5's barriers
    auto arr = [&](uint32_t li, int b) -> unsigned long long * {
        return (p.trace && li == 5 && p.n_layers > 6) ? p.trace + (size_t)p.n_layers * 13 + (size_t)b * gridDim.x : nullptr;
    };
    auto stamp = [&](uint32_t li, int i) {
        if (tr) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            tr[li * 13 + i] = t;
        }
    };
    // RoPE table of this token's position (ComputeForwardRopeFP32's pow/cos/sin in f64, ml.go:2307-2310)
    if (threadIdx.x < HD / 2) {
        double sn, cs;
        sincos((double)past * pow(10000.0, ((double)(-(int)(2 * threadIdx.x))) / (double)HD), &sn, &cs);
        sh.rope_cs[threadIdx.x][0] = cs;
        sh.rope_cs[threadIdx.x][1] = sn;
    }
    MegaPre pre;
    pre.cap = p.pre_bytes;
    pre.bar = (uint32_t)__cvta_generic_to_shared(&pre_bar);
    pre.buf = p.pre_bytes ? (uint32_t)__cvta_generic_to_shared(scores) + (((2 * p.chunk_cap * 4u) + 127u) & ~127u) : 0u;
    uint32_t pre_parity = 0;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(pre.bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    csync();
    // Pipeline stage hand-off fused into this kernel: the upstream stage's kernel stored the residual stream straight into this
    // context's x over NVLink and then raised in_flag.  Before this launch may overwrite the downstream context's x (in its
    // last phase) the downstream stage must have consumed the previous step: ack >= seq.
    unsigned p2p_seq = 0;
    if (p.p2p_flags) {
        p2p_seq = p.p2p_flags[2];
        if (threadIdx.x == 0) {
            if (p.p2p_wait_in) p2p_wait(p.p2p_flags + 0, p2p_seq + 1);
            if (p.p2p_x_out) p2p_wait(p.p2p_flags + 1, p2p_seq);
        }
        csync();
    }
    // thread 32 (warp 1; thread 0 fences and polls in the grid barriers) starts the head-start copies
    const bool pre_thread = threadIdx.x == 32;
    if (pre_thread && p.n_layers) mg_pre_issue(pre, p.layers[0].wqkv, nullptr, 3 * dim, dim);
    unsigned *sched = p.barrier + 1;  // [n_layers * 4 + 1] ticket counters, zeroed with the barrier
    for (uint32_t li = 0; li < p.n_layers; li++) {
        const MegaLayer L = p.layers[li];
        stamp(li, 0);
        {   // ---- P1: rmsnorm * attention_norm, then [wq;wk;wv] (llama.go:255-265)
            float4 xs[VD];
            rms_slice<VD>(xin, L.attention_norm, dim, xs, sh);
            stamp(li, 1);
            gemv_phase<VD, false>(L.wqkv, nullptr, 3 * dim, dim, xs, p.qkv, nullptr, sh, sched + li * 4 + 0, pre, pre_parity);
        }
        if (pre_thread) mg_pre_issue(pre, L.wo, nullptr, dim, dim);   // in flight under barrier 1, the attention phase, barrier 2
        stamp(li, 2);
        grid_barrier(p.barrier, target, gridDim.x, arr(li, 0));
        stamp(li, 3);
        // ---- P2: RoPE, KV store, split attention partials (llama.go:274-333)
        attention_phase<HD>(p, L, past, sh, scores);
        stamp(li, 4);
        grid_barrier(p.barrier, target, gridDim.x, arr(li, 1));
        stamp(li, 5);
        {   // ---- P3: merge the attention splits, wo + residual (llama.go:336-340)
            float4 xs[VD];
            merged_attention_slice<VD, HD>(p, xs, sh);
            gemv_phase<VD, false>(L.wo, nullptr, dim, dim, xs, p.y, xin, sh, sched + li * 4 + 1, pre, pre_parity);
        }
        if (pre_thread) mg_pre_issue(pre, L.w1, L.w3, ff, dim);
        stamp(li, 6);
        grid_barrier(p.barrier, target, gridDim.x, arr(li, 2));
        stamp(li, 7);
        {   // ---- P4: rmsnorm * ffn_norm, silu(w1·)·(w3·) (llama.go:346-361)
            float4 xs[VD];
            rms_slice<VD>(p.y, L.ffn_norm, dim, xs, sh);
            stamp(li, 8);
            gemv_phase<VD, true>(L.w1, L.w3, ff, dim, xs, p.act, nullptr, sh, sched + li * 4 + 2, pre, pre_parity);
        }
        if (pre_thread) mg_pre_issue(pre, L.w2, nullptr, dim, ff);
        stamp(li, 9);
        grid_barrier(p.barrier, target, gridDim.x, arr(li, 3));
        stamp(li, 10);
        {   // ---- P5: w2 + residual (llama.go:363-366)
            float4 xf[VF];
            load_slice<VF>(p.act, ff, xf);
            // (the stage's last layer writes the residual into the next stage's x)
            const bool to_peer = p.p2p_x_out != nullptr && li + 1 == p.n_layers;
            gemv_phase<VF, false>(L.w2, nullptr, dim, ff, xf, to_peer ? p.p2p_x_out : p.x, p.y, sh, sched + li * 4 + 3, pre, pre_parity, to_peer);
        }
        if (pre_thread) {
            if (li + 1 < p.n_layers) mg_pre_issue(pre, p.layers[li + 1].wqkv, nullptr, 3 * dim, dim);
            else if (p.final_norm) mg_pre_issue(pre, p.output, nullptr, p.vocab, dim);
        }
        stamp(li, 11);
        grid_barrier(p.barrier, target, gridDim.x, arr(li, 4), p.p2p_x_out != nullptr && li + 1 == p.n_layers);
        stamp(li, 12);
        xin = p.x;
    }
    if (p.final_norm) {  // final norm + lm_head (llama.go:374-384), row N-1 = the only row
        float4 xs[VD];
        rms_slice<VD>(xin, p.final_norm, dim, xs, sh);
        gemv_phase<VD, false>(p.output, nullptr, p.vocab, dim, xs, p.logits, nullptr, sh, sched + p.n_layers * 4, pre, pre_parity);
    }
    if (p.p2p_flags && blockIdx.x == 0 && threadIdx.x == 0) {
        // every CTA passed the last grid barrier (system-scope fences) after storing its rows of the residual
        __threadfence_system();
        if (p.p2p_flag_out) st_release_sys_u32(p.p2p_flag_out + 0, p2p_seq + 1);   // downstream: your input for step seq+1 is there
        if (p.p2p_ack_out) st_release_sys_u32(p.p2p_ack_out + 1, p2p_seq + 1);     // upstream: I am done with what you sent for step seq+1
    }
}


// =================================================================================================================
// EXPERIMENT (LB_Q8_MEGA=1, unmeasured): the decode megakernel for Q8_0 weights on the int8 tensor cores.
// Same phases, barriers, attention and merge as decode_mega_kernel.  A GEMV phase differs:
//  * the phase's activation vector (RMSNorm output / merged attention / SwiGLU output) is written to shared memory
//    and turned, one warp per Q8 block, into 4 balanced base-128 digits per element relative to the block's power
//    of two (exact to 2^-28 of the block maximum) stored as B fragments of mma.sync.m16n8k32.s8 (digit j = column j);
//  * work unit = a tile of 16 rows; the 16 warps of the CTA split the tile's K blocks, every warp feeds its
//    (16 rows x 32 k) sub-tiles from HBM straight into the A fragment (in the 4-row interleaved planes one 32-bit
//    word = 4 consecutive k of one row = one A register), one IMMA per sub-tile, s32 results exact, then
//    acc[row] += d_w[row][blk] * 2^e[blk] * sum_j 128^-(j+1) c_j;
//  * row partials of the 16 warps are combined through shared memory exactly as in gemv_phase.
// Fragment/index math: tools/studies/q8_mma_layout_emulation.py.  Numerics: tools/studies/q8_int8_digits.py.
constexpr int MGQ_U = 8;  // K blocks in flight per warp

__device__ __forceinline__ uint32_t ldq_stream_u32(const void *p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

struct MegaQ8Smem {       // carved out of dynamic shared memory after the attention scores
    float *vec;           // [Kmax]   the phase's activation vector
    uint32_t *bfrag;      // [Kmax/32][32] words: B fragments of the 16 lanes with gid < 4 (2 words each)
    float *xsc;           // [Kmax/32] 2^e per block
};

template <int V>
__device__ __forceinline__ void slice_to_smem(const float4 (&xs)[V], uint32_t K, float *vec) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t KS = K / MG_WARPS;
#pragma unroll
    for (int j = 0; j < V; j++) {
        const uint32_t e = (j * 32 + lane) * 4;
        if (e < KS) *reinterpret_cast<float4 *>(vec + (size_t)warp * KS + e) = xs[j];
    }
}

// vec (shared or global, K floats) -> B fragments + block scales; one warp per block of 32
__device__ __forceinline__ void q8_digits_phase(const float *vec, uint32_t K, const MegaQ8Smem &q, bool vec_global) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t NB = K >> 5;
    const int tig = (lane & 15) >> 2, reg = lane >> 4;   // where element `lane` of a block sits in the B fragment
    for (uint32_t b = warp; b < NB; b += MG_WARPS) {
        const float v = vec_global ? __ldcg(vec + (size_t)b * 32 + lane) : vec[(size_t)b * 32 + lane];
        const float mx = warp_max(fabsf(v));
        uint32_t pack = 0;
        float scale = 0.f;
        if (mx >= 1e-30f && mx <= 1e30f) {
            const int e = ilogbf(mx) + 2;  // |v| / 2^e < 0.5
            scale = ldexpf(1.0f, e);
            float r = v * ldexpf(1.0f, -e);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                r *= 128.0f;
                const float dj = rintf(r);
                r -= dj;
                pack |= ((uint32_t)(int)dj & 0xffu) << (8 * j);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            uint32_t w = ((pack >> (8 * j)) & 0xffu) << (8 * (lane & 3));
            w |= __shfl_xor_sync(0xffffffffu, w, 1);
            w |= __shfl_xor_sync(0xffffffffu, w, 2);
            if ((lane & 3) == 0) q.bfrag[(size_t)b * 32 + (j * 4 + tig) * 2 + reg] = w;  // column j, rows tig*4.. (+16)
        }
        if (lane == 0) q.xsc[b] = scale;
    }
}

// this warp's share (K blocks [b_begin, b_end)) of one 16-row tile of a Q8 matrix -> per-lane partial sums of rows
// R0 + gid (lo) and R0 + gid + 8 (hi), already reduced over the digit columns (valid in every lane of the quad)
__device__ __forceinline__ void q8_tile_partial(const int8_t *__restrict__ Q, const float *__restrict__ D, uint32_t R0, uint32_t K,
                                                uint32_t b_begin, uint32_t b_end, const MegaQ8Smem &q, float &out_lo, float &out_hi) {
    const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
    const uint32_t NB = K >> 5, K4 = K >> 2;
    const uint32_t r_lo = R0 + gid, r_hi = r_lo + 8;
    const uint32_t *qa = reinterpret_cast<const uint32_t *>(Q) + ((size_t)(r_lo >> 2) * K4 + tig) * 4 + (r_lo & 3);
    const uint32_t *qb = reinterpret_cast<const uint32_t *>(Q) + ((size_t)(r_hi >> 2) * K4 + tig) * 4 + (r_hi & 3);
    const float *da = D + (size_t)(r_lo >> 2) * NB * 4 + (r_lo & 3);
    const float *db = D + (size_t)(r_hi >> 2) * NB * 4 + (r_hi & 3);
    const float w0 = tig == 0 ? 0x1p-7f : 0x1p-21f, w1 = w0 * 0x1p-7f;  // tig 0: digits 0,1; tig 1: digits 2,3
    float acc_lo = 0.f, acc_hi = 0.f;
    for (uint32_t bb = b_begin; bb < b_end; bb += MGQ_U) {
        uint32_t a[MGQ_U][4];
        float s_lo[MGQ_U], s_hi[MGQ_U];
#pragma unroll
        for (int u = 0; u < MGQ_U; u++) {
            const uint32_t b = bb + u;
            const bool ok = b < b_end;
            const size_t w = (size_t)b * 32;
            a[u][0] = ok ? ldq_stream_u32(qa + w) : 0u;
            a[u][1] = ok ? ldq_stream_u32(qb + w) : 0u;
            a[u][2] = ok ? ldq_stream_u32(qa + w + 16) : 0u;
            a[u][3] = ok ? ldq_stream_u32(qb + w + 16) : 0u;
            s_lo[u] = ok ? __ldg(da + (size_t)b * 4) : 0.f;
            s_hi[u] = ok ? __ldg(db + (size_t)b * 4) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < MGQ_U; u++) {
            const uint32_t b = bb + u;
            if (b < b_end) {  // warp-uniform
                uint2 bf = make_uint2(0u, 0u);
                if (gid < 4) bf = *reinterpret_cast<const uint2 *>(q.bfrag + (size_t)b * 32 + (gid * 4 + tig) * 2);
                const float xs = q.xsc[b];
                int c0, c1, c2, c3;
                asm volatile(
                    "mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                    : "=r"(c0), "=r"(c1), "=r"(c2), "=r"(c3)
                    : "r"(a[u][0]), "r"(a[u][1]), "r"(a[u][2]), "r"(a[u][3]), "r"(bf.x), "r"(bf.y), "r"(0));
                const float v_lo = fmaf((float)c0, w0, (float)c1 * w1), v_hi = fmaf((float)c2, w0, (float)c3 * w1);
                acc_lo = fmaf(s_lo[u] * xs, v_lo, acc_lo);
                acc_hi = fmaf(s_hi[u] * xs, v_hi, acc_hi);
            }
        }
    }
    // digit columns live in tig 0 and 1; tig 2 and 3 hold the zero columns
    acc_lo += __shfl_xor_sync(0xffffffffu, acc_lo, 1); acc_lo += __shfl_xor_sync(0xffffffffu, acc_lo, 2);
    acc_hi += __shfl_xor_sync(0xffffffffu, acc_hi, 1); acc_hi += __shfl_xor_sync(0xffffffffu, acc_hi, 2);
    out_lo = acc_lo; out_hi = acc_hi;
}

constexpr int MGQ_TILE = 16;  // rows per work unit (one IMMA tile)

template <bool SWIGLU>
__device__ __forceinline__ void gemv_phase_q8(const int8_t *__restrict__ Q1, const float *__restrict__ D1, const int8_t *__restrict__ Q3,
                                              const float *__restrict__ D3, uint32_t M, uint32_t K, const MegaQ8Smem &q, float *out,
                                              const float *res, MegaShared &sh, unsigned *ctr) {
    constexpr int NM = SWIGLU ? 2 : 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
    const uint32_t NB = K >> 5;
    const uint32_t per = (NB + MG_WARPS - 1) / MG_WARPS, b_begin = min((uint32_t)warp * per, NB), b_end = min(b_begin + per, NB);
    const uint32_t tiles = M / MGQ_TILE;
    const uint32_t Qt = (uint32_t)(((uint64_t)tiles * 4) / (5 * gridDim.x));  // static tiles per CTA
    const uint32_t pool0 = Qt * gridDim.x;
    if (threadIdx.x == 0) sh.ticket_slot[0] = atomicAdd(ctr, 1u);
    int buf = 0;
    auto do_tiles = [&](uint32_t t0, uint32_t nt) {  // nt = 1 or 2 tiles (MG_ROWBLK = 32 rows per combine)
        for (uint32_t ti = 0; ti < nt; ti++) {
#pragma unroll
            for (int mtx = 0; mtx < NM; mtx++) {
                float lo, hi;
                q8_tile_partial(mtx ? Q3 : Q1, mtx ? D3 : D1, (t0 + ti) * MGQ_TILE, K, b_begin, b_end, q, lo, hi);
                if (tig == 0) {
                    sh.part[buf][mtx][ti * MGQ_TILE + gid][warp] = lo;
                    sh.part[buf][mtx][ti * MGQ_TILE + gid + 8][warp] = hi;
                }
            }
        }
        csync();
        if (threadIdx.x < nt * MGQ_TILE) {
            float s1 = 0.f, s3 = 0.f;
#pragma unroll
            for (int wv = 0; wv < MG_WARPS; wv++) {
                s1 += sh.part[buf][0][threadIdx.x][wv];
                if (SWIGLU) s3 += sh.part[buf][NM - 1][threadIdx.x][wv];
            }
            const uint32_t row = t0 * MGQ_TILE + threadIdx.x;
            float v;
            if (SWIGLU) v = __fmul_rn(silu_ref(s1), s3);
            else v = res ? __fadd_rn(s1, __ldcg(res + row)) : s1;
            out[row] = v;
        }
        buf ^= 1;
    };
    const uint32_t t0 = blockIdx.x * Qt, t1 = t0 + Qt;
    for (uint32_t t = t0; t < t1; t += 2) do_tiles(t, min(2u, t1 - t));
    int slot = 0;
    csync();
    uint32_t tk = sh.ticket_slot[0];
    while ((uint64_t)pool0 + tk < tiles) {
        const uint32_t t = pool0 + tk;
        if (threadIdx.x == 0) sh.ticket_slot[slot ^ 1] = atomicAdd(ctr, 1u);
        do_tiles(t, 1);
        slot ^= 1;
        tk = sh.ticket_slot[slot];
    }
}

template <int VD, int HD>
__global__ void __launch_bounds__(MG_THREADS, 1) decode_mega_q8_kernel(const MegaParams p, uint32_t kmax) {
    extern __shared__ float scores[];  // [2][chunk_cap] | vec [kmax] | bfrag [kmax/32][32] | xsc [kmax/32]
    __shared__ MegaShared sh;
    MegaQ8Smem q;
    q.vec = scores + ((2 * (size_t)p.chunk_cap + 3) & ~(size_t)3);  // 16-byte aligned (float4 stores)
    q.bfrag = reinterpret_cast<uint32_t *>(q.vec + kmax);
    q.xsc = reinterpret_cast<float *>(q.bfrag + (size_t)(kmax >> 5) * 32);
    const uint32_t dim = p.dim, ff = p.ff;
    unsigned target = 0;
    const uint32_t past = p.state[0];
    const float *xin = p.x;
    if (p.tok_embeddings) xin = p.tok_embeddings + (size_t)p.tokens[p.state[1]] * dim;
    if (threadIdx.x < HD / 2) {
        double sn, cs;
        sincos((double)past * pow(10000.0, ((double)(-(int)(2 * threadIdx.x))) / (double)HD), &sn, &cs);
        sh.rope_cs[threadIdx.x][0] = cs;
        sh.rope_cs[threadIdx.x][1] = sn;
    }
    csync();
    unsigned *sched = p.barrier + 1;
    // activation slice (registers) -> shared vector -> digits; every CTA does this redundantly, like the RMSNorm
    auto stage = [&](const float4 (&xs)[VD]) {
        slice_to_smem<VD>(xs, dim, q.vec);
        csync();
        q8_digits_phase(q.vec, dim, q, false);
        csync();
    };
    for (uint32_t li = 0; li < p.n_layers; li++) {
        const MegaLayer L = p.layers[li];
        {   // P1
            float4 xs[VD];
            rms_slice<VD>(xin, L.attention_norm, dim, xs, sh);
            stage(xs);
            gemv_phase_q8<false>(L.q_wqkv, L.d_wqkv, nullptr, nullptr, 3 * dim, dim, q, p.qkv, nullptr, sh, sched + li * 4 + 0);
        }
        grid_barrier(p.barrier, target, gridDim.x);
        attention_phase<HD>(p, L, past, sh, scores);
        grid_barrier(p.barrier, target, gridDim.x);
        {   // P3
            float4 xs[VD];
            merged_attention_slice<VD, HD>(p, xs, sh);
            stage(xs);
            gemv_phase_q8<false>(L.q_wo, L.d_wo, nullptr, nullptr, dim, dim, q, p.y, xin, sh, sched + li * 4 + 1);
        }
        grid_barrier(p.barrier, target, gridDim.x);
        {   // P4
            float4 xs[VD];
            rms_slice<VD>(p.y, L.ffn_norm, dim, xs, sh);
            stage(xs);
            gemv_phase_q8<true>(L.q_w1, L.d_w1, L.q_w3, L.d_w3, ff, dim, q, p.act, nullptr, sh, sched + li * 4 + 2);
        }
        grid_barrier(p.barrier, target, gridDim.x);
        {   // P5: the SwiGLU output was written by other CTAs -> digits straight from L2
            q8_digits_phase(p.act, ff, q, true);
            csync();
            gemv_phase_q8<false>(L.q_w2, L.d_w2, nullptr, nullptr, dim, ff, q, p.x, p.y, sh, sched + li * 4 + 3);
        }
        grid_barrier(p.barrier, target, gridDim.x);
        xin = p.x;
    }
    if (p.final_norm) {
        float4 xs[VD];
        rms_slice<VD>(xin, p.final_norm, dim, xs, sh);
        stage(xs);
        gemv_phase_q8<false>(p.q_output, p.d_output, nullptr, nullptr, p.vocab, dim, q, p.logits, nullptr, sh, sched + p.n_layers * 4);
    }
}

// ---- host side ---------------------------------------------------------------------------------
struct MegaHost {
    MegaParams p;
};

static bool pick_variant(uint32_t dim, uint32_t ff, uint32_t hd, int &vd, int &vf) {
    if (dim % (MG_WARPS * 4) || ff % (MG_WARPS * 4)) return false;
    if (hd != 128 && hd != 64 && hd != 32) return false;
    vd = (int)((dim / MG_WARPS + 127) / 128);
    vf = (int)((ff / MG_WARPS + 127) / 128);
    return true;
}

template <int VD, int VF, int HD>
static cudaError_t raise_smem_limit(size_t smem) {
    static size_t set_for[64] = {};  // function attributes are per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || set_for[dev] < smem) {
        e = cudaFuncSetAttribute(decode_mega_kernel<VD, VF, HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) set_for[dev] = smem;
    }
    return cudaSuccess;
}
template <int VD, int VF>
static cudaError_t launch_hd(const MegaParams &p, uint32_t hd, size_t smem, cudaStream_t st) {
    cudaError_t ea = hd == 128 ? raise_smem_limit<VD, VF, 128>(smem) : hd == 64 ? raise_smem_limit<VD, VF, 64>(smem) : raise_smem_limit<VD, VF, 32>(smem);
    if (ea != cudaSuccess) return ea;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs); cfg.blockDim = dim3(MG_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (hd == 128) return cudaLaunchKernelEx(&cfg, decode_mega_kernel<VD, VF, 128>, p);
    if (hd == 64) return cudaLaunchKernelEx(&cfg, decode_mega_kernel<VD, VF, 64>, p);
    return cudaLaunchKernelEx(&cfg, decode_mega_kernel<VD, VF, 32>, p);
}

bool decode_mega_supported(uint32_t dim, uint32_t ff, uint32_t heads) {
    int vd, vf;
    if (heads == 0 || dim % heads) return false;
    if (!pick_variant(dim, ff, dim / heads, vd, vf)) return false;
    // instantiated variants: (1,1) tiny test models, (2,6) 7B, (3,7) 13B, (4,9) 30B, (4,11) 65B
    return (vd == 1 && vf == 1) || (vd == 2 && vf == 6) || (vd == 3 && vf == 7) || (vd == 4 && vf == 9) || (vd == 4 && vf == 11);
}

uint32_t decode_mega_splits(uint32_t heads) {
    uint32_t s = (2 * kNumSMs) / heads;  // <= 2 attention items per CTA = one per half, run concurrently
    return s < 1 ? 1 : (s > 32 ? 32 : s);
}

bool decode_mega_q8_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab) {
    int vd, vf;
    if (heads == 0 || dim % heads) return false;
    if (!pick_variant(dim, ff, dim / heads, vd, vf) || vd > 4) return false;
    if (dim % 32 || ff % 32) return false;                                                  // whole Q8 blocks
    return (3 * dim) % MGQ_TILE == 0 && dim % MGQ_TILE == 0 && ff % MGQ_TILE == 0 && vocab % MGQ_TILE == 0;  // whole row tiles
}

template <int VD, int HDV>
static cudaError_t launch_q8_one(cudaLaunchConfig_t &cfg, const MegaParams &p, uint32_t kmax, size_t smem) {
    static size_t set_for = 0;  // the first (eager) launch raises the limit; graph capture then finds it set
    if (set_for < smem) {
        cudaError_t ea = cudaFuncSetAttribute(decode_mega_q8_kernel<VD, HDV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (ea != cudaSuccess) return ea;
        set_for = smem;
    }
    return cudaLaunchKernelEx(&cfg, decode_mega_q8_kernel<VD, HDV>, p, kmax);
}

template <int VD>
static cudaError_t launch_q8_hd(const MegaParams &p, uint32_t hd, uint32_t kmax, size_t smem, cudaStream_t st) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs); cfg.blockDim = dim3(MG_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (hd == 128) return launch_q8_one<VD, 128>(cfg, p, kmax, smem);
    if (hd == 64) return launch_q8_one<VD, 64>(cfg, p, kmax, smem);
    return launch_q8_one<VD, 32>(cfg, p, kmax, smem);
}

void decode_mega(const MegaParamsHost &h, cudaStream_t st) {
    MegaParams p;
    p.q_output = h.q_output; p.d_output = h.d_output;
    p.layers = reinterpret_cast<const MegaLayer *>(h.layers_dev);
    p.n_layers = h.n_layers;
    p.tok_embeddings = h.tok_embeddings; p.tokens = h.tokens; p.state = h.state;
    p.final_norm = h.final_norm; p.output = h.output;
    p.x = h.x; p.y = h.y; p.qkv = h.qkv; p.attn = h.attn; p.act = h.act; p.logits = h.logits;
    p.part_o = h.part_o; p.part_ml = h.part_ml; p.tickets = h.tickets; p.barrier = h.barrier;
    p.dim = h.dim; p.ff = h.ff; p.heads = h.heads; p.vocab = h.vocab; p.ctx = h.ctx;
    p.splits = decode_mega_splits(h.heads);
    p.chunk_cap = (h.ctx + p.splits - 1) / p.splits;
    int vd, vf;
    const uint32_t hd = h.dim / h.heads;
    LB_CHECK(pick_variant(h.dim, h.ff, hd, vd, vf) && decode_mega_supported(h.dim, h.ff, h.heads), "decode_mega: unsupported shape");
    size_t smem = 2 * (size_t)p.chunk_cap * sizeof(float);
    p.trace = reinterpret_cast<unsigned long long *>(h.trace);
    p.p2p_flags = h.q8 ? nullptr : h.p2p_flags; p.p2p_wait_in = h.p2p_wait_in ? 1u : 0u;
    p.p2p_x_out = h.p2p_x_out; p.p2p_flag_out = h.p2p_flag_out; p.p2p_ack_out = h.p2p_ack_out;
    // head-start buffer (opt-in, LB_MEGA_PRE_KB=<KB>): measured SLOWER than no buffer (profiles/README.md r02j: 180 tok/s with
    // 196 KB, 217 with 96 KB, 221.5 without) — every MulMat phase streams slower once the shared-memory carve-out
    // shrinks the L1 that the 128 KB of LDGs in flight per SM pass through, and the barriers grow with the copy traffic.
    static const uint32_t pre_kb = getenv("LB_MEGA_PRE_KB") ? (uint32_t)atoi(getenv("LB_MEGA_PRE_KB")) : 0u;
    p.pre_bytes = 0;
    if (!h.q8 && pre_kb) {
        const size_t scores_pad = (smem + 127) & ~(size_t)127;
        const size_t budget = 227 * 1024 - (sizeof(MegaShared) + 256);
        if (scores_pad + 32 * 1024 <= budget) {
            size_t pb = (budget - scores_pad) & ~(size_t)1023;
            if ((size_t)pre_kb * 1024 < pb) pb = (size_t)pre_kb * 1024;
            p.pre_bytes = (uint32_t)pb;
            smem = scores_pad + pb;
        }
    }
    LB_CUDA(cudaMemsetAsync(h.barrier, 0, sizeof(unsigned) * (2 + 4 * (size_t)h.n_layers), st));  // barrier + ticket counters
    cudaError_t e;
    if (h.q8) {  // experiment: Q8 megakernel (int8 tensor cores)
        LB_CHECK(decode_mega_q8_supported(h.dim, h.ff, h.heads, h.vocab), "decode_mega: unsupported Q8 shape");
        const uint32_t kmax = h.dim > h.ff ? h.dim : h.ff;
        const size_t smem_q8 = ((2 * (size_t)p.chunk_cap + 3) & ~(size_t)3) * 4 + (size_t)kmax * 4 + (size_t)(kmax / 32) * 32 * 4 + (size_t)(kmax / 32) * 4;
        LB_CHECK(smem_q8 <= 200 * 1024, "decode_mega: Q8 activation staging does not fit in shared memory");
        if (vd == 1) e = launch_q8_hd<1>(p, hd, kmax, smem_q8, st);
        else if (vd == 2) e = launch_q8_hd<2>(p, hd, kmax, smem_q8, st);
        else if (vd == 3) e = launch_q8_hd<3>(p, hd, kmax, smem_q8, st);
        else e = launch_q8_hd<4>(p, hd, kmax, smem_q8, st);
        LB_CUDA(e);
        count_launch();
        return;
    }
    if (vd == 1 && vf == 1) e = launch_hd<1, 1>(p, hd, smem, st);
    else if (vd == 2 && vf == 6) e = launch_hd<2, 6>(p, hd, smem, st);
    else if (vd == 3 && vf == 7) e = launch_hd<3, 7>(p, hd, smem, st);
    else if (vd == 4 && vf == 9) e = launch_hd<4, 9>(p, hd, smem, st);
    else e = launch_hd<4, 11>(p, hd, smem, st);
    LB_CUDA(e);
    count_launch();
}

static_assert(sizeof(MegaLayer) == sizeof(MegaLayerHost), "MegaLayer / MegaLayerHost layout mismatch");

}  // namespace k
}  // namespace lb
