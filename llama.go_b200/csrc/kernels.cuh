// kernels.cuh — launchers of every CUDA kernel in the library (definitions in kernels_*.cu).
// All pointers are device pointers; every launcher enqueues on `st` and returns immediately.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lb {

// strided view of a device tensor: mirrors ml.Tensor's NE/NB (pkg/ml/ml.go:187-188) with the
// strides already divided down to floats.
struct TView {
    float *data;
    uint32_t ne[4];
    uint32_t nb[4];
};

// Per-pod pointers of a batched decode step (SURVEY §8f-1): sequence b has its own KV cache base and
// position; all pods share the layer offset inside their caches (same ctx size) and the row pitches.
struct PodPtrs {
    float *const *K = nullptr;      // device array [B]: base of pod b's K cache
    float *const *V = nullptr;
    const uint32_t *pasts = nullptr;  // device array [B]: position of pod b's new token
    size_t layer_off = 0;           // floats: layer * ctx * dim
    uint32_t ldq = 0, ldo = 0;      // row pitch of q rows / output rows
};

namespace k {

// ---- generic op kernels (one per reference ComputeForward*; used by the pkg/ml mirror) ----
void get_rows_f32ids(const float *table, uint32_t nc, const float *ids, uint32_t nr, float *dst, cudaStream_t st);
void get_rows_u32ids(const float *table, uint32_t nc, const uint32_t *ids, uint32_t nr, float *dst, cudaStream_t st);
// y = x * f32(1/sqrt(mean_f64(x^2) + 1e-5)); if w != nullptr additionally y = y * w (w broadcast over rows)
void rms_norm(const float *x, const float *w, float *y, uint32_t nc, uint32_t nr, cudaStream_t st);
void repeat_rows(const float *a, uint32_t nc0, uint32_t nr0, float *dst, uint32_t nc, uint32_t nr, cudaStream_t st);
void mul(const float *a, const float *b, float *dst, size_t n, cudaStream_t st);
void add(const float *a, const float *b, float *dst, size_t n, cudaStream_t st);
void scale_inplace(float *x, float v, size_t n, cudaStream_t st);
void silu(const float *x, float *y, size_t n, cudaStream_t st);
void diag_mask_inf(float *x, uint32_t ne0, uint32_t ne1, uint32_t ne2, uint32_t past, cudaStream_t st);
void soft_max_rows(float *x, uint32_t nc, uint32_t nr, cudaStream_t st);
void cpy_strided(const TView &src, float *dst, cudaStream_t st);
// rope on a contiguous [ne0, ne1, ne2] tensor, in place (ComputeForwardRopeFP32, ml.go:2253-2328)
void rope(float *x, uint32_t ne0, uint32_t ne1, uint32_t ne2, uint32_t past, uint32_t dims, uint32_t mode, cudaStream_t st);
void mul_mat_generic(const TView &a, const TView &b, const TView &dst, cudaStream_t st);
void init_random(float *dst, uint64_t count, uint64_t seed, uint64_t tid, float mean, float sigma_scale, cudaStream_t st);
void f16_to_f32(const uint16_t *src, float *dst, size_t n, cudaStream_t st);
// binary16 round to nearest even (numpy's astype(float16)); *overflow = 1 if a finite value rounds to +-inf
void f32_to_f16(const float *src, uint16_t *dst, size_t n, unsigned *overflow, cudaStream_t st);

// ---- fused hot-path kernels (llama::Eval) ----
enum Epilogue { EPI_NONE = 0, EPI_ADD_RESIDUAL = 1 };
// y[n][m] = sum_k W[m][k] * x[n][k]   (+ residual[n][m]);  W row-major [M][K]; x rows ldx apart,
// y/residual rows ldy apart.  N = 1..8 columns per weight pass (decode / pod batch).
void gemv_f32(const float *W, uint32_t M, uint32_t K, const float *x, uint32_t ldx, uint32_t N,
              float *y, uint32_t ldy, const float *residual, cudaStream_t st);
// act[n][m] = silu(W1[m]·x[n]) * (W3[m]·x[n])   (llama.go:354-361)
void gemv_f32_swiglu(const float *W1, const float *W3, uint32_t M, uint32_t K, const float *x, uint32_t ldx,
                     uint32_t N, float *act, uint32_t ldy, cudaStream_t st);
// the same two with IEEE binary16 weights, widened in registers: each lane reads the elements it reads in the F32
// kernels and issues the same FMAs in the same order, so the results equal the F32 kernels' on the widened weights
void gemv_f16(const uint16_t *W, uint32_t M, uint32_t K, const float *x, uint32_t ldx, uint32_t N,
              float *y, uint32_t ldy, const float *residual, cudaStream_t st);
void gemv_f16_swiglu(const uint16_t *W1, const uint16_t *W3, uint32_t M, uint32_t K, const float *x, uint32_t ldx,
                     uint32_t N, float *act, uint32_t ldy, cudaStream_t st);
// prefill GEMM, any N: Y[n][m] = sum_k W[m][k] X[n][k] (+ residual)
void gemm_f32(const float *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
              float *Y, uint32_t ldy, const float *residual, cudaStream_t st);
void swiglu(const float *gate, const float *up, float *dst, size_t n, cudaStream_t st);
// prefill GEMM on tcgen05 tensor cores (kernels_tc.cu): TMA-fed kind::tf32 tiles, TMEM accumulators,
// FP32 operands split hi/lo in the shared-memory stage (3xTF32) so the result is FP32-class.
bool gemm_tf32x3_supported(uint32_t M, uint32_t K, uint32_t ldx, const float *W, const float *X);
void gemm_tf32x3(const float *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
                 float *Y, uint32_t ldy, const float *residual, cudaStream_t st);
// dispatcher for N > 8: tensor-core path when the shape allows (and LB_NO_TC is unset), else gemm_f32
void gemm_auto(const float *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
               float *Y, uint32_t ldy, const float *residual, cudaStream_t st);
// the same tcgen05 GEMM with a row-major binary16 weight operand (K % 32 == 0), widened in the shared-memory stage;
// binary16 is exact in TF32, so the weight has no lo part and each K step issues two MMAs (W*X_hi + W*X_lo)
void gemm_f16_tc(const uint16_t *W, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
                 float *Y, uint32_t ldy, const float *residual, cudaStream_t st);
// q (rows ldq apart, [N][dim]) rotated in place at positions past+n; k rotated and stored to
// Kc[(past+n)][dim]; v stored to Vc[(past+n)][dim]   (llama.go:274-297 — K is cached rotated)
// `past_dev` is a DEVICE pointer to the position of the first new token, so that a captured CUDA
// graph can be replayed for every decode step without re-baking the position.
void rope_qk_store(float *q, const float *k, const float *v, uint32_t ld, float *Kc, float *Vc,
                   uint32_t N, const uint32_t *past_dev, uint32_t dim, uint32_t heads, cudaStream_t st);
// causal attention over the FP32 cache: out[n][h*hd+d] for queries n (position past+n), head dim 128|64|32
// max_T bounds past+N (sizes the shared-memory score buffer at launch/capture time).
void attention(const float *q, uint32_t ldq, const float *Kc, const float *Vc, float *out, uint32_t N,
               const uint32_t *past_dev, uint32_t max_T, uint32_t dim, uint32_t heads, cudaStream_t st);
// decode (N == 1) variant: T split over many CTAs per head + merge; scratch from
// attention_decode_scratch_floats() must be zero-initialised once (ticket counters).
void attention_decode(const float *q, const float *Kc, const float *Vc, float *out, const uint32_t *past_dev,
                      uint32_t max_T, uint32_t dim, uint32_t heads, float *scratch, cudaStream_t st);
size_t attention_decode_scratch_floats(uint32_t heads, uint32_t hd);   // per pod
// pod batch: B sequences, each with its own cache / position (pods.*), one launch
void attention_decode_pods(const float *q, float *out, uint32_t B, const PodPtrs &pods, uint32_t max_T, uint32_t dim,
                           uint32_t heads, float *scratch, cudaStream_t st);
void rope_qk_store_pods(float *q, const float *k, const float *v, uint32_t ld, uint32_t B, const PodPtrs &pods, uint32_t dim,
                        uint32_t heads, cudaStream_t st);
// row b = table[tokens[b * row_stride + *step_dev]]
void get_rows_pods(const float *table, uint32_t nc, const uint32_t *tokens, uint32_t row_stride, const uint32_t *step_dev,
                   uint32_t B, float *dst, cudaStream_t st);
// pasts[b] += 1 for b < B; state[1] (= step) += 1
void advance_pods(uint32_t *pasts, uint32_t *state, uint32_t B, cudaStream_t st);
// single-token embedding gather for graph replay: row = table[tokens[*step_dev + n]]
void get_rows_indirect(const float *table, uint32_t nc, const uint32_t *tokens, const uint32_t *step_dev,
                       uint32_t nr, float *dst, cudaStream_t st);
// greedy (temp -> 0) sampling with the reference's repetition penalty, on the device (kernels_elementwise.cu)
void sample_greedy(const float *logits, uint32_t V, float scale, float penalty, uint32_t *present, uint32_t *ring,
                   uint32_t ring_size, uint32_t *ring_pos, uint32_t *tokens, const uint32_t *state, cudaStream_t st);
// SampleTopPTopK on the device (kernels_sample.cu): candidate ids/probabilities after the top-k and top-p cuts
// (out_ids/out_probs sized top_k), out_n_token = {count, picked token}
size_t sample_top_p_top_k_smem(uint32_t V, uint32_t top_k);
void sample_top_p_top_k(const float *logits, uint32_t V, const uint32_t *last_n_dev, uint32_t n_last, uint32_t top_k, float top_p,
                        float temp, float penalty, uint64_t seed, uint32_t *out_ids, float *out_probs, uint32_t *out_n_token,
                        cudaStream_t st);
// device state of the pods generate loop (every pointer device memory; all nullptr for a one-shot batch sample)
struct PodSampleState {
    uint32_t *ring = nullptr;       // [B][n_last] last-N ids (the sampler's last_n rows): the pick is appended at ring_pos
    uint32_t *ring_pos = nullptr;   // [B]
    uint32_t *produced = nullptr;   // [B] ids sampled so far: seed offset and column of `out`
    uint32_t *out = nullptr;        // [B][out_stride]
    uint32_t out_stride = 0;
    uint32_t *tokens = nullptr;     // [B][tok_stride]: the pick goes to column state[1], read by the next pod step
    uint32_t tok_stride = 0;
    const uint32_t *state = nullptr;
};
// the same sampler on B rows of logits ([B][V]), one CTA per pod: last_n rows n_last apart, pod b seeded with
// seeds_dev[b] (+ g.produced[b]); out_ids/out_probs [B][top_k], out_n/out_tok [B] (all optional)
void sample_top_p_top_k_pods(const float *logits, uint32_t V, uint32_t B, const uint32_t *last_n_dev, uint32_t n_last, uint32_t top_k,
                             float top_p, float temp, float penalty, const uint64_t *seeds_dev, uint32_t *out_ids, float *out_probs,
                             uint32_t *out_n, uint32_t *out_tok, const PodSampleState &g, cudaStream_t st);
// state[0] (= past) += dp; state[1] (= step) += ds; if seq != nullptr, *seq += 1 (pipeline hand-off step counter)
void advance_state(uint32_t *state, uint32_t dp, uint32_t ds, cudaStream_t st, uint32_t *seq = nullptr);

// ---- persistent single-token megakernel (kernels_mega.cu) ----
struct MegaLayerHost {  // one per layer, array lives in device memory
    const float *attention_norm, *wqkv, *wo, *ffn_norm, *w1, *w3, *w2;
    float *Kc, *Vc;
    // Q8_0 planes (nullptr for F32 models).  No kernel reads them (kernels_ring_q8.cu streams RingQ8Layer); they keep the
    // layout of this table, which the decode kernels' register allocation depends on.
    const int8_t *q_wqkv, *q_wo, *q_w1, *q_w3, *q_w2;
    const float *d_wqkv, *d_wo, *d_w1, *d_w3, *d_w2;
    const uint16_t *h_wqkv, *h_wo, *h_w1, *h_w3, *h_w2;  // binary16 matrices (F16 models, TMA-ring kernel only)
};
struct MegaParamsHost {
    const MegaLayerHost *layers_dev;
    uint32_t n_layers;
    const float *tok_embeddings;      // nullptr: residual comes in through x (pipeline stage > 0)
    const uint32_t *tokens, *state;   // device: token ids, {past, step}
    const float *final_norm, *output; // final_norm == nullptr: no lm_head on this stage
    bool f16 = false;                 // F16 weights: the layers' h_* matrices and h_output (decode_ring only)
    const uint16_t *h_output = nullptr;
    float *x, *y, *qkv, *attn, *act, *logits;
    float *part_o, *part_ml;
    unsigned *tickets, *barrier;
    uint32_t dim, ff, heads, vocab, ctx;
    void *trace = nullptr;            // optional uint64[n_layers*13] phase time stamps (profiling aid)
    // ---- fused stage hand-off over NVLink peer memory (pipeline stages, kernels_ring.cu only; all optional) ----
    // flags = this context's {in_flag, ack, seq, -} in LOCAL device memory: the upstream stage's kernel stores the
    // residual into this context's x and then in_flag = step number; the downstream stage stores ack = step number once
    // it has consumed what this stage sent; seq = steps this context has completed (advanced with the state).
    uint32_t *p2p_flags = nullptr;
    bool p2p_wait_in = false;         // wait for in_flag >= seq + 1 before touching x (stage > 0)
    float *p2p_x_out = nullptr;       // peer-mapped x of the downstream stage's context: the last phase writes the residual there
    uint32_t *p2p_flag_out = nullptr; // peer-mapped flags of the downstream context (its in_flag is [0])
    uint32_t *p2p_ack_out = nullptr;  // peer-mapped flags of the upstream context (its ack is [1])
};
bool decode_mega_supported(uint32_t dim, uint32_t ff, uint32_t heads);
uint32_t decode_mega_splits(uint32_t heads);
void decode_mega(const MegaParamsHost &p, cudaStream_t st);

// ---- the same token as one persistent kernel fed by a producer warp through a shared-memory ring of TMA bulk copies
//      (kernels_ring.cu): the weight stream runs ahead across phases and grid barriers
bool decode_ring_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx);
void ring_layout_query(uint32_t K, uint32_t *out);                                             // CPU layout tests
bool ring_q8_layout_query(uint32_t what, uint32_t M, uint32_t K, uint32_t idx, uint32_t *out);
void ring_pods_layout_query(uint32_t M, uint32_t idx, uint32_t *out);
void decode_ring(const MegaParamsHost &p, cudaStream_t st);

// ---- Q8_0 single-token decode on the TMA ring with the MulMat on the INT8 tensor cores (kernels_ring_q8.cu)
struct RingQ8Layer {   // tile-major decode planes (q8_to_tile_major) of one layer's matrices; array lives in device memory
    const uint8_t *wqkv, *wo, *w1, *w3, *w2;
};
size_t q8_tile_major_bytes(uint32_t rows, uint32_t K);
// rows [row0, row0 + nrows) of an M-row matrix (q/d: the 4-row-interleaved planes of THOSE rows) into the matrix's decode plane
void q8_to_tile_major(const int8_t *q, const float *d, uint8_t *plane, uint32_t M, uint32_t row0, uint32_t nrows, uint32_t K, cudaStream_t st);
bool decode_ring_q8_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx);
void decode_ring_q8(const MegaParamsHost &p, const RingQ8Layer *planes_dev, const uint8_t *out_plane, cudaStream_t st);

// ---- persistent pod-batch megakernel (kernels_mega_pods.cu): one decode step of B <= 8 pods, weights streamed once,
//      B-column MulMat on the tensor cores (mma.sync tf32, 3xTF32 split in registers)
struct MegaPodsParamsHost {
    const MegaLayerHost *layers_dev;
    uint32_t n_layers, B;
    const float *tok_embeddings;
    const uint32_t *tokens;        // device [B][tok_stride]
    uint32_t tok_stride;
    const uint32_t *state;         // device {unused, step}
    const uint32_t *pasts;         // device [B]
    float *const *Kb, *const *Vb;  // device [B]: cache bases of the pods
    const float *final_norm, *output;
    float *x, *y, *qkv, *attn, *act, *logits;
    float *part_o, *part_ml;
    unsigned *barrier;             // 2 counters, zeroed by the launcher
    const void *tmaps = nullptr;   // host pointer to the ring_pods_make_maps() blob (TMA-ring variant only)
    void *trace = nullptr;         // optional uint64[n_layers * 13] phase time stamps (TMA-ring variant, profiling aid)
    uint32_t dim, ff, heads, vocab, ctx;
};
bool decode_mega_pods_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx);
uint32_t decode_mega_pods_splits(uint32_t B, uint32_t heads);
void decode_mega_pods(const MegaPodsParamsHost &p, cudaStream_t st);
// the same step with the weights arriving through a producer warp's TMA ring (kernels_ring_pods.cu)
bool decode_ring_pods_supported(uint32_t dim, uint32_t ff, uint32_t heads, uint32_t vocab, uint32_t ctx);
void decode_ring_pods(const MegaPodsParamsHost &p, cudaStream_t st);
size_t ring_pods_maps_bytes();
void ring_pods_make_maps(const MegaLayerHost *layers_host, uint32_t n_layers, uint32_t dim, uint32_t ff, uint32_t vocab,
                         const float *output, void *maps_out);

// ---- Q8_0 block-quantised weights (kernels_q8.cu; format in DESIGN.md §6) ----
// W / out are plain row-major [rows][K]; q / d are the 4-row-interleaved planes (rows % 4 == 0, K % 32 == 0)
void quantize_q8(const float *W, int8_t *q, float *d, uint32_t rows, uint32_t K, cudaStream_t st);
void dequantize_q8(const int8_t *q, const float *d, float *out, uint32_t rows, uint32_t K, cudaStream_t st);
void gemv_q8(const int8_t *Q, const float *D, uint32_t M, uint32_t K, const float *x, uint32_t ldx, uint32_t N,
             float *y, uint32_t ldy, const float *residual, cudaStream_t st);
void gemv_q8_swiglu(const int8_t *Q1, const float *D1, const int8_t *Q3, const float *D3, uint32_t M, uint32_t K,
                    const float *x, uint32_t ldx, uint32_t N, float *act, uint32_t ldy, cudaStream_t st);
void gemm_q8(const int8_t *Q, const float *D, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
             float *Y, uint32_t ldy, const float *residual, cudaStream_t st);
// prefill GEMM on tcgen05 with the Q8_0 dequantisation fused into the shared-memory stage (kernels_tc.cu)
void gemm_q8_tc(const int8_t *Q, const float *D, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
                float *Y, uint32_t ldy, const float *residual, cudaStream_t st);
void gemm_q8_auto(const int8_t *Q, const float *D, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
                  float *Y, uint32_t ldy, const float *residual, cudaStream_t st);

}  // namespace k
}  // namespace lb
