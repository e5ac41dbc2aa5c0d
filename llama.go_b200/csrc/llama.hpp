// llama.hpp — device-resident mirror of pkg/llama's Model / Context / Eval
// (pkg/llama/llama.go:83-113, 127-204, 211-426).
#pragma once
#include <stdint.h>

#include <map>
#include <memory>
#include <string>
#include <vector>

#include "ml.hpp"

namespace lb {
namespace llama {

struct HParams {  // llama.go:149-158
    uint32_t vocab = 0, dim = 0, mult = 0, heads = 0, layers = 0;
    uint32_t ff() const { return ((2 * (4 * dim) / 3 + mult - 1) / mult) * mult; }  // llama.go:761
    uint32_t head_dim() const { return dim / heads; }
};

struct Q8Mat {  // Q8_0 planes of one matrix: 4-row-interleaved q / d (kernels_q8.cu: per-op GEMV, tcgen05 GEMM) and the
                // tile-major decode plane streamed by the ring megakernel (kernels_ring_q8.cu: q8_to_tile_major)
    int8_t *q = nullptr;
    float *d = nullptr;
    uint8_t *tm = nullptr;      // decode plane of the WHOLE matrix this tensor is part of (wq/wk/wv share the [3*dim][dim] plane)
    uint32_t tm_row0 = 0;       // first row of this tensor inside that matrix
    uint32_t tm_rows = 0;       // rows of the whole matrix (the plane's row grouping depends on it)
};

struct Layer {  // llama.go:128-146; wq|wk|wv are stored as one [3*dim][dim] matrix
    float *attention_norm = nullptr;
    float *wqkv = nullptr;  // rows [0,dim) = wq, [dim,2dim) = wk, [2dim,3dim) = wv
    float *wo = nullptr;
    float *ffn_norm = nullptr;
    float *w1 = nullptr, *w2 = nullptr, *w3 = nullptr;
    Q8Mat wqkv8, wo8, w18, w28, w38;  // used instead of the float matrices when weight_type == Q8_0
    uint16_t *wqkvh = nullptr, *woh = nullptr, *w1h = nullptr, *w2h = nullptr, *w3h = nullptr;  // IEEE binary16 (weight_type == F16)
};

// llama.Model (llama.go:181-193) for one pipeline stage: layers [layer_begin, layer_end).
struct Model {
    DeviceOwner mem;  // first member: owns the weight slabs
    HParams hp;
    int device = 0;
    uint32_t layer_begin = 0, layer_end = 0;
    int weight_type = 0;
    bool has_embedding() const { return layer_begin == 0; }
    bool has_head() const { return layer_end == hp.layers; }

    float *slab = nullptr;  // one allocation for every weight of the stage
    size_t slab_floats = 0;
    float *tok_embeddings = nullptr, *norm = nullptr, *output = nullptr;
    Q8Mat output8;
    int8_t *qslab = nullptr;  // Q8_0: int8 plane of every MulMat matrix of the stage
    float *dslab = nullptr;   //       and the per-block scales
    uint8_t *tmslab = nullptr;   // the same matrices as tile-major decode planes (ring megakernel)
    uint16_t *hslab = nullptr;   // F16: every MulMat matrix of the stage as IEEE binary16, row-major
    uint16_t *outputh = nullptr;
    unsigned *f16_overflow = nullptr;  // F16: set by the device rounding when a finite value rounds to +-inf
    std::vector<Layer> layers;  // index = global layer - layer_begin
    bool f32() const { return weight_type == 0; }
    bool f16() const { return weight_type == 1; }
    bool q8() const { return weight_type == 16; }

    struct Entry { float *ptr; size_t nelem; uint64_t tid; float mean, sigma; Q8Mat q8; uint32_t cols = 0; uint16_t *h = nullptr; };
    std::map<std::string, Entry> tensors;  // ggjt names (llama.go:826-861) owned by this stage

    Model(const HParams &hp, int device, uint32_t lb, uint32_t le, int weight_type);
    ~Model();
    bool owns(const std::string &name) const { return tensors.count(name) != 0; }
    static bool known_name(const HParams &hp, const std::string &name);
    void set_tensor(const std::string &name, int dtype, const void *host, size_t nbytes);
    void get_tensor(const std::string &name, float *host, size_t nelem);
    void init_random(uint64_t seed);
    uint64_t weight_bytes_per_token() const;
    // n FP32 values on the device -> binary16 at dst, round to nearest even; a finite value that rounds to +-inf is an error
    void round_to_f16(const float *src, uint16_t *dst, size_t n, const std::string &name, cudaStream_t st);
};

// llama.Context (llama.go:83-113): FP32 KV cache in HBM + activations + stream + decode graph.
struct Context {
    DeviceOwner mem;  // first member: owns every buffer, event and the stream below
    Model *model;
    uint32_t ctx_size;
    cudaStream_t stream = nullptr;
    uint32_t max_batch;

    float *kv_k = nullptr, *kv_v = nullptr;  // [local_layers][ctx][dim]  (llama.go:93-97)
    float *x = nullptr, *y = nullptr, *cur = nullptr, *qkv = nullptr, *attn = nullptr, *act = nullptr, *up = nullptr;
    float *attn_scratch = nullptr; // split-T decode attention partials + tickets
    void *mega_layers_dev = nullptr;   // k::MegaLayerHost[local layers]
    unsigned *mega_barrier = nullptr;  // grid-barrier counter of the megakernel
    void *mega_trace = nullptr;        // LB_MEGA_TRACE=1: per-phase globaltimer stamps of CTA 0
    bool use_mega = false;             // single-token forward = one persistent cooperative kernel
    bool use_ring = false;             // ... the TMA-ring variant (kernels_ring.cu) instead of the register-fed one
    bool use_ring_q8 = false;          // Q8_0 weights: TMA ring + int8 tensor cores (kernels_ring_q8.cu)
    void *q8_planes_dev = nullptr;     // k::RingQ8Layer[local layers]
    float *logits = nullptr;       // [vocab] (last row)
    float *all_logits = nullptr;   // [max_batch][vocab], allocated on first use
    uint32_t *tokens_dev = nullptr;  // [max_batch + resident window]
    uint32_t tokens_cap = 0;
    uint32_t *ring_dev = nullptr, *present_dev = nullptr, *ring_pos_dev = nullptr;  // sampler state (last-N ring)
    uint32_t *smp_last_dev = nullptr, *smp_ids_dev = nullptr, *smp_nt_dev = nullptr, *smp_host = nullptr;  // top-k/top-p sampler buffers
    float *smp_probs_dev = nullptr;
    uint32_t smp_last_cap = 0;
    uint32_t *state_dev = nullptr;   // {past, step}
    uint32_t *state_host = nullptr;  // pinned {past, step}
    uint32_t *tokens_host = nullptr; // pinned staging
    float *logits_host = nullptr;    // pinned staging [vocab]
    cudaGraphExec_t decode_graph = nullptr;
    cudaGraphExec_t stage_graph = nullptr;   // this stage's layers for one token (pipeline mode)
    // fused stage hand-off over NVLink peer memory (pipeline.cpp p2p_export / p2p_import; kernels_ring.cu)
    uint32_t *p2p_flags = nullptr;       // local {in_flag, ack, seq, -}
    float *p2p_x_out = nullptr;          // downstream context's x, peer-mapped (cudaIpcOpenMemHandle)
    uint32_t *p2p_flag_out = nullptr;    // downstream context's flags, peer-mapped
    uint32_t *p2p_ack_out = nullptr;     // upstream context's flags, peer-mapped
    bool p2p_ready = false;              // import done: the stage graph is captured with the hand-off fused in
    bool p2p_on = false;                 // (set only while that graph is being captured)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    uint32_t last_n = 0;
    bool use_graph = true;

    Context(Model *m, uint32_t ctx_size);
    ~Context();

    // llama.Eval (llama.go:211-426), fused path
    void eval(const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out, bool all_rows,
              const float *hidden_in_dev = nullptr, float *hidden_out_dev = nullptr);
    // llama.Eval built node for node with the ml:: op API (slow path)
    void eval_graph(const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out);
    float decode_resident(const uint32_t *tokens, uint32_t steps, uint32_t past);
    // server.Do's generate loop at temp -> 0 (server.go:110-237) fully on the device: prompt eval, then
    // `predict` x (penalised argmax -> single-token eval); returns the generated ids
    void generate_greedy(const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, float temp, float repeat_penalty,
                         uint32_t *out_tokens);
    // llama.SampleTopPTopK (llama.go:455-707) on the device, on the logits of the last eval.  last_n = the ids of the
    // last-N ring (membership is all the reference uses, :501-511).  Returns the picked token; ids/probs (optional,
    // capacity top_k) receive the candidate set after the top-k and top-p cuts, *n_out its size.
    uint32_t sample(const uint32_t *last_n, uint32_t n_last, uint32_t top_k, float top_p, float temp, float repeat_penalty,
                    uint64_t seed, uint32_t *ids_out, float *probs_out, uint32_t *n_out);
    // the generate loop of pkg/server.Do (server.go:127-237): prompt in batches, context swap when the context is
    // full (:158-172), one sample per generated token; out_tokens receives the `predict` sampled ids
    void generate(const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, uint32_t top_k, float top_p, float temp,
                  float repeat_penalty, uint32_t keep_count, uint32_t batch_size, uint64_t seed, uint32_t *out_tokens);
    float bench_kernel(int which, uint32_t iters, uint32_t past, uint64_t *bytes_per_launch);
    // capture (once) the single-token forward of this stage's layers on stream `st`:
    // [embedding gather on stage 0] -> layers -> [norm + lm_head on the last stage] -> advance {past, step}
    void ensure_stage_graph(cudaStream_t st);
    // this stage's layers for n tokens, eagerly, on stream `st` (x holds the incoming residual on stages > 0)
    void forward_on(cudaStream_t st, uint32_t n);

   private:
    void forward(uint32_t n, bool tokens_indirect, bool all_rows, const float *hidden_in, float *hidden_out);
    void build_decode_graph();
};

// Pod batching (pods.cpp, SURVEY §8f-1): B contexts ("pods") of one model decode one token each per step
// in a single pass over the weights.
struct PodBatch {
    DeviceOwner mem;  // first member: owns every buffer, event and the stream below
    static constexpr uint32_t kTokensCap = 4096;
    std::vector<Context *> ctxs;
    Model *model = nullptr;
    uint32_t B = 0, ctx_size = 0;
    cudaStream_t stream = nullptr;
    float *x = nullptr, *y = nullptr, *cur = nullptr, *qkv = nullptr, *attn = nullptr, *act = nullptr, *logits = nullptr;
    float *attn_scratch = nullptr;
    float **kb_dev = nullptr, **vb_dev = nullptr;
    uint32_t *pasts_dev = nullptr, *state_dev = nullptr, *tokens_dev = nullptr;
    uint32_t *tokens_host = nullptr, *pasts_host = nullptr;
    float *logits_host = nullptr;
    cudaGraphExec_t graph = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool use_mega = false;              // one persistent megakernel per step (kernels_mega_pods.cu / kernels_ring_pods.cu)
    bool use_ring = false;              // ... the TMA-ring variant
    void *mega_layers_dev = nullptr;    // k::MegaLayerHost[layers]
    unsigned *mega_barrier = nullptr;
    std::vector<uint8_t> tmaps;         // TMA tensor maps of the weight matrices (k::ring_pods_make_maps)
    const void *tmaps_ptr = nullptr;
    void *mega_trace = nullptr;         // LB_MEGA_TRACE=1: per-phase globaltimer stamps of CTA 0 (TMA-ring variant)
    // batched sampler (allocated on first use): generate loop state [B][ctx] ring, [B] ring position / produced count,
    // [B][out_cap] sampled ids; one-shot sample inputs / outputs
    uint32_t *ring_dev = nullptr, *ring_pos_dev = nullptr, *produced_dev = nullptr, *out_dev = nullptr;
    uint32_t out_cap = 0;
    uint64_t *seeds_dev = nullptr;
    uint32_t *smp_last_dev = nullptr, *smp_ids_dev = nullptr, *smp_n_dev = nullptr, *smp_tok_dev = nullptr;
    float *smp_probs_dev = nullptr;
    uint32_t smp_last_cap = 0;

    explicit PodBatch(const std::vector<Context *> &ctxs);
    ~PodBatch();
    void eval(const uint32_t *tokens, const uint32_t *pasts, float *logits_out);          // one token per pod, host buffers
    float decode_resident(const uint32_t *tokens, uint32_t steps, const uint32_t *pasts);  // teacher-forced, device timed
    void read_logits(float *out);
    // Context::sample for every pod at once, on the batch's last logits: last_n [B][n_last], seeds [B]; tokens_out [B];
    // ids_out / probs_out ([B][top_k]) and n_out ([B]) optional, as in Context::sample
    void sample(const uint32_t *last_n, uint32_t n_last, uint32_t top_k, float top_p, float temp, float repeat_penalty,
                const uint64_t *seeds, uint32_t *ids_out, float *probs_out, uint32_t *n_out, uint32_t *tokens_out);
    // Context::generate (server.Do's loop) for every pod: pod b's prompt is the next n_prompts[b] ids of `prompts`, its
    // seed seeds[b]; the prompts go through each pod's own Context, then every step is one batched sample + one pod step
    // with no host round trip, except where a pod's context swap is due.  out_tokens [B][predict]; returns the CUDA-event
    // time of the decode phase in ms
    float generate(const uint32_t *prompts, const uint32_t *n_prompts, uint32_t predict, uint32_t top_k, float top_p, float temp,
                   float repeat_penalty, uint32_t keep_count, uint32_t batch_size, const uint64_t *seeds, uint32_t *out_tokens);

   private:
    void forward();
    void ensure_graph();
    void stage_inputs(const uint32_t *tokens, uint32_t steps, const uint32_t *pasts);
    void ensure_sampler(uint32_t predict);
};

}  // namespace llama
namespace pipe {
void unique_id(void *out128);
void comm_init(const void *id128, int rank, int world, int device);
void comm_destroy();
int nccl_version();
float pipeline_decode(llama::Context **ctxs, uint32_t n_seq, const uint32_t *tokens, uint32_t steps, uint32_t past);
void pipeline_prefill(llama::Context **ctxs, uint32_t n_seq, const uint32_t *tokens, uint32_t n, uint32_t past);
void p2p_export(llama::Context **ctxs, uint32_t n_seq, void *out /* n_seq x 128 bytes */);
void p2p_import(llama::Context **ctxs, uint32_t n_seq, const void *down /* n_seq x 128 or null */, const void *up /* or null */);
void p2p_disable(llama::Context **ctxs, uint32_t n_seq);
}  // namespace pipe
namespace llama {
// The context-swap rule of server.Do (pkg/server/server.go:158-172; main.go:190-200): when pastCount + len(embd)
// would exceed the context, keep the first `keep` positions, re-evaluate the last (pastCount - keep) / 2 tokens of
// the last-N history in front of embd.  history = ids oldest first (the ring in chronological order, which at that
// point already ends with the just-sampled token — the reference appends to the ring before it extends embd).
// Returns the new embd length (written to embd_out, capacity cap) and updates *past; no swap -> embd copied as is.
int64_t context_swap(uint32_t ctx_size, uint32_t keep, const uint32_t *history, uint32_t n_history, uint32_t *past,
                     const uint32_t *embd, uint32_t n_embd, uint32_t *embd_out, uint32_t cap);
// ggjt v1 file -> device model (loader.cpp); vocab strings/scores are returned for the tokenizer side
struct LoadedModel {
    std::unique_ptr<Model> model;
    std::vector<std::string> vocab;
    std::vector<float> scores;
    uint32_t tensors_loaded = 0;
};
LoadedModel load_ggjt(const std::string &path, int device, uint32_t layer_begin, uint32_t layer_end_or_0, int weight_type);
void synth_fill_host(float *dst, uint64_t count, uint64_t seed, uint64_t tid, uint64_t start, float mean, double sigma);

}  // namespace llama
}  // namespace lb
