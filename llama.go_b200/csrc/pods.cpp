// pods.cpp — pod batching (SURVEY.md §8f-1): one decode step of B independent sequences in a single pass
// over the weights.  The reference runs up to --pods concurrent jobs, each with its own llama.Context
// (KV cache) sharing one read-only Model (pkg/server/server.go:84-106, 151-175); on a GPU their N = 1
// evals are HBM-bound on the same weights, so the B tokens are evaluated as one B-column MulMat per
// weight: the weights stream once for B tokens.  Every pod keeps its own cache and position; RoPE, the
// KV store and attention run per pod inside one launch (blockIdx.z / row = pod).
#include <stdlib.h>

#include "llama.hpp"

namespace lb {
namespace llama {

PodBatch::PodBatch(const std::vector<Context *> &cs) : ctxs(cs) {
    B = (uint32_t)cs.size();
    LB_CHECK(B >= 1 && B <= 8, "pod batch: 1..8 contexts");
    model = cs[0]->model;
    ctx_size = cs[0]->ctx_size;
    LB_CHECK(model->has_embedding() && model->has_head(), "pod batch: needs a single-stage model");
    for (Context *c : cs) {
        LB_CHECK(c->model == model, "pod batch: contexts must share one model");
        LB_CHECK(c->ctx_size == ctx_size, "pod batch: contexts must have the same context size");
    }
    for (size_t i = 0; i < cs.size(); i++)
        for (size_t j = i + 1; j < cs.size(); j++) LB_CHECK(cs[i] != cs[j], "pod batch: the same context twice");
    const HParams &hp = model->hp;
    const size_t d = hp.dim, ff = hp.ff(), V = hp.vocab;
    LB_CUDA(cudaSetDevice(model->device));
    mem.device = model->device;
    stream = mem.stream();
    auto dalloc = [&](size_t floats) { return mem.dmalloc<float>(floats); };
    x = dalloc(B * d); y = dalloc(B * d); cur = dalloc(B * d); qkv = dalloc(B * 3 * d); attn = dalloc(B * d);
    act = dalloc(B * ff); logits = dalloc(B * V);
    attn_scratch = dalloc(B * k::attention_decode_scratch_floats(hp.heads, hp.head_dim()));
    std::vector<float *> kb(B), vb(B);
    for (uint32_t b = 0; b < B; b++) { kb[b] = cs[b]->kv_k; vb[b] = cs[b]->kv_v; }
    kb_dev = mem.dmalloc<float *>(B, false);
    vb_dev = mem.dmalloc<float *>(B, false);
    LB_CUDA(cudaMemcpy(kb_dev, kb.data(), B * sizeof(float *), cudaMemcpyHostToDevice));
    LB_CUDA(cudaMemcpy(vb_dev, vb.data(), B * sizeof(float *), cudaMemcpyHostToDevice));
    pasts_dev = mem.dmalloc<uint32_t>(8);
    state_dev = mem.dmalloc<uint32_t>(2);
    tokens_dev = mem.dmalloc<uint32_t>((size_t)B * kTokensCap);
    tokens_host = mem.hmalloc<uint32_t>((size_t)B * kTokensCap);
    pasts_host = mem.hmalloc<uint32_t>(10);
    logits_host = mem.hmalloc<float>(B * V);
    ev0 = mem.event();
    ev1 = mem.event();
    // one persistent megakernel per step (kernels_mega_pods.cu) for FP32 weights and supported shapes;
    // LB_NO_MEGA_PODS=1 keeps the per-op B-column kernels
    // (TMA-ring variant kernels_ring_pods.cu when the shape allows, LB_NO_RING_PODS=1: the register-fed kernels_mega_pods.cu)
    // (Q8_0 and F16 models keep the per-op B-column kernels)
    use_ring = getenv("LB_NO_MEGA_PODS") == nullptr && getenv("LB_NO_RING_PODS") == nullptr && model->f32() &&
               k::decode_ring_pods_supported(hp.dim, hp.ff(), hp.heads, hp.vocab, ctx_size);
    use_mega = use_ring || (getenv("LB_NO_MEGA_PODS") == nullptr && model->f32() &&
                            k::decode_mega_pods_supported(hp.dim, hp.ff(), hp.heads, hp.vocab, ctx_size));
    if (use_mega) {
        const size_t nl = model->layers.size();
        std::vector<k::MegaLayerHost> ml(nl);
        for (size_t i = 0; i < nl; i++) {
            const Layer &L = model->layers[i];
            ml[i] = k::MegaLayerHost();
            ml[i].attention_norm = L.attention_norm; ml[i].wqkv = L.wqkv; ml[i].wo = L.wo; ml[i].ffn_norm = L.ffn_norm;
            ml[i].w1 = L.w1; ml[i].w3 = L.w3; ml[i].w2 = L.w2;
        }
        mega_layers_dev = mem.dmalloc<k::MegaLayerHost>(nl, false);
        LB_CUDA(cudaMemcpy(mega_layers_dev, ml.data(), nl * sizeof(k::MegaLayerHost), cudaMemcpyHostToDevice));
        mega_barrier = mem.dmalloc<unsigned>(2);
        if (getenv("LB_MEGA_TRACE")) mega_trace = mem.dmalloc<unsigned long long>(nl * 13);
        if (use_ring) {
            tmaps.resize(k::ring_pods_maps_bytes() + 64);
            void *al = reinterpret_cast<void *>(((uintptr_t)tmaps.data() + 63) & ~(uintptr_t)63);
            k::ring_pods_make_maps(ml.data(), (uint32_t)nl, hp.dim, hp.ff(), hp.vocab, model->output, al);
            tmaps_ptr = al;
        }
    }
}

PodBatch::~PodBatch() {
    cudaSetDevice(model->device);
    if (stream) cudaStreamSynchronize(stream);
    if (graph) cudaGraphExecDestroy(graph);
    // buffers, events and the stream are released by `mem`
}

static void mm(const float *W, const Q8Mat &W8, const uint16_t *Wh, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
               float *Y, uint32_t ldy, const float *res, cudaStream_t st) {
    if (W8.q) k::gemv_q8(W8.q, W8.d, M, K, X, ldx, N, Y, ldy, res, st);
    else if (Wh) k::gemv_f16(Wh, M, K, X, ldx, N, Y, ldy, res, st);
    else k::gemv_f32(W, M, K, X, ldx, N, Y, ldy, res, st);
}

// llama.go:246-384 for B single-token rows, one row per pod
void PodBatch::forward() {
    const HParams &hp = model->hp;
    const uint32_t d = hp.dim, ff = hp.ff(), V = hp.vocab, H = hp.heads;
    cudaStream_t st = stream;
    if (use_mega) {
        k::MegaPodsParamsHost mp;
        mp.layers_dev = static_cast<const k::MegaLayerHost *>(mega_layers_dev);
        mp.n_layers = (uint32_t)model->layers.size(); mp.B = B;
        mp.tok_embeddings = model->tok_embeddings; mp.tokens = tokens_dev; mp.tok_stride = kTokensCap;
        mp.state = state_dev; mp.pasts = pasts_dev; mp.Kb = kb_dev; mp.Vb = vb_dev;
        mp.final_norm = model->norm; mp.output = model->output;
        mp.x = x; mp.y = y; mp.qkv = qkv; mp.attn = attn; mp.act = act; mp.logits = logits;
        mp.part_o = attn_scratch;
        mp.part_ml = attn_scratch + (size_t)B * H * 32 * hp.head_dim();
        mp.barrier = mega_barrier;
        mp.tmaps = tmaps_ptr;
        mp.trace = mega_trace;
        mp.dim = d; mp.ff = ff; mp.heads = H; mp.vocab = V; mp.ctx = ctx_size;
        if (use_ring) k::decode_ring_pods(mp, st);
        else k::decode_mega_pods(mp, st);
        k::advance_pods(pasts_dev, state_dev, B, st);
        return;
    }
    PodPtrs pp;
    pp.K = kb_dev; pp.V = vb_dev; pp.pasts = pasts_dev; pp.ldq = 3 * d; pp.ldo = d;
    k::get_rows_pods(model->tok_embeddings, d, tokens_dev, kTokensCap, state_dev + 1, B, x, st);
    for (size_t li = 0; li < model->layers.size(); li++) {
        const Layer &L = model->layers[li];
        pp.layer_off = li * (size_t)ctx_size * d;
        k::rms_norm(x, L.attention_norm, cur, d, B, st);
        mm(L.wqkv, L.wqkv8, L.wqkvh, 3 * d, d, cur, d, B, qkv, 3 * d, nullptr, st);
        k::rope_qk_store_pods(qkv, qkv + d, qkv + 2 * d, 3 * d, B, pp, d, H, st);
        k::attention_decode_pods(qkv, attn, B, pp, ctx_size, d, H, attn_scratch, st);
        mm(L.wo, L.wo8, L.woh, d, d, attn, d, B, y, d, x, st);
        k::rms_norm(y, L.ffn_norm, cur, d, B, st);
        if (model->q8()) k::gemv_q8_swiglu(L.w18.q, L.w18.d, L.w38.q, L.w38.d, ff, d, cur, d, B, act, ff, st);
        else if (model->f16()) k::gemv_f16_swiglu(L.w1h, L.w3h, ff, d, cur, d, B, act, ff, st);
        else k::gemv_f32_swiglu(L.w1, L.w3, ff, d, cur, d, B, act, ff, st);
        mm(L.w2, L.w28, L.w2h, d, ff, act, ff, B, x, d, y, st);
    }
    k::rms_norm(x, model->norm, cur, d, B, st);
    mm(model->output, model->output8, model->outputh, V, d, cur, d, B, logits, V, nullptr, st);
    k::advance_pods(pasts_dev, state_dev, B, st);
}

void PodBatch::ensure_graph() {
    if (graph) return;
    forward();  // eager warm-up (kernel attributes), then restore the state it advanced
    LB_CUDA(cudaMemcpyAsync(pasts_dev, pasts_host, B * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(state_dev, pasts_host + 8, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    cudaGraph_t g = nullptr;
    LB_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    try {
        forward();
    } catch (...) {
        cudaStreamEndCapture(stream, &g);
        if (g) cudaGraphDestroy(g);
        throw;
    }
    LB_CUDA(cudaStreamEndCapture(stream, &g));
    LB_CUDA(cudaGraphInstantiate(&graph, g, 0));
    cudaGraphDestroy(g);
}

void PodBatch::stage_inputs(const uint32_t *tokens, uint32_t steps, const uint32_t *pasts) {
    const HParams &hp = model->hp;
    LB_CHECK(tokens && pasts, "pod batch: nil argument");
    LB_CHECK(steps >= 1 && steps <= kTokensCap, "pod batch: too many steps");
    for (uint32_t b = 0; b < B; b++) {
        LB_CHECK((uint64_t)pasts[b] + steps <= ctx_size, "pod batch: past + steps exceeds the context size");
        pasts_host[b] = pasts[b];
        for (uint32_t i = 0; i < steps; i++) {
            LB_CHECK(tokens[(size_t)b * steps + i] < hp.vocab, "pod batch: token id out of range");
            tokens_host[(size_t)b * kTokensCap + i] = tokens[(size_t)b * steps + i];
        }
    }
    pasts_host[8] = 0; pasts_host[9] = 0;  // state {unused, step}
    LB_CUDA(cudaSetDevice(model->device));
    for (uint32_t b = 0; b < B; b++)
        LB_CUDA(cudaMemcpyAsync(tokens_dev + (size_t)b * kTokensCap, tokens_host + (size_t)b * kTokensCap, steps * sizeof(uint32_t),
                                cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(pasts_dev, pasts_host, B * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(state_dev, pasts_host + 8, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
}

void PodBatch::eval(const uint32_t *tokens, const uint32_t *pasts, float *logits_out) {
    stage_inputs(tokens, 1, pasts);
    ensure_graph();
    LB_CUDA(cudaGraphLaunch(graph, stream));
    count_launch(use_mega ? 2 : model->layers.size() * 8 + 4);
    const size_t nb = (size_t)B * model->hp.vocab * sizeof(float);
    if (logits_out) LB_CUDA(cudaMemcpyAsync(logits_host, logits, nb, cudaMemcpyDeviceToHost, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    if (logits_out) memcpy(logits_out, logits_host, nb);
}

float PodBatch::decode_resident(const uint32_t *tokens, uint32_t steps, const uint32_t *pasts) {
    stage_inputs(tokens, steps, pasts);
    ensure_graph();
    LB_CUDA(cudaStreamSynchronize(stream));
    LB_CUDA(cudaEventRecord(ev0, stream));
    for (uint32_t i = 0; i < steps; i++) {
        LB_CUDA(cudaGraphLaunch(graph, stream));
        count_launch(use_mega ? 2 : model->layers.size() * 8 + 4);
    }
    LB_CUDA(cudaEventRecord(ev1, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    LB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    return ms;
}

void PodBatch::read_logits(float *out) {
    LB_CUDA(cudaSetDevice(model->device));
    LB_CUDA(cudaStreamSynchronize(stream));
    LB_CUDA(cudaMemcpy(out, logits, (size_t)B * model->hp.vocab * sizeof(float), cudaMemcpyDeviceToHost));
}

}  // namespace llama
}  // namespace lb
