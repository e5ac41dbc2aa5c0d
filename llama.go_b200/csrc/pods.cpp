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

void PodBatch::ensure_sampler(uint32_t predict) {
    const uint32_t V = model->hp.vocab;
    if (!ring_dev) {
        ring_dev = mem.dmalloc<uint32_t>((size_t)B * ctx_size);
        ring_pos_dev = mem.dmalloc<uint32_t>(B);
        produced_dev = mem.dmalloc<uint32_t>(B);
        seeds_dev = mem.dmalloc<uint64_t>(B);
        smp_ids_dev = mem.dmalloc<uint32_t>((size_t)B * V);
        smp_probs_dev = mem.dmalloc<float>((size_t)B * V);
        smp_n_dev = mem.dmalloc<uint32_t>(B);
        smp_tok_dev = mem.dmalloc<uint32_t>(B);
    }
    if (predict > out_cap) {
        out_cap = predict;
        out_dev = mem.dmalloc<uint32_t>((size_t)B * out_cap, false);
    }
}

void PodBatch::sample(const uint32_t *last_n, uint32_t n_last, uint32_t top_k, float top_p, float temp, float repeat_penalty,
                      const uint64_t *seeds, uint32_t *ids_out, float *probs_out, uint32_t *n_out, uint32_t *tokens_out) {
    LB_CHECK(last_n || !n_last, "SampleTopPTopK : nil lastNTokens");
    LB_CHECK(seeds && tokens_out, "pod batch: nil argument");
    LB_CHECK(top_k >= 1 && top_k <= model->hp.vocab, "SampleTopPTopK : topK must be in 1..vocab");
    LB_CUDA(cudaSetDevice(model->device));
    ensure_sampler(0);
    if (n_last > smp_last_cap) {
        smp_last_cap = n_last;
        smp_last_dev = mem.dmalloc<uint32_t>((size_t)B * smp_last_cap, false);
    }
    LB_CUDA(cudaStreamSynchronize(stream));   // the previous call's buffers are idle before they are overwritten
    if (n_last) LB_CUDA(cudaMemcpyAsync(smp_last_dev, last_n, (size_t)B * n_last * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(seeds_dev, seeds, B * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    k::sample_top_p_top_k_pods(logits, model->hp.vocab, B, smp_last_dev, n_last, top_k, top_p, temp, repeat_penalty, seeds_dev,
                               smp_ids_dev, smp_probs_dev, smp_n_dev, smp_tok_dev, k::PodSampleState(), stream);
    std::vector<uint32_t> n(B);
    LB_CUDA(cudaMemcpyAsync(n.data(), smp_n_dev, B * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    LB_CUDA(cudaMemcpyAsync(tokens_out, smp_tok_dev, B * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    if (ids_out) LB_CUDA(cudaMemcpyAsync(ids_out, smp_ids_dev, (size_t)B * top_k * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    if (probs_out) LB_CUDA(cudaMemcpyAsync(probs_out, smp_probs_dev, (size_t)B * top_k * sizeof(float), cudaMemcpyDeviceToHost, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    if (n_out) memcpy(n_out, n.data(), B * sizeof(uint32_t));
}

// server.Do (server.go:127-237) for B jobs at once.  Context::generate's loop, restated per pod:
//   prompt phase: each pod's prompt in batch_size chunks through its own Context, with the same context_swap; the last
//     row of logits is copied into row b of the batch logits, so every pod's first sample is a batched one;
//   decode phase: [batched sample] then (predict - 1) x [pod step, batched sample].  A pod step evaluates each pod's
//     pending token at its own position, and every position grows by one per step, so the host knows the first step at
//     which some pod's pending token would land at past == ctx_size.  Every step up to there is enqueued as one segment
//     with no host synchronisation (segments also restart at kTokensCap steps, the token buffer's width).
//   context swap (server.go:165-172) of a pod that is due: its device ring, oldest first, goes through context_swap with
//     embd = [pending]; the re-fed prefix (which ends with the pending id itself, as in the reference) is evaluated
//     through the pod's Context at keep_count in one eval, and its past becomes keep_count + n_front.  The next pod step
//     then evaluates the pending id: the same tokens at the same positions as the reference's single Eval(embd).
// The last sampled id is never evaluated (server.go:153-237).
float PodBatch::generate(const uint32_t *prompts, const uint32_t *n_prompts, uint32_t predict, uint32_t top_k, float top_p, float temp,
                         float repeat_penalty, uint32_t keep_count, uint32_t batch_size, const uint64_t *seeds, uint32_t *out_tokens) {
    const HParams &hp = model->hp;
    const uint32_t V = hp.vocab;
    LB_CHECK(prompts && n_prompts && seeds && out_tokens && predict >= 1 && batch_size >= 1, "generate : bad arguments");
    std::vector<size_t> first(B);
    size_t off = 0;
    for (uint32_t b = 0; b < B; b++) {
        LB_CHECK(n_prompts[b] >= 1, "generate : bad arguments");
        first[b] = off;
        for (uint32_t i = 0; i < n_prompts[b]; i++) LB_CHECK(prompts[off + i] < V, "generate : token id out of range");
        off += n_prompts[b];
    }
    LB_CHECK(top_k >= 1 && top_k <= V, "SampleTopPTopK : topK must be in 1..vocab");
    LB_CHECK(temp > 0.f, "SampleTopPTopK : temp must be > 0 (the reference replaces 0 by 0.5, main.go:379-381)");
    LB_CHECK(keep_count < ctx_size, "generate : keep_count must be smaller than the context size");
    LB_CUDA(cudaSetDevice(model->device));
    ensure_sampler(predict);
    LB_CUDA(cudaStreamSynchronize(stream));

    // ---- prompt phase, per pod (Context::generate until its first sample)
    std::vector<uint32_t> ring((size_t)B * ctx_size, 0u), ring_pos(B, 0u), past(B, 0u), produced(B, 0u);
    std::vector<uint32_t> embd, tmp((size_t)ctx_size * 2 + batch_size);
    for (uint32_t b = 0; b < B; b++) {
        uint32_t *rb = ring.data() + (size_t)b * ctx_size;
        const uint32_t *prompt = prompts + first[b];
        uint32_t consumed = 0;
        embd.clear();
        for (;;) {
            if (!embd.empty()) {
                if ((uint64_t)past[b] + embd.size() > ctx_size) {   // server.go:165-172
                    std::vector<uint32_t> h(ctx_size);
                    for (uint32_t i = 0; i < ctx_size; i++) h[i] = rb[(ring_pos[b] + i) % ctx_size];
                    const int64_t n = context_swap(ctx_size, keep_count, h.data(), ctx_size, &past[b], embd.data(), (uint32_t)embd.size(),
                                                   tmp.data(), (uint32_t)tmp.size());
                    embd.assign(tmp.begin(), tmp.begin() + n);
                }
                ctxs[b]->eval(embd.data(), (uint32_t)embd.size(), past[b], nullptr, false);   // synchronous
            }
            past[b] += (uint32_t)embd.size();
            embd.clear();
            if (consumed == n_prompts[b]) break;
            while (consumed < n_prompts[b] && embd.size() < batch_size) {
                embd.push_back(prompt[consumed]);
                rb[ring_pos[b]] = prompt[consumed];
                ring_pos[b] = (ring_pos[b] + 1) % ctx_size;
                consumed++;
            }
        }
        LB_CUDA(cudaMemcpyAsync(logits + (size_t)b * V, ctxs[b]->logits, V * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    }
    // pageable sources: each copy returns once its data is staged, in stream order before the sampler
    LB_CUDA(cudaMemcpyAsync(ring_dev, ring.data(), ring.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(ring_pos_dev, ring_pos.data(), B * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(produced_dev, produced.data(), B * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(seeds_dev, seeds, B * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    pasts_host[8] = 0; pasts_host[9] = 0;   // state {unused, step}: the first sample writes token column 0
    LB_CUDA(cudaMemcpyAsync(state_dev, pasts_host + 8, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaStreamSynchronize(stream));

    // ---- decode phase
    k::PodSampleState g;
    g.ring = ring_dev; g.ring_pos = ring_pos_dev; g.produced = produced_dev; g.out = out_dev; g.out_stride = out_cap;
    g.tokens = tokens_dev; g.tok_stride = kTokensCap; g.state = state_dev;
    auto sample_all = [&]() {
        k::sample_top_p_top_k_pods(logits, V, B, ring_dev, ctx_size, top_k, top_p, temp, repeat_penalty, seeds_dev, nullptr, nullptr,
                                   nullptr, nullptr, g, stream);
    };
    LB_CUDA(cudaEventRecord(ev0, stream));
    sample_all();
    const uint32_t steps = predict - 1;
    uint32_t done = 0, col = 0;   // col = token column holding the pending ids (= state[1] on the device)
    while (done < steps) {
        LB_CUDA(cudaStreamSynchronize(stream));
        for (uint32_t b = 0; b < B; b++) {
            if (past[b] < ctx_size) continue;
            std::vector<uint32_t> rb(ctx_size), h(ctx_size);
            uint32_t pos = 0;
            LB_CUDA(cudaMemcpy(rb.data(), ring_dev + (size_t)b * ctx_size, ctx_size * sizeof(uint32_t), cudaMemcpyDeviceToHost));
            LB_CUDA(cudaMemcpy(&pos, ring_pos_dev + b, sizeof(uint32_t), cudaMemcpyDeviceToHost));
            for (uint32_t i = 0; i < ctx_size; i++) h[i] = rb[(pos + i) % ctx_size];
            const uint32_t pending = h[ctx_size - 1];   // the ring already ends with the pending id (server.go:207-211)
            const int64_t n = context_swap(ctx_size, keep_count, h.data(), ctx_size, &past[b], &pending, 1, tmp.data(), (uint32_t)tmp.size());
            if (n > 1) ctxs[b]->eval(tmp.data(), (uint32_t)(n - 1), past[b], nullptr, false);
            past[b] += (uint32_t)(n - 1);
        }
        uint32_t seg = steps - done < kTokensCap - 1 ? steps - done : kTokensCap - 1;
        for (uint32_t b = 0; b < B; b++) seg = ctx_size - past[b] < seg ? ctx_size - past[b] : seg;
        if (col) {   // move the pending ids to column 0 and restart the step counter
            LB_CUDA(cudaMemcpy2DAsync(tokens_dev, kTokensCap * sizeof(uint32_t), tokens_dev + col, kTokensCap * sizeof(uint32_t),
                                      sizeof(uint32_t), B, cudaMemcpyDeviceToDevice, stream));
            col = 0;
        }
        for (uint32_t b = 0; b < B; b++) pasts_host[b] = past[b];
        pasts_host[8] = 0; pasts_host[9] = 0;
        LB_CUDA(cudaMemcpyAsync(pasts_dev, pasts_host, B * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        LB_CUDA(cudaMemcpyAsync(state_dev, pasts_host + 8, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        ensure_graph();   // first use: an eager run of this very step, then capture (ensure_graph restores pasts / state)
        for (uint32_t i = 0; i < seg; i++) {
            LB_CUDA(cudaGraphLaunch(graph, stream));
            count_launch(use_mega ? 2 : model->layers.size() * 8 + 4);
            sample_all();
        }
        for (uint32_t b = 0; b < B; b++) past[b] += seg;
        col = seg;
        done += seg;
    }
    LB_CUDA(cudaEventRecord(ev1, stream));
    LB_CUDA(cudaMemcpy2DAsync(out_tokens, predict * sizeof(uint32_t), out_dev, out_cap * sizeof(uint32_t), predict * sizeof(uint32_t), B,
                              cudaMemcpyDeviceToHost, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    LB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    return ms;
}

}  // namespace llama
}  // namespace lb
