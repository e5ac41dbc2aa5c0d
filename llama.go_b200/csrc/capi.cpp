// capi.cpp — the extern "C" boundary declared in include/llamab200.h.
#include "../../include/llamab200.h"

#include <string.h>

#include <string>
#include <vector>

#include "llama.hpp"
#include "ml.hpp"

using namespace lb;

struct lb_model { llama::Model *m; };
struct lb_context { llama::Context *c; };
struct lb_mlctx { ml::Context *c; };
struct lb_graph { ml::Graph g; };
struct lb_batch { llama::PodBatch *b; };
// lb_tensor* is an ml::Tensor* (owned by its lb_mlctx)
static inline ml::Tensor *T(lb_tensor *t) { return reinterpret_cast<ml::Tensor *>(t); }
static inline const ml::Tensor *T(const lb_tensor *t) { return reinterpret_cast<const ml::Tensor *>(t); }
static inline lb_tensor *W(ml::Tensor *t) { return reinterpret_cast<lb_tensor *>(t); }

static thread_local std::string g_err;

#define LB_TRY_INT(body)                 \
    try {                                \
        body;                            \
        return 0;                        \
    } catch (const std::exception &e) {  \
        g_err = e.what();                \
        return 1;                        \
    } catch (...) {                      \
        g_err = "unknown error";         \
        return 1;                        \
    }
#define LB_TRY_PTR(type, expr)           \
    try {                                \
        return (type)(expr);             \
    } catch (const std::exception &e) {  \
        g_err = e.what();                \
        return nullptr;                  \
    } catch (...) {                      \
        g_err = "unknown error";         \
        return nullptr;                  \
    }

static void require_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        throw Error(std::string("no CUDA device is usable (there is no CPU fallback): ") + cudaGetErrorString(e));
    LB_CHECK(device >= 0 && device < n, "device index out of range");
    cudaDeviceProp p;
    LB_CUDA(cudaGetDeviceProperties(&p, device));
    LB_CHECK(p.major == 10, "this library is built for sm_100a (B200) only; device is sm_" + std::to_string(p.major) +
                                std::to_string(p.minor));
}

extern "C" {

const char *lb_last_error(void) { return g_err.c_str(); }
const char *lb_version(void) { return "llamab200 0.1 (sm_100a)"; }
uint64_t lb_kernel_launches(void) { return g_launches.load(); }

int lb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; i++) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ok++;
    }
    return ok;
}

lb_model *lb_model_create(const lb_hparams *hp, int device, uint32_t layer_begin, uint32_t layer_end, int weight_type) {
    try {
        LB_CHECK(hp != nullptr, "lb_model_create: nil hparams");
        require_device(device);
        llama::HParams h;
        h.vocab = hp->vocab; h.dim = hp->dim; h.mult = hp->mult; h.heads = hp->heads; h.layers = hp->layers;
        auto *m = new lb_model{nullptr};
        try {
            m->m = new llama::Model(h, device, layer_begin, layer_end, weight_type);
        } catch (...) { delete m; throw; }
        return m;
    } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
void lb_model_free(lb_model *m) { if (m) { delete m->m; delete m; } }
lb_model *lb_model_load_ggjt(const char *path, int device, uint32_t layer_begin, uint32_t layer_end, int weight_type, lb_hparams *hp_out) {
    try {
        LB_CHECK(path != nullptr, "lb_model_load_ggjt: nil path");
        require_device(device);
        llama::LoadedModel lm = llama::load_ggjt(path, device, layer_begin, layer_end, weight_type);
        if (hp_out) {
            const llama::HParams &h = lm.model->hp;
            hp_out->vocab = h.vocab; hp_out->dim = h.dim; hp_out->mult = h.mult; hp_out->heads = h.heads; hp_out->layers = h.layers;
        }
        auto *m = new lb_model{lm.model.release()};
        return m;
    } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
int lb_model_set_tensor(lb_model *m, const char *name, int dtype, const void *host, size_t nbytes) {
    LB_TRY_INT(LB_CHECK(m && name && host, "lb_model_set_tensor: nil argument"); m->m->set_tensor(name, dtype, host, nbytes));
}
int lb_model_get_tensor(lb_model *m, const char *name, float *host, size_t nelem) {
    LB_TRY_INT(LB_CHECK(m && name && host, "lb_model_get_tensor: nil argument"); m->m->get_tensor(name, host, nelem));
}
int lb_model_init_random(lb_model *m, uint64_t seed) { LB_TRY_INT(LB_CHECK(m, "nil model"); m->m->init_random(seed)); }
uint64_t lb_model_weight_bytes(const lb_model *m) { return m ? m->m->weight_bytes_per_token() : 0; }

int lb_synth_fill_host(float *dst, uint64_t count, uint64_t seed, uint64_t tid, uint64_t start, float mean, double sigma) {
    LB_TRY_INT(LB_CHECK(dst, "nil dst"); llama::synth_fill_host(dst, count, seed, tid, start, mean, sigma));
}
int lb_bench_kernel(lb_context *c, int which, uint32_t iters, uint32_t past, float *ms_out, uint64_t *bytes_out) {
    LB_TRY_INT(LB_CHECK(c && ms_out && bytes_out, "nil argument"); *ms_out = c->c->bench_kernel(which, iters, past, bytes_out));
}

lb_context *lb_context_create(lb_model *m, uint32_t ctx_size) {
    try {
        LB_CHECK(m != nullptr, "lb_context_create: nil model");
        auto *c = new lb_context{nullptr};
        try { c->c = new llama::Context(m->m, ctx_size); } catch (...) { delete c; throw; }
        return c;
    } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
void lb_context_free(lb_context *c) { if (c) { delete c->c; delete c; } }

int lb_eval(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out) {
    LB_TRY_INT(LB_CHECK(c, "nil context"); c->c->eval(tokens, n, past, logits_out, false));
}
int lb_eval_all_logits(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out) {
    LB_TRY_INT(LB_CHECK(c, "nil context"); c->c->eval(tokens, n, past, logits_out, true));
}
int lb_eval_graph(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out) {
    LB_TRY_INT(LB_CHECK(c && tokens, "nil argument"); c->c->eval_graph(tokens, n, past, logits_out));
}
int lb_decode_resident(lb_context *c, const uint32_t *tokens, uint32_t steps, uint32_t past, float *ms_out) {
    LB_TRY_INT(LB_CHECK(c && tokens, "nil argument"); float ms = c->c->decode_resident(tokens, steps, past); if (ms_out) *ms_out = ms);
}
int lb_generate_greedy(lb_context *c, const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, float temp, float repeat_penalty,
                       uint32_t *out_tokens) {
    LB_TRY_INT(LB_CHECK(c, "nil context"); c->c->generate_greedy(prompt, n_prompt, predict, temp, repeat_penalty, out_tokens));
}
int lb_sample_top_p_top_k(lb_context *c, const uint32_t *last_n_tokens, uint32_t n_last, uint32_t top_k, float top_p, float temp,
                          float repeat_penalty, uint64_t seed, uint32_t *cand_ids_out, float *cand_probs_out, uint32_t *n_cand_out,
                          uint32_t *token_out) {
    LB_TRY_INT(LB_CHECK(c && token_out, "nil argument");
               *token_out = c->c->sample(last_n_tokens, n_last, top_k, top_p, temp, repeat_penalty, seed, cand_ids_out, cand_probs_out, n_cand_out));
}
int lb_generate(lb_context *c, const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, uint32_t top_k, float top_p, float temp,
                float repeat_penalty, uint32_t keep_count, uint32_t batch_size, uint64_t seed, uint32_t *out_tokens) {
    LB_TRY_INT(LB_CHECK(c, "nil context");
               c->c->generate(prompt, n_prompt, predict, top_k, top_p, temp, repeat_penalty, keep_count, batch_size, seed, out_tokens));
}
int64_t lb_context_swap(uint32_t ctx_size, uint32_t keep_count, const uint32_t *history, uint32_t n_history, uint32_t *past_io,
                        const uint32_t *embd, uint32_t n_embd, uint32_t *embd_out, uint32_t cap) {
    try {
        return lb::llama::context_swap(ctx_size, keep_count, history, n_history, past_io, embd, n_embd, embd_out, cap);
    } catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}
int lb_context_read_logits(lb_context *c, float *out) {
    LB_TRY_INT(LB_CHECK(c && out, "nil argument"); LB_CHECK(c->c->model->has_head(), "this stage has no lm_head");
               LB_CUDA(cudaSetDevice(c->c->model->device));
               LB_CUDA(cudaMemcpyAsync(out, c->c->logits, c->c->model->hp.vocab * sizeof(float), cudaMemcpyDeviceToHost, c->c->stream));
               LB_CUDA(cudaStreamSynchronize(c->c->stream)));
}
int lb_context_read_kv(lb_context *c, uint32_t layer, uint32_t t0, uint32_t nt, float *k_out, float *v_out) {
    LB_TRY_INT(LB_CHECK(c, "nil context"); llama::Context *x = c->c;
               LB_CHECK(layer >= x->model->layer_begin && layer < x->model->layer_end, "layer not held by this stage");
               LB_CHECK((uint64_t)t0 + nt <= x->ctx_size, "kv range out of bounds");
               size_t d = x->model->hp.dim; size_t off = ((size_t)(layer - x->model->layer_begin) * x->ctx_size + t0) * d;
               LB_CUDA(cudaSetDevice(x->model->device)); LB_CUDA(cudaStreamSynchronize(x->stream));
               if (k_out) LB_CUDA(cudaMemcpy(k_out, x->kv_k + off, (size_t)nt * d * 4, cudaMemcpyDeviceToHost));
               if (v_out) LB_CUDA(cudaMemcpy(v_out, x->kv_v + off, (size_t)nt * d * 4, cudaMemcpyDeviceToHost)));
}
int lb_context_read_hidden(lb_context *c, uint32_t n, float *out) {
    LB_TRY_INT(LB_CHECK(c && out, "nil argument"); llama::Context *x = c->c; LB_CHECK(n <= x->max_batch, "n too large");
               LB_CUDA(cudaSetDevice(x->model->device)); LB_CUDA(cudaStreamSynchronize(x->stream));
               LB_CUDA(cudaMemcpy(out, x->x, (size_t)n * x->model->hp.dim * 4, cudaMemcpyDeviceToHost)));
}
int lb_context_mega_trace(lb_context *c, uint64_t *out, uint32_t n) {
    LB_TRY_INT(LB_CHECK(c && out, "nil argument"); LB_CHECK(c->c->mega_trace != nullptr, "no trace (set LB_MEGA_TRACE=1 before creating the context)");
               LB_CHECK(n <= c->c->model->layers.size() * 13 + 13 * 148, "trace: n too large");
               LB_CUDA(cudaSetDevice(c->c->model->device)); LB_CUDA(cudaStreamSynchronize(c->c->stream));
               LB_CUDA(cudaMemcpy(out, c->c->mega_trace, n * sizeof(uint64_t), cudaMemcpyDeviceToHost)));
}
int lb_context_synchronize(lb_context *c) {
    LB_TRY_INT(LB_CHECK(c, "nil context"); LB_CUDA(cudaSetDevice(c->c->model->device)); LB_CUDA(cudaStreamSynchronize(c->c->stream)));
}
int lb_eval_stage(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, const float *hidden_in_dev,
                  float *hidden_out_dev, float *logits_out) {
    LB_TRY_INT(LB_CHECK(c, "nil context"); c->c->eval(tokens, n, past, logits_out, false, hidden_in_dev, hidden_out_dev));
}
float *lb_context_hidden_buffer(lb_context *c) { return c ? c->c->x : nullptr; }
void *lb_context_stream(lb_context *c) { return c ? (void *)c->c->stream : nullptr; }
int lb_layout_query(uint32_t kind, uint32_t a, uint32_t b, uint32_t c, uint32_t out[4]) {
    if (!out) return -1;
    out[0] = out[1] = out[2] = out[3] = 0;
    switch (kind) {
        case 0: lb::k::ring_layout_query(a, out); return 0;
        case 1: return lb::k::ring_q8_layout_query(0, a, b, c, out) ? 0 : -1;
        case 2: return lb::k::ring_q8_layout_query(1, a, b, c, out) ? 0 : -1;
        case 3: lb::k::ring_pods_layout_query(a, c, out); return 0;
        default: return -1;
    }
}
const char *lb_context_decode_path(lb_context *c) {
    if (!c) return "";
    if (c->c->use_ring_q8) return "ring_q8";
    if (!c->c->use_mega) return "perop";
    if (c->c->use_ring) return c->c->model->f16() ? "ring_f16" : "ring";
    return "mega";
}

// ---- pod batching ----
lb_batch *lb_batch_create(lb_context **ctxs, uint32_t n) {
    try {
        LB_CHECK(ctxs && n >= 1, "lb_batch_create: nil argument");
        std::vector<llama::Context *> v(n);
        for (uint32_t i = 0; i < n; i++) { LB_CHECK(ctxs[i], "nil context"); v[i] = ctxs[i]->c; }
        auto *h = new lb_batch{nullptr};
        try { h->b = new llama::PodBatch(v); } catch (...) { delete h; throw; }
        return h;
    } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
void lb_batch_free(lb_batch *b) { if (b) { delete b->b; delete b; } }
int lb_batch_eval(lb_batch *b, const uint32_t *tokens, const uint32_t *pasts, float *logits_out) {
    LB_TRY_INT(LB_CHECK(b, "nil batch"); b->b->eval(tokens, pasts, logits_out));
}
int lb_batch_decode_resident(lb_batch *b, const uint32_t *tokens, uint32_t steps, const uint32_t *pasts, float *ms_out) {
    LB_TRY_INT(LB_CHECK(b, "nil batch"); float ms = b->b->decode_resident(tokens, steps, pasts); if (ms_out) *ms_out = ms);
}
int lb_batch_mega_trace(lb_batch *b, uint64_t *out, uint32_t n) {
    LB_TRY_INT(LB_CHECK(b && out, "nil argument"); llama::PodBatch *x = b->b;
               LB_CHECK(x->mega_trace != nullptr, "no trace buffer: create the batch with LB_MEGA_TRACE=1 in the environment");
               LB_CHECK(n <= x->model->layers.size() * 13, "trace: n too large");
               LB_CUDA(cudaSetDevice(x->model->device));
               LB_CUDA(cudaStreamSynchronize(x->stream));
               LB_CUDA(cudaMemcpy(out, x->mega_trace, (size_t)n * sizeof(uint64_t), cudaMemcpyDeviceToHost)));
}
int lb_batch_read_logits(lb_batch *b, float *logits_out) { LB_TRY_INT(LB_CHECK(b && logits_out, "nil argument"); b->b->read_logits(logits_out)); }

// ---- multi-GPU pipeline ----
int lb_comm_unique_id(void *out128) { LB_TRY_INT(LB_CHECK(out128, "nil argument"); pipe::unique_id(out128)); }
int lb_comm_init(const void *id128, int rank, int world, int device) {
    LB_TRY_INT(LB_CHECK(id128, "nil argument"); require_device(device); pipe::comm_init(id128, rank, world, device));
}
void lb_comm_destroy(void) { try { pipe::comm_destroy(); } catch (...) {} }
int lb_nccl_version(void) { try { return pipe::nccl_version(); } catch (const std::exception &e) { g_err = e.what(); return 0; } }
int lb_pipeline_decode(lb_context **ctxs, uint32_t n_seq, const uint32_t *tokens, uint32_t steps, uint32_t past, float *ms_out) {
    LB_TRY_INT(LB_CHECK(ctxs && n_seq >= 1, "nil argument");
               std::vector<llama::Context *> v(n_seq);
               for (uint32_t i = 0; i < n_seq; i++) { LB_CHECK(ctxs[i], "nil context"); v[i] = ctxs[i]->c; }
               float ms = pipe::pipeline_decode(v.data(), n_seq, tokens, steps, past);
               if (ms_out) *ms_out = ms);
}

int lb_pipeline_p2p_export(lb_context **ctxs, uint32_t n_seq, void *handles_out) {
    LB_TRY_INT(LB_CHECK(ctxs && n_seq >= 1 && handles_out, "nil argument");
               std::vector<llama::Context *> v(n_seq);
               for (uint32_t i = 0; i < n_seq; i++) { LB_CHECK(ctxs[i], "nil context"); v[i] = ctxs[i]->c; }
               pipe::p2p_export(v.data(), n_seq, handles_out));
}
int lb_pipeline_p2p_import(lb_context **ctxs, uint32_t n_seq, const void *downstream_handles, const void *upstream_handles) {
    LB_TRY_INT(LB_CHECK(ctxs && n_seq >= 1, "nil argument");
               std::vector<llama::Context *> v(n_seq);
               for (uint32_t i = 0; i < n_seq; i++) { LB_CHECK(ctxs[i], "nil context"); v[i] = ctxs[i]->c; }
               pipe::p2p_import(v.data(), n_seq, downstream_handles, upstream_handles));
}
int lb_pipeline_p2p_disable(lb_context **ctxs, uint32_t n_seq) {
    LB_TRY_INT(LB_CHECK(ctxs && n_seq >= 1, "nil argument");
               std::vector<llama::Context *> v(n_seq);
               for (uint32_t i = 0; i < n_seq; i++) { LB_CHECK(ctxs[i], "nil context"); v[i] = ctxs[i]->c; }
               pipe::p2p_disable(v.data(), n_seq));
}
int lb_pipeline_prefill(lb_context **ctxs, uint32_t n_seq, const uint32_t *tokens, uint32_t n, uint32_t past) {
    LB_TRY_INT(LB_CHECK(ctxs && n_seq >= 1, "nil argument");
               std::vector<llama::Context *> v(n_seq);
               for (uint32_t i = 0; i < n_seq; i++) { LB_CHECK(ctxs[i], "nil context"); v[i] = ctxs[i]->c; }
               pipe::pipeline_prefill(v.data(), n_seq, tokens, n, past));
}

// ---- pkg/ml mirror ----
lb_mlctx *lb_ml_new_context(int device) {
    try {
        require_device(device);
        auto *x = new lb_mlctx{nullptr};
        try { x->c = new ml::Context(device); } catch (...) { delete x; throw; }
        return x;
    } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
void lb_ml_release_context(lb_mlctx *ctx) { if (ctx) { delete ctx->c; delete ctx; } }

lb_tensor *lb_new_tensor(lb_mlctx *ctx, int dtype, uint32_t dims, uint32_t ne0, uint32_t ne1, uint32_t ne2, uint32_t ne3,
                         const float *host) {
    try {
        LB_CHECK(ctx, "nil context");
        LB_CHECK(dims >= 1 && dims <= 4, "NewTensor : dims must be 1..4");
        ml::Tensor *t = ml::NewTensor(ctx->c, (ml::DType)dtype, dims, ne0, ne1, ne2, ne3, nullptr, 0);
        if (host) {
            LB_CUDA(cudaMemcpyAsync(t->data, host, (size_t)t->nelements() * 4, cudaMemcpyHostToDevice, ctx->c->stream));
            LB_CUDA(cudaStreamSynchronize(ctx->c->stream));
        }
        return W(t);
    } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
int lb_tensor_write(lb_tensor *t, const float *host, size_t nelem) {
    LB_TRY_INT(LB_CHECK(t && host, "nil argument"); LB_CHECK(nelem <= T(t)->avail, "tensor write out of bounds");
               LB_CUDA(cudaMemcpy(T(t)->data, host, nelem * 4, cudaMemcpyHostToDevice)));
}
int lb_tensor_read(lb_tensor *t, float *host, size_t nelem) {
    LB_TRY_INT(LB_CHECK(t && host, "nil argument"); LB_CHECK(nelem <= T(t)->avail, "tensor read out of bounds");
               LB_CUDA(cudaDeviceSynchronize()); LB_CUDA(cudaMemcpy(host, T(t)->data, nelem * 4, cudaMemcpyDeviceToHost)));
}
int lb_tensor_shape(const lb_tensor *t, uint32_t ne[4], uint32_t nb[4]) {
    LB_TRY_INT(LB_CHECK(t, "nil tensor"); for (int i = 0; i < 4; i++) { if (ne) ne[i] = T(t)->ne[i]; if (nb) nb[i] = T(t)->nb[i]; });
}

static inline void chk(bool ok, const char *msg) { if (!ok) throw Error(std::string("[HALT] ") + msg); }
#define LB_OP1(name, fn) \
    lb_tensor *name(lb_mlctx *c, lb_tensor *a) { try { chk(c && a, "nil argument"); return W(fn(c->c, T(a))); } catch (const std::exception &e) { g_err = e.what(); return nullptr; } }
#define LB_OP2(name, fn) \
    lb_tensor *name(lb_mlctx *c, lb_tensor *a, lb_tensor *b) { try { chk(c && a && b, "nil argument"); return W(fn(c->c, T(a), T(b))); } catch (const std::exception &e) { g_err = e.what(); return nullptr; } }

LB_OP2(lb_get_rows, ml::GetRows)
LB_OP1(lb_rms_norm, ml::RMSNorm)
LB_OP2(lb_repeat, ml::Repeat)
LB_OP2(lb_mul, ml::Mul)
LB_OP2(lb_add, ml::Add)
LB_OP2(lb_mul_mat, ml::MulMat)
LB_OP2(lb_cpy, ml::Copy)
LB_OP1(lb_transpose, ml::Transpose)
LB_OP2(lb_scale, ml::Scale)
LB_OP1(lb_soft_max, ml::SoftMax)
LB_OP1(lb_silu, ml::Silu)

lb_tensor *lb_view_1d(lb_mlctx *c, lb_tensor *a, uint32_t ne0, uint32_t off) {
    try { chk(c && a, "nil argument"); return W(ml::View1D(c->c, T(a), ne0, off)); } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
lb_tensor *lb_rope(lb_mlctx *c, lb_tensor *a, uint32_t past, uint32_t dims, uint32_t mode) {
    try { chk(c && a, "nil argument"); return W(ml::Rope(c->c, T(a), past, dims, mode)); } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
lb_tensor *lb_permute(lb_mlctx *c, lb_tensor *a, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3) {
    try { chk(c && a, "nil argument"); return W(ml::Permute(c->c, T(a), a0, a1, a2, a3)); } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
lb_tensor *lb_reshape_3d(lb_mlctx *c, lb_tensor *a, uint32_t ne0, uint32_t ne1, uint32_t ne2) {
    try { chk(c && a, "nil argument"); return W(ml::Reshape3D(c->c, T(a), ne0, ne1, ne2)); } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
lb_tensor *lb_new_f32(lb_mlctx *c, float v) {
    try { chk(c, "nil argument"); return W(ml::NewFP32(c->c, v)); } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}
lb_tensor *lb_diag_mask_inf(lb_mlctx *c, lb_tensor *a, uint32_t past) {
    try { chk(c && a, "nil argument"); return W(ml::DiagMaskInf(c->c, T(a), past)); } catch (const std::exception &e) { g_err = e.what(); return nullptr; }
}

lb_graph *lb_graph_new(void) { return new lb_graph(); }
void lb_graph_free(lb_graph *g) { delete g; }
int lb_build_forward_expand(lb_graph *g, lb_tensor *t) { LB_TRY_INT(LB_CHECK(g && t, "nil argument"); ml::BuildForwardExpand(&g->g, T(t))); }
int lb_graph_compute(lb_mlctx *ctx, lb_graph *g) { LB_TRY_INT(LB_CHECK(ctx && g, "nil argument"); ml::GraphCompute(ctx->c, &g->g, true)); }
uint32_t lb_graph_nodes(const lb_graph *g) { return g ? (uint32_t)g->g.nodes.size() : 0; }

}  // extern "C"
