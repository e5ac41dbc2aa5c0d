// llama.cpp — see llama.hpp.
#include "llama.hpp"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <thread>

namespace lb {
namespace llama {

static const double IH_STD = 37837.22539803592;  // llama.go_b200/synth.py

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

bool Model::known_name(const HParams &hp, const std::string &name) {
    if (name == "tok_embeddings.weight" || name == "norm.weight" || name == "output.weight") return true;
    unsigned il;
    char rest[64];
    if (sscanf(name.c_str(), "layers.%u.%63s", &il, rest) == 2 && il < hp.layers) {
        static const char *kinds[] = {"attention_norm.weight", "attention.wq.weight", "attention.wk.weight",
                                      "attention.wv.weight", "attention.wo.weight", "ffn_norm.weight",
                                      "feed_forward.w1.weight", "feed_forward.w2.weight", "feed_forward.w3.weight"};
        for (const char *kname : kinds)
            if (!strcmp(rest, kname)) return true;
    }
    return false;
}

Model::Model(const HParams &h, int dev, uint32_t lb_, uint32_t le_, int wt) : hp(h), device(dev), layer_begin(lb_), layer_end(le_), weight_type(wt) {
    LB_CHECK(hp.vocab && hp.dim && hp.mult && hp.heads && hp.layers, "model: zero hyper-parameter");
    LB_CHECK(hp.dim % hp.heads == 0, "model: dim must be divisible by heads");
    LB_CHECK(hp.dim % 4 == 0, "model: dim must be a multiple of 4");
    LB_CHECK(layer_begin < layer_end && layer_end <= hp.layers, "model: bad layer range");
    LB_CHECK(wt == 0 || wt == 1 || wt == 16, "model: weight type must be LB_TYPE_F32, LB_TYPE_F16 or LB_TYPE_Q8_0");
    if (q8()) LB_CHECK(hp.dim % 32 == 0 && hp.ff() % 32 == 0 && hp.vocab % 4 == 0, "model: Q8_0 needs dim and ff to be multiples of 32 and vocab of 4");
    // F16: the tcgen05 prefill GEMM always applies (K % 32) and every row is a whole number of 64-byte bulk-copy units
    if (f16()) LB_CHECK(hp.dim % 32 == 0 && hp.ff() % 32 == 0, "model: F16 needs dim and ff to be multiples of 32");
    LB_CUDA(cudaSetDevice(device));
    const size_t d = hp.dim, ff = hp.ff(), V = hp.vocab;
    const size_t A = 64;  // floats: 256-byte alignment of every tensor
    size_t total = 0, qtotal = 0, dtotal = 0, htotal = 0;
    auto reserve = [&](size_t n) { size_t off = total; total += align_up(n, A); return off; };
    // a MulMat matrix: float slab (F32), q/d planes (Q8_0) or half slab (F16); returns {float off, q off, d off, half off}
    struct MOff { size_t f, q, d, h; };
    auto reserve_mat = [&](size_t n) {
        MOff o{0, 0, 0, 0};
        if (q8()) { o.q = qtotal; qtotal += align_up(n, 512); o.d = dtotal; dtotal += align_up(n / 32, A); }   // 512 = one 16 x 32 tile block (tile-major plane offsets)
        else if (f16()) { o.h = htotal; htotal += align_up(n, 2 * A); }   // 256-byte alignment
        else o.f = reserve(n);
        return o;
    };
    size_t o_emb = 0, o_norm = 0;
    MOff o_out{0, 0, 0, 0};
    if (has_embedding()) o_emb = reserve(V * d);
    if (has_head()) { o_norm = reserve(d); o_out = reserve_mat(V * d); }
    struct LOff { size_t an, fn; MOff qkv, wo, w1, w2, w3; };
    std::vector<LOff> lo(layer_end - layer_begin);
    for (auto &l : lo) {
        l.an = reserve(d); l.qkv = reserve_mat(3 * d * d); l.wo = reserve_mat(d * d); l.fn = reserve(d);
        l.w1 = reserve_mat(ff * d); l.w3 = reserve_mat(ff * d); l.w2 = reserve_mat(d * ff);
    }
    slab_floats = total;
    mem.device = device;
    slab = mem.dmalloc<float>(total);
    if (q8()) {
        qslab = mem.dmalloc<int8_t>(qtotal);
        dslab = mem.dmalloc<float>(dtotal);
        tmslab = mem.dmalloc<uint8_t>(qtotal / 512 * 576 + 256);   // every matrix: (rows / 16) x (K / 32) records of 576 bytes
    }
    if (f16()) {
        hslab = mem.dmalloc<uint16_t>(htotal);
        f16_overflow = mem.dmalloc<unsigned>(1);
    }
    auto fptr = [&](const MOff &o) { return f32() ? slab + o.f : nullptr; };
    auto hptr = [&](const MOff &o) { return f16() ? hslab + o.h : nullptr; };
    // (matrix offsets o.q are multiples of 512 elements; the decode plane holds 36 bytes per 32 elements, k::q8_tile_major_bytes)
    auto qmat = [&](const MOff &o, size_t rows_total, size_t cols, size_t row_off = 0) {
        Q8Mat m;
        if (q8()) {
            m.q = qslab + o.q + row_off * cols; m.d = dslab + o.d + row_off * cols / 32;
            m.tm = tmslab + o.q / 512 * 576;
            m.tm_row0 = (uint32_t)row_off; m.tm_rows = (uint32_t)rows_total;
        }
        return m;
    };
    const float sdd = (float)pow((double)d, -0.5), sf = (float)pow((double)ff, -0.5);
    if (has_embedding()) {
        tok_embeddings = slab + o_emb;
        tensors["tok_embeddings.weight"] = {tok_embeddings, V * d, 1, 0.f, 1.f, Q8Mat()};
    }
    if (has_head()) {
        norm = slab + o_norm; output = fptr(o_out); output8 = qmat(o_out, V, d); outputh = hptr(o_out);
        tensors["norm.weight"] = {norm, d, 2, 1.f, 0.1f, Q8Mat()};
        tensors["output.weight"] = {output, V * d, 3, 0.f, sdd, output8, (uint32_t)d, outputh};
    }
    layers.resize(lo.size());
    for (size_t i = 0; i < lo.size(); i++) {
        Layer &L = layers[i];
        L.attention_norm = slab + lo[i].an; L.ffn_norm = slab + lo[i].fn;
        L.wqkv = fptr(lo[i].qkv); L.wo = fptr(lo[i].wo); L.w1 = fptr(lo[i].w1); L.w3 = fptr(lo[i].w3); L.w2 = fptr(lo[i].w2);
        L.wqkv8 = qmat(lo[i].qkv, 3 * d, d); L.wo8 = qmat(lo[i].wo, d, d); L.w18 = qmat(lo[i].w1, ff, d); L.w38 = qmat(lo[i].w3, ff, d); L.w28 = qmat(lo[i].w2, d, ff);
        L.wqkvh = hptr(lo[i].qkv); L.woh = hptr(lo[i].wo); L.w1h = hptr(lo[i].w1); L.w3h = hptr(lo[i].w3); L.w2h = hptr(lo[i].w2);
        uint32_t il = layer_begin + (uint32_t)i;
        std::string p = "layers." + std::to_string(il) + ".";
        uint64_t base = 16ull * (il + 1);
        auto fq = [&](size_t rows_off) { return f32() ? L.wqkv + rows_off : nullptr; };
        auto hq = [&](size_t rows_off) { return f16() ? L.wqkvh + rows_off : nullptr; };
        tensors[p + "attention_norm.weight"] = {L.attention_norm, d, base + 0, 1.f, 0.1f, Q8Mat()};
        tensors[p + "attention.wq.weight"] = {fq(0), d * d, base + 1, 0.f, sdd, qmat(lo[i].qkv, 3 * d, d, 0), (uint32_t)d, hq(0)};
        tensors[p + "attention.wk.weight"] = {fq(d * d), d * d, base + 2, 0.f, sdd, qmat(lo[i].qkv, 3 * d, d, d), (uint32_t)d, hq(d * d)};
        tensors[p + "attention.wv.weight"] = {fq(2 * d * d), d * d, base + 3, 0.f, sdd, qmat(lo[i].qkv, 3 * d, d, 2 * d), (uint32_t)d, hq(2 * d * d)};
        tensors[p + "attention.wo.weight"] = {L.wo, d * d, base + 4, 0.f, sdd, L.wo8, (uint32_t)d, L.woh};
        tensors[p + "ffn_norm.weight"] = {L.ffn_norm, d, base + 5, 1.f, 0.1f, Q8Mat()};
        tensors[p + "feed_forward.w1.weight"] = {L.w1, ff * d, base + 6, 0.f, sdd, L.w18, (uint32_t)d, L.w1h};
        tensors[p + "feed_forward.w2.weight"] = {L.w2, d * ff, base + 7, 0.f, sf, L.w28, (uint32_t)ff, L.w2h};
        tensors[p + "feed_forward.w3.weight"] = {L.w3, ff * d, base + 8, 0.f, sdd, L.w38, (uint32_t)d, L.w3h};
    }
}

Model::~Model() {}  // `mem` releases the slabs

void Model::set_tensor(const std::string &name, int dtype, const void *host, size_t nbytes) {
    // LoadModel's tensor loop, llama.go:889-959: unknown names abort (:906-910); only F32 and F16
    // are accepted (:937-959), F16 is widened to FP32.  With Q8_0 weights the MulMat matrices are
    // block-quantised on the device as they arrive; with F16 weights they keep F16 input byte for
    // byte and round F32 input to nearest even.
    LB_CHECK(known_name(hp, name), "Unknown tensor '" + name + "' in model file");
    auto it = tensors.find(name);
    if (it == tensors.end()) return;  // belongs to another pipeline stage
    LB_CHECK(dtype == 0 || dtype == 1, "Tensor data type is not supported yet!");
    const Entry &e = it->second;
    const size_t esz = dtype == 0 ? 4 : 2;
    LB_CHECK(nbytes == e.nelem * esz, "tensor '" + name + "' has the wrong size");
    LB_CUDA(cudaSetDevice(device));
    if (e.h) {
        if (dtype == 1) {
            LB_CUDA(cudaMemcpy(e.h, host, nbytes, cudaMemcpyHostToDevice));
        } else {
            void *tmp = nullptr;
            LB_CUDA(cudaMalloc(&tmp, nbytes));
            try {
                LB_CUDA(cudaMemcpy(tmp, host, nbytes, cudaMemcpyHostToDevice));
                round_to_f16(static_cast<const float *>(tmp), e.h, e.nelem, name, 0);
            } catch (...) { cudaFree(tmp); throw; }
            cudaFree(tmp);
        }
        return;
    }
    const bool quant = e.q8.q != nullptr;
    float *dst = e.ptr;
    void *tmp16 = nullptr, *tmp32 = nullptr;
    if (quant) { LB_CUDA(cudaMalloc(&tmp32, e.nelem * sizeof(float))); dst = static_cast<float *>(tmp32); }
    if (dtype == 0) {
        LB_CUDA(cudaMemcpy(dst, host, nbytes, cudaMemcpyHostToDevice));
    } else {
        LB_CUDA(cudaMalloc(&tmp16, nbytes));
        LB_CUDA(cudaMemcpy(tmp16, host, nbytes, cudaMemcpyHostToDevice));
        k::f16_to_f32(static_cast<const uint16_t *>(tmp16), dst, e.nelem, 0);
    }
    if (quant) {
        k::quantize_q8(dst, e.q8.q, e.q8.d, (uint32_t)(e.nelem / e.cols), e.cols, 0);
        k::q8_to_tile_major(e.q8.q, e.q8.d, e.q8.tm, e.q8.tm_rows, e.q8.tm_row0, (uint32_t)(e.nelem / e.cols), e.cols, 0);
    }
    LB_CUDA(cudaDeviceSynchronize());
    if (tmp16) cudaFree(tmp16);
    if (tmp32) cudaFree(tmp32);
}

void Model::round_to_f16(const float *src, uint16_t *dst, size_t n, const std::string &name, cudaStream_t st) {
    unsigned over = 0;
    LB_CUDA(cudaMemsetAsync(f16_overflow, 0, sizeof(unsigned), st));
    k::f32_to_f16(src, dst, n, f16_overflow, st);
    LB_CUDA(cudaMemcpyAsync(&over, f16_overflow, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    LB_CUDA(cudaStreamSynchronize(st));
    LB_CHECK(over == 0, "tensor '" + name + "' holds a finite value outside the F16 range (|x| > 65504)");
}

void Model::get_tensor(const std::string &name, float *host, size_t nelem) {
    auto it = tensors.find(name);
    LB_CHECK(it != tensors.end(), "tensor '" + name + "' is not held by this stage");
    const Entry &e = it->second;
    LB_CHECK(nelem == e.nelem, "tensor '" + name + "' has the wrong size");
    LB_CUDA(cudaSetDevice(device));
    if (e.h) {
        void *tmp = nullptr;
        LB_CUDA(cudaMalloc(&tmp, nelem * sizeof(float)));
        k::f16_to_f32(e.h, static_cast<float *>(tmp), nelem, 0);
        const cudaError_t err = cudaMemcpy(host, tmp, nelem * sizeof(float), cudaMemcpyDeviceToHost);
        cudaFree(tmp);
        LB_CUDA(err);
    } else if (e.q8.q) {
        void *tmp = nullptr;
        LB_CUDA(cudaMalloc(&tmp, nelem * sizeof(float)));
        k::dequantize_q8(e.q8.q, e.q8.d, static_cast<float *>(tmp), (uint32_t)(nelem / e.cols), e.cols, 0);
        LB_CUDA(cudaMemcpy(host, tmp, nelem * sizeof(float), cudaMemcpyDeviceToHost));
        cudaFree(tmp);
    } else {
        LB_CUDA(cudaMemcpy(host, e.ptr, nelem * sizeof(float), cudaMemcpyDeviceToHost));
    }
}

void Model::init_random(uint64_t seed) {
    LB_CUDA(cudaSetDevice(device));
    void *tmp = nullptr;
    size_t tmp_elems = 0;
    for (auto &kv : tensors)
        if ((kv.second.q8.q || kv.second.h) && kv.second.nelem > tmp_elems) tmp_elems = kv.second.nelem;
    if (tmp_elems) LB_CUDA(cudaMalloc(&tmp, tmp_elems * sizeof(float)));
    for (auto &kv : tensors) {
        const Entry &e = kv.second;
        // float32(sigma / IH_STD): the division is done in double on the host exactly like numpy does
        float sscale = (float)((double)e.sigma / IH_STD);
        if (e.q8.q) {
            k::init_random(static_cast<float *>(tmp), e.nelem, seed, e.tid, e.mean, sscale, 0);
            k::quantize_q8(static_cast<float *>(tmp), e.q8.q, e.q8.d, (uint32_t)(e.nelem / e.cols), e.cols, 0);
            k::q8_to_tile_major(e.q8.q, e.q8.d, e.q8.tm, e.q8.tm_rows, e.q8.tm_row0, (uint32_t)(e.nelem / e.cols), e.cols, 0);
        } else if (e.h) {
            k::init_random(static_cast<float *>(tmp), e.nelem, seed, e.tid, e.mean, sscale, 0);
            round_to_f16(static_cast<const float *>(tmp), e.h, e.nelem, kv.first, 0);
        } else {
            k::init_random(e.ptr, e.nelem, seed, e.tid, e.mean, sscale, 0);
        }
    }
    LB_CUDA(cudaDeviceSynchronize());
    if (tmp) cudaFree(tmp);
}

uint64_t Model::weight_bytes_per_token() const {
    // SURVEY §8(d): every layer matrix + both norms, lm_head, final norm, one embedding row
    const uint64_t d = hp.dim, ff = hp.ff(), V = hp.vocab;
    // matrices cost 4 B/weight (F32), 2 B/weight (F16) or 36 B per 32 weights (Q8_0); vectors are always F32
    const uint64_t nl = layer_end - layer_begin;
    uint64_t mat = nl * (4 * d * d + 3 * d * ff) + (has_head() ? V * d : 0);
    uint64_t vec = nl * 2 * d + (has_head() ? d : 0) + (has_embedding() ? d : 0);
    return (q8() ? mat / 32 * 36 : f16() ? mat * 2 : mat * 4) + vec * 4;
}

// ---------------------------------------------------------------------------------------------
Context::Context(Model *m, uint32_t cs) : model(m), ctx_size(cs) {
    LB_CHECK(cs > 0, "context: ctx_size must be > 0");
    LB_CUDA(cudaSetDevice(m->device));
    mem.device = m->device;
    stream = mem.stream();
    const HParams &hp = m->hp;
    const size_t d = hp.dim, ff = hp.ff(), V = hp.vocab, nl = m->layers.size();
    max_batch = cs;
    auto dalloc = [&](size_t floats) { return mem.dmalloc<float>(floats); };
    kv_k = dalloc(nl * cs * d);
    kv_v = dalloc(nl * cs * d);
    x = dalloc((size_t)max_batch * d); y = dalloc((size_t)max_batch * d); cur = dalloc((size_t)max_batch * d);
    qkv = dalloc((size_t)max_batch * 3 * d); attn = dalloc((size_t)max_batch * d);
    act = dalloc((size_t)max_batch * ff); up = dalloc((size_t)max_batch * ff);
    logits = dalloc(V);
    attn_scratch = dalloc(k::attention_decode_scratch_floats(hp.heads, hp.head_dim()));
    tokens_cap = max_batch + 4096;
    tokens_dev = mem.dmalloc<uint32_t>(tokens_cap);
    state_dev = mem.dmalloc<uint32_t>(2);
    state_host = mem.hmalloc<uint32_t>(2);
    tokens_host = mem.hmalloc<uint32_t>(tokens_cap);
    logits_host = mem.hmalloc<float>(V);
    ev0 = mem.event();
    ev1 = mem.event();
    use_graph = getenv("LB_NO_GRAPH") == nullptr;  // profiling aid: plain launches instead of graph replay
    // persistent megakernel for N == 1 (FP32 weights, supported shapes); LB_NO_MEGA=1 keeps the per-op kernels
    // (Q8_0 models keep the per-op kernels: a Q8 variant of the megakernel's K-sliced phases was measured
    //  slower — 173 vs 240 tok/s on 7B, too few bytes in flight per warp with 1-byte weights)
    const bool mega_ok = k::decode_mega_supported(hp.dim, hp.ff(), hp.heads);
    const bool ring_ok = getenv("LB_NO_RING") == nullptr && k::decode_ring_supported(hp.dim, hp.ff(), hp.heads, hp.vocab, cs);
    // (F16 models: only the TMA-ring megakernel has an F16 weight stream; the register-fed one never runs them)
    use_mega = getenv("LB_NO_MEGA") == nullptr && ((m->f32() && (mega_ok || ring_ok)) || (m->f16() && ring_ok));
    // TMA-ring megakernel (kernels_ring.cu, version 3): 234 vs 221 tok/s on an un-capped box, 224 vs 216 under the power cap
    // (profiles/README.md r02o/r02p) — the default; LB_NO_RING=1 keeps the register-fed megakernel (kernels_mega.cu)
    use_ring = use_mega && ring_ok;
    // Q8_0 weights: TMA ring + int8 tensor cores (kernels_ring_q8.cu); LB_NO_RING_Q8=1 keeps the per-op kernels
    use_ring_q8 = m->q8() && getenv("LB_NO_MEGA") == nullptr && getenv("LB_NO_RING_Q8") == nullptr &&
                  k::decode_ring_q8_supported(hp.dim, hp.ff(), hp.heads, hp.vocab, cs);
    if (use_ring_q8) use_mega = true;
    if (use_mega) {
        std::vector<k::MegaLayerHost> ml(nl);
        for (size_t i = 0; i < nl; i++) {
            const Layer &L = m->layers[i];
            ml[i] = {L.attention_norm, L.wqkv, L.wo, L.ffn_norm, L.w1, L.w3, L.w2,
                     kv_k + i * (size_t)cs * d, kv_v + i * (size_t)cs * d,
                     L.wqkv8.q, L.wo8.q, L.w18.q, L.w38.q, L.w28.q, L.wqkv8.d, L.wo8.d, L.w18.d, L.w38.d, L.w28.d,
                     L.wqkvh, L.woh, L.w1h, L.w3h, L.w2h};
        }
        mega_layers_dev = mem.dmalloc<k::MegaLayerHost>(nl, false);
        LB_CUDA(cudaMemcpy(mega_layers_dev, ml.data(), nl * sizeof(k::MegaLayerHost), cudaMemcpyHostToDevice));
        mega_barrier = mem.dmalloc<unsigned>(4 + 4 * nl);  // grid barrier + per-phase ticket counters
        if (getenv("LB_MEGA_TRACE")) mega_trace = mem.dmalloc<unsigned long long>(nl * 13 + 13 * 148);   // + 5 arrival stamps, 4 producer stall times, 4 job counts per CTA (layer 5)
        if (use_ring_q8) {
            std::vector<k::RingQ8Layer> pl(nl);
            for (size_t i = 0; i < nl; i++) {
                const Layer &L = m->layers[i];
                pl[i] = {L.wqkv8.tm, L.wo8.tm, L.w18.tm, L.w38.tm, L.w28.tm};
            }
            q8_planes_dev = mem.dmalloc<k::RingQ8Layer>(nl, false);
            LB_CUDA(cudaMemcpy(q8_planes_dev, pl.data(), nl * sizeof(k::RingQ8Layer), cudaMemcpyHostToDevice));
        }
    }
}

Context::~Context() {
    cudaSetDevice(model->device);
    if (stream) cudaStreamSynchronize(stream);
    if (decode_graph) cudaGraphExecDestroy(decode_graph);
    if (stage_graph) cudaGraphExecDestroy(stage_graph);
    if (p2p_x_out) cudaIpcCloseMemHandle(p2p_x_out);
    if (p2p_flag_out) cudaIpcCloseMemHandle(p2p_flag_out);
    if (p2p_ack_out) cudaIpcCloseMemHandle(p2p_ack_out);
    // buffers, events and the stream are released by `mem`
}

// MulMat of a weight matrix: F32, Q8_0 planes or F16, GEMV (N <= 8) or GEMM
static void matmul(const float *W, const Q8Mat &W8, const uint16_t *Wh, uint32_t M, uint32_t K, const float *X, uint32_t ldx, uint32_t N,
                   float *Y, uint32_t ldy, const float *res, cudaStream_t st) {
    if (W8.q) {
        if (N <= 8) k::gemv_q8(W8.q, W8.d, M, K, X, ldx, N, Y, ldy, res, st);
        else k::gemm_q8_auto(W8.q, W8.d, M, K, X, ldx, N, Y, ldy, res, st);
    } else if (Wh) {
        if (N <= 8) k::gemv_f16(Wh, M, K, X, ldx, N, Y, ldy, res, st);
        else k::gemm_f16_tc(Wh, M, K, X, ldx, N, Y, ldy, res, st);
    } else {
        if (N <= 8) k::gemv_f32(W, M, K, X, ldx, N, Y, ldy, res, st);
        else k::gemm_auto(W, M, K, X, ldx, N, Y, ldy, res, st);
    }
}

// The fused forward pass.  Per layer (llama.go:246-370):
//   cur  = rmsnorm(x) * attention_norm                      (:255-259)      1 kernel
//   qkv  = [wq;wk;wv] · cur                                 (:263-265)      1 kernel
//   rope(q), rope(k) -> K cache, v -> V cache               (:274-297)      1 kernel
//   attn = softmax(mask(K·q / sqrt(hd))) · V                (:300-333)      1 kernel
//   y    = wo · attn + x                                    (:336-340)      1 kernel
//   cur  = rmsnorm(y) * ffn_norm                            (:346-351)      1 kernel
//   act  = silu(w1 · cur) * (w3 · cur)                      (:354-361)      1 kernel (decode)
//   x    = w2 · act + y                                     (:363-366)      1 kernel
void Context::forward(uint32_t n, bool tokens_indirect, bool all_rows, const float *hidden_in, float *hidden_out) {
    const HParams &hp = model->hp;
    const uint32_t d = hp.dim, ff = hp.ff(), V = hp.vocab, H = hp.heads;
    const uint32_t *past_dev = state_dev, *step_dev = state_dev + 1;
    cudaStream_t st = stream;
    if (use_mega && n == 1 && !all_rows) {
        // the whole token in one persistent cooperative kernel (kernels_mega.cu)
        if (!model->has_embedding()) {
            LB_CHECK(hidden_in != nullptr, "eval_stage: this stage needs hidden_in");
            if (hidden_in != x) LB_CUDA(cudaMemcpyAsync(x, hidden_in, (size_t)d * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        k::MegaParamsHost mp;
        mp.layers_dev = static_cast<const k::MegaLayerHost *>(mega_layers_dev);
        mp.n_layers = (uint32_t)model->layers.size();
        mp.tok_embeddings = model->has_embedding() ? model->tok_embeddings : nullptr;
        mp.tokens = tokens_dev; mp.state = state_dev;
        mp.final_norm = model->has_head() ? model->norm : nullptr;
        mp.output = model->has_head() ? model->output : nullptr;
        mp.q_output = model->has_head() ? model->output8.q : nullptr;
        mp.d_output = model->has_head() ? model->output8.d : nullptr;
        mp.q8 = model->q8();
        mp.f16 = model->f16();
        mp.h_output = model->has_head() ? model->outputh : nullptr;
        mp.x = x; mp.y = y; mp.qkv = qkv; mp.attn = attn; mp.act = act; mp.logits = logits;
        const uint32_t hd = hp.head_dim();
        mp.part_o = attn_scratch;
        mp.part_ml = attn_scratch + (size_t)H * 32 * hd;
        mp.tickets = reinterpret_cast<unsigned *>(mp.part_ml + (size_t)H * 32 * 2);
        mp.barrier = mega_barrier;
        mp.trace = mega_trace;
        if (p2p_on && !use_ring_q8) {
            mp.p2p_flags = p2p_flags;
            mp.p2p_wait_in = !model->has_embedding();
            mp.p2p_x_out = p2p_x_out; mp.p2p_flag_out = p2p_flag_out; mp.p2p_ack_out = p2p_ack_out;
        }
        mp.dim = d; mp.ff = ff; mp.heads = H; mp.vocab = V; mp.ctx = ctx_size;
        if (use_ring_q8) k::decode_ring_q8(mp, static_cast<const k::RingQ8Layer *>(q8_planes_dev), model->has_head() ? model->output8.tm : nullptr, st);
        else if (use_ring) k::decode_ring(mp, st);
        else k::decode_mega(mp, st);
        if (hidden_out && hidden_out != x)
            LB_CUDA(cudaMemcpyAsync(hidden_out, x, (size_t)d * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return;
    }
    if (model->has_embedding()) {
        if (tokens_indirect) k::get_rows_indirect(model->tok_embeddings, d, tokens_dev, step_dev, n, x, st);
        else k::get_rows_u32ids(model->tok_embeddings, d, tokens_dev, n, x, st);
    } else {
        LB_CHECK(hidden_in != nullptr, "eval_stage: this stage needs hidden_in");
        if (hidden_in != x) LB_CUDA(cudaMemcpyAsync(x, hidden_in, (size_t)n * d * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    for (size_t li = 0; li < model->layers.size(); li++) {
        const Layer &L = model->layers[li];
        float *Kc = kv_k + li * (size_t)ctx_size * d, *Vc = kv_v + li * (size_t)ctx_size * d;
        k::rms_norm(x, L.attention_norm, cur, d, n, st);
        matmul(L.wqkv, L.wqkv8, L.wqkvh, 3 * d, d, cur, d, n, qkv, 3 * d, nullptr, st);
        k::rope_qk_store(qkv, qkv + d, qkv + 2 * d, 3 * d, Kc, Vc, n, past_dev, d, H, st);
        if (n == 1) k::attention_decode(qkv, Kc, Vc, attn, past_dev, ctx_size, d, H, attn_scratch, st);
        else k::attention(qkv, 3 * d, Kc, Vc, attn, n, past_dev, ctx_size, d, H, st);
        matmul(L.wo, L.wo8, L.woh, d, d, attn, d, n, y, d, x, st);
        k::rms_norm(y, L.ffn_norm, cur, d, n, st);
        if (n <= 8) {
            if (model->q8()) k::gemv_q8_swiglu(L.w18.q, L.w18.d, L.w38.q, L.w38.d, ff, d, cur, d, n, act, ff, st);
            else if (model->f16()) k::gemv_f16_swiglu(L.w1h, L.w3h, ff, d, cur, d, n, act, ff, st);
            else k::gemv_f32_swiglu(L.w1, L.w3, ff, d, cur, d, n, act, ff, st);
        } else {
            matmul(L.w3, L.w38, L.w3h, ff, d, cur, d, n, up, ff, nullptr, st);
            matmul(L.w1, L.w18, L.w1h, ff, d, cur, d, n, act, ff, nullptr, st);
            k::swiglu(act, up, act, (size_t)n * ff, st);
        }
        matmul(L.w2, L.w28, L.w2h, d, ff, act, ff, n, x, d, y, st);
    }
    if (hidden_out && hidden_out != x)
        LB_CUDA(cudaMemcpyAsync(hidden_out, x, (size_t)n * d * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (model->has_head()) {
        if (all_rows) {
            if (!all_logits) all_logits = mem.dmalloc<float>((size_t)max_batch * V, false);
            k::rms_norm(x, model->norm, cur, d, n, st);
            matmul(model->output, model->output8, model->outputh, V, d, cur, d, n, all_logits, V, nullptr, st);
        } else {
            // only row n-1 is ever read (llama.go:394-401); the reference computes all n (:384)
            k::rms_norm(x + (size_t)(n - 1) * d, model->norm, cur, d, 1, st);
            matmul(model->output, model->output8, model->outputh, V, d, cur, d, 1, logits, V, nullptr, st);
        }
    }
}

void Context::build_decode_graph() {
    cudaGraph_t g = nullptr;
    LB_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    try {
        forward(1, /*tokens_indirect=*/true, false, nullptr, nullptr);
        k::advance_state(state_dev, 1, 1, stream);
    } catch (...) {
        cudaStreamEndCapture(stream, &g);
        if (g) cudaGraphDestroy(g);
        throw;
    }
    LB_CUDA(cudaStreamEndCapture(stream, &g));
    LB_CUDA(cudaGraphInstantiate(&decode_graph, g, 0));
    cudaGraphDestroy(g);
}

void Context::forward_on(cudaStream_t st, uint32_t n) {
    cudaStream_t saved = stream;
    stream = st;
    try {
        forward(n, false, false, x, nullptr);
    } catch (...) {
        stream = saved;
        throw;
    }
    stream = saved;
    last_n = n;
}

void Context::ensure_stage_graph(cudaStream_t st) {
    if (stage_graph) return;
    LB_CUDA(cudaSetDevice(model->device));
    cudaStream_t saved = stream;
    stream = st;
    // eager warm-up run first (sets kernel attributes; leaves state untouched: no advance)
    try {
        forward(1, true, false, x, nullptr);
        LB_CUDA(cudaStreamSynchronize(st));
        cudaGraph_t g = nullptr;
        LB_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        try {
            p2p_on = p2p_ready;   // the captured kernel waits for / raises the peer flags; the eager warm-up above did not
            forward(1, true, false, x, nullptr);
            k::advance_state(state_dev, 1, 1, st, p2p_on ? p2p_flags + 2 : nullptr);
            p2p_on = false;
        } catch (...) {
            p2p_on = false;
            cudaStreamEndCapture(st, &g);
            if (g) cudaGraphDestroy(g);
            throw;
        }
        LB_CUDA(cudaStreamEndCapture(st, &g));
        LB_CUDA(cudaGraphInstantiate(&stage_graph, g, 0));
        cudaGraphDestroy(g);
    } catch (...) {
        stream = saved;
        throw;
    }
    stream = saved;
}

void Context::eval(const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out, bool all_rows,
                   const float *hidden_in, float *hidden_out) {
    const HParams &hp = model->hp;
    LB_CHECK(n >= 1, "Eval : no tokens");
    LB_CHECK(n <= max_batch, "Eval : batch larger than the context");
    LB_CHECK((uint64_t)past + n <= ctx_size, "Eval : pastCount + N exceeds the context size");
    LB_CUDA(cudaSetDevice(model->device));
    if (model->has_embedding()) {
        LB_CHECK(tokens != nullptr, "Eval : nil tokens");
        for (uint32_t i = 0; i < n; i++) {
            LB_CHECK(tokens[i] < hp.vocab, "Eval : token id out of range");
            tokens_host[i] = tokens[i];
        }
        LB_CUDA(cudaMemcpyAsync(tokens_dev, tokens_host, n * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    }
    state_host[0] = past; state_host[1] = 0;
    LB_CUDA(cudaMemcpyAsync(state_dev, state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    const bool single_stage = model->has_embedding() && model->has_head();
    if (n == 1 && !all_rows && single_stage && use_graph && !hidden_in && !hidden_out) {
        if (!decode_graph) {
            // first single-token eval runs eagerly (also sets kernel attributes), then capture
            forward(1, true, false, nullptr, nullptr);
            LB_CUDA(cudaStreamSynchronize(stream));
            build_decode_graph();
        } else {
            LB_CUDA(cudaGraphLaunch(decode_graph, stream));
            count_launch(use_mega ? 2 : model->layers.size() * 8 + 4);
        }
    } else {
        forward(n, false, all_rows, hidden_in, hidden_out);
    }
    last_n = n;
    if (logits_out && model->has_head()) {
        if (all_rows) {
            LB_CUDA(cudaMemcpyAsync(logits_out, all_logits, (size_t)n * hp.vocab * sizeof(float), cudaMemcpyDeviceToHost, stream));
        } else {
            LB_CUDA(cudaMemcpyAsync(logits_host, logits, hp.vocab * sizeof(float), cudaMemcpyDeviceToHost, stream));
        }
    }
    LB_CUDA(cudaStreamSynchronize(stream));  // Eval is synchronous (llama.go:389-401)
    if (logits_out && model->has_head() && !all_rows) memcpy(logits_out, logits_host, hp.vocab * sizeof(float));
}

float Context::decode_resident(const uint32_t *tokens, uint32_t steps, uint32_t past) {
    const HParams &hp = model->hp;
    LB_CHECK(model->has_embedding() && model->has_head(), "decode_resident : needs a single-stage model");
    LB_CHECK(steps >= 1 && steps <= tokens_cap, "decode_resident : too many steps");
    LB_CHECK((uint64_t)past + steps <= ctx_size, "decode_resident : past + steps exceeds the context size");
    LB_CUDA(cudaSetDevice(model->device));
    for (uint32_t i = 0; i < steps; i++) {
        LB_CHECK(tokens[i] < hp.vocab, "decode_resident : token id out of range");
        tokens_host[i] = tokens[i];
    }
    LB_CUDA(cudaMemcpyAsync(tokens_dev, tokens_host, steps * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    state_host[0] = past; state_host[1] = 0;
    LB_CUDA(cudaMemcpyAsync(state_dev, state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    uint32_t done = 0;
    if (!decode_graph) {
        forward(1, true, false, nullptr, nullptr);
        k::advance_state(state_dev, 1, 1, stream);
        LB_CUDA(cudaStreamSynchronize(stream));
        build_decode_graph();
        done = 1;
    }
    LB_CUDA(cudaStreamSynchronize(stream));
    LB_CUDA(cudaEventRecord(ev0, stream));
    for (uint32_t i = done; i < steps; i++) {
        LB_CUDA(cudaGraphLaunch(decode_graph, stream));
        count_launch(use_mega ? 2 : model->layers.size() * 8 + 4);
    }
    LB_CUDA(cudaEventRecord(ev1, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    LB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    last_n = 1;
    return ms;
}

void Context::generate_greedy(const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, float temp, float repeat_penalty,
                              uint32_t *out_tokens) {
    const HParams &hp = model->hp;
    LB_CHECK(model->has_embedding() && model->has_head(), "generate_greedy : needs a single-stage model");
    LB_CHECK(prompt && out_tokens && n_prompt >= 1 && predict >= 1, "generate_greedy : bad arguments");
    LB_CHECK((uint64_t)n_prompt + predict - 1 <= ctx_size, "generate_greedy : prompt + predict exceeds the context (context swapping is host policy, server.go:165-172)");
    LB_CHECK(predict <= tokens_cap, "generate_greedy : predict too large");
    LB_CHECK(temp > 0.f, "generate_greedy : temp must be > 0 (the reference replaces 0 by 0.5, main.go:379-381)");
    for (uint32_t i = 0; i < n_prompt; i++) LB_CHECK(prompt[i] < hp.vocab, "generate_greedy : token id out of range");
    LB_CUDA(cudaSetDevice(model->device));
    if (!ring_dev) {
        ring_dev = mem.dmalloc<uint32_t>(ctx_size);
        present_dev = mem.dmalloc<uint32_t>(hp.vocab);
        ring_pos_dev = mem.dmalloc<uint32_t>(1);
    }
    // ring of the last ctx_size ids: zeros, then the prompt (server.go:127-138, 190)
    std::vector<uint32_t> ring(ctx_size, 0u), present(hp.vocab, 0u);
    uint32_t pos = 0;
    for (uint32_t i = 0; i < n_prompt; i++) { ring[pos] = prompt[i]; pos = (pos + 1) % ctx_size; }
    for (uint32_t v : ring) present[v]++;
    LB_CUDA(cudaMemcpyAsync(ring_dev, ring.data(), ctx_size * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(present_dev, present.data(), hp.vocab * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaMemcpyAsync(ring_pos_dev, &pos, sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    eval(prompt, n_prompt, 0, nullptr, false);                         // prompt eval -> logits on the device
    if (!decode_graph) {                                               // make sure the decode graph exists
        const uint32_t t0 = prompt[n_prompt - 1];
        LB_CHECK((uint64_t)n_prompt < ctx_size || predict == 1, "generate_greedy : no room to warm up");
        if (predict > 1) {
            eval(&t0, 1, n_prompt, nullptr, false);                    // eager + capture (overwrites logits, KV slot n_prompt)
            eval(prompt, n_prompt, 0, nullptr, false);                 // restore prompt logits
        }
    }
    state_host[0] = n_prompt; state_host[1] = 0;
    LB_CUDA(cudaMemcpyAsync(state_dev, state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    const float scale = 1.0f / temp;                                   // float32(1.0 / temp), llama.go:500
    for (uint32_t i = 0; i < predict; i++) {
        k::sample_greedy(logits, hp.vocab, scale, repeat_penalty, present_dev, ring_dev, ctx_size, ring_pos_dev, tokens_dev, state_dev, stream);
        if (i + 1 < predict) {                                         // the last sampled token is never evaluated (server.go:153-237)
            LB_CUDA(cudaGraphLaunch(decode_graph, stream));
            count_launch(use_mega ? 2 : model->layers.size() * 8 + 4);
        } else {
            k::advance_state(state_dev, 0, 1, stream);
        }
    }
    LB_CUDA(cudaMemcpyAsync(tokens_host, tokens_dev, predict * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    memcpy(out_tokens, tokens_host, predict * sizeof(uint32_t));
}

int64_t context_swap(uint32_t ctx_size, uint32_t keep, const uint32_t *history, uint32_t n_history, uint32_t *past,
                     const uint32_t *embd, uint32_t n_embd, uint32_t *embd_out, uint32_t cap) {
    LB_CHECK(past && (embd || !n_embd) && embd_out, "context_swap : nil argument");
    uint32_t n_front = 0;
    if ((uint64_t)*past + n_embd > ctx_size) {              // server.go:165
        LB_CHECK(keep <= *past, "context_swap : keep exceeds pastCount");
        const uint32_t left = *past - keep;                  // :166
        *past = keep;                                        // :167
        n_front = left / 2;                                  // :171  ExtractTokens(lastNTokens.Move(-left/2), left/2)
        LB_CHECK(n_front <= n_history, "context_swap : history shorter than the tokens to re-evaluate");
    }
    LB_CHECK((uint64_t)n_front + n_embd <= cap, "context_swap : output capacity too small");
    for (uint32_t i = 0; i < n_front; i++) embd_out[i] = history[n_history - n_front + i];
    for (uint32_t i = 0; i < n_embd; i++) embd_out[n_front + i] = embd[i];
    return (int64_t)n_front + n_embd;
}

uint32_t Context::sample(const uint32_t *last_n, uint32_t n_last, uint32_t top_k, float top_p, float temp, float repeat_penalty,
                         uint64_t seed, uint32_t *ids_out, float *probs_out, uint32_t *n_out) {
    const HParams &hp = model->hp;
    LB_CHECK(model->has_head(), "SampleTopPTopK : this stage has no logits");
    LB_CHECK(last_n || !n_last, "SampleTopPTopK : nil lastNTokens");
    LB_CHECK(top_k >= 1 && top_k <= hp.vocab, "SampleTopPTopK : topK must be in 1..vocab");
    LB_CUDA(cudaSetDevice(model->device));
    if (!smp_ids_dev) {
        smp_ids_dev = mem.dmalloc<uint32_t>(hp.vocab);
        smp_probs_dev = mem.dmalloc<float>(hp.vocab);
        smp_nt_dev = mem.dmalloc<uint32_t>(2);
        smp_host = mem.hmalloc<uint32_t>(2);
    }
    if (n_last > smp_last_cap) {
        smp_last_cap = n_last > ctx_size ? n_last : ctx_size;
        smp_last_dev = mem.dmalloc<uint32_t>(smp_last_cap, false);
    }
    if (n_last) LB_CUDA(cudaMemcpyAsync(smp_last_dev, last_n, n_last * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    k::sample_top_p_top_k(logits, hp.vocab, smp_last_dev, n_last, top_k, top_p, temp, repeat_penalty, seed, smp_ids_dev, smp_probs_dev,
                          smp_nt_dev, stream);
    LB_CUDA(cudaMemcpyAsync(smp_host, smp_nt_dev, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    const uint32_t n = smp_host[0], tok = smp_host[1];
    if (ids_out) LB_CUDA(cudaMemcpy(ids_out, smp_ids_dev, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (probs_out) LB_CUDA(cudaMemcpy(probs_out, smp_probs_dev, n * sizeof(float), cudaMemcpyDeviceToHost));
    if (n_out) *n_out = n;
    return tok;
}

void Context::generate(const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, uint32_t top_k, float top_p, float temp,
                       float repeat_penalty, uint32_t keep_count, uint32_t batch_size, uint64_t seed, uint32_t *out_tokens) {
    const HParams &hp = model->hp;
    LB_CHECK(model->has_embedding() && model->has_head(), "generate : needs a single-stage model");
    LB_CHECK(prompt && out_tokens && n_prompt >= 1 && predict >= 1 && batch_size >= 1, "generate : bad arguments");
    for (uint32_t i = 0; i < n_prompt; i++) LB_CHECK(prompt[i] < hp.vocab, "generate : token id out of range");
    // ring of the last ctx_size ids, zero-filled (server.go:127-138); kept here oldest-first in a flat history
    std::vector<uint32_t> ring(ctx_size, 0u);
    uint32_t rpos = 0;
    auto append = [&](uint32_t t) { ring[rpos] = t; rpos = (rpos + 1) % ctx_size; };
    auto history = [&]() {   // chronological order, oldest first
        std::vector<uint32_t> h(ctx_size);
        for (uint32_t i = 0; i < ctx_size; i++) h[i] = ring[(rpos + i) % ctx_size];
        return h;
    };
    std::vector<uint32_t> embd, tmp((size_t)ctx_size * 2 + batch_size);
    uint32_t past = 0, consumed = 0, remained = predict, produced = 0;
    while (remained > 0) {   // server.go:153
        if (!embd.empty()) {
            if ((uint64_t)past + embd.size() > ctx_size) {   // :165-172
                const std::vector<uint32_t> h = history();
                const int64_t n = context_swap(ctx_size, keep_count, h.data(), ctx_size, &past, embd.data(), (uint32_t)embd.size(), tmp.data(),
                                               (uint32_t)tmp.size());
                embd.assign(tmp.begin(), tmp.begin() + n);
            }
            eval(embd.data(), (uint32_t)embd.size(), past, nullptr, false);   // :175
        }
        past += (uint32_t)embd.size();   // :183
        embd.clear();
        if (consumed < n_prompt) {        // :186-194
            while (consumed < n_prompt && embd.size() < batch_size) {
                embd.push_back(prompt[consumed]);
                append(prompt[consumed]);
                consumed++;
            }
        } else {                           // :196-214
            const uint32_t id = sample(ring.data(), ctx_size, top_k, top_p, temp, repeat_penalty, seed + produced, nullptr, nullptr, nullptr);
            append(id);
            embd.push_back(id);
            out_tokens[produced++] = id;
            remained--;
        }
    }
}

float Context::bench_kernel(int which, uint32_t iters, uint32_t past, uint64_t *bytes_per_launch) {
    const HParams &hp = model->hp;
    const uint32_t d = hp.dim, ff = hp.ff(), V = hp.vocab, H = hp.heads;
    const size_t nl = model->layers.size();
    LB_CHECK(iters >= 1 && nl >= 1, "bench_kernel : nothing to run");
    LB_CHECK(model->f32() || model->q8(), "bench_kernel : F32 and Q8_0 weights only");
    LB_CHECK(past < ctx_size, "bench_kernel : past exceeds the context");
    LB_CUDA(cudaSetDevice(model->device));
    state_host[0] = past; state_host[1] = 0;
    LB_CUDA(cudaMemcpyAsync(state_dev, state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    const uint32_t pf_n = max_batch < 512 ? max_batch : 512;  // tokens of the prefill GEMM probe
    auto launch = [&](uint32_t i) {
        const Layer &L = model->layers[i % nl];
        float *Kc = kv_k + (i % nl) * (size_t)ctx_size * d, *Vc = kv_v + (i % nl) * (size_t)ctx_size * d;
        switch (which) {
            case 0: matmul(L.wqkv, L.wqkv8, nullptr, 3 * d, d, cur, d, 1, qkv, 3 * d, nullptr, stream); break;
            case 1: matmul(L.wo, L.wo8, nullptr, d, d, attn, d, 1, y, d, x, stream); break;
            case 2: if (model->q8()) k::gemv_q8_swiglu(L.w18.q, L.w18.d, L.w38.q, L.w38.d, ff, d, cur, d, 1, act, ff, stream);
                    else k::gemv_f32_swiglu(L.w1, L.w3, ff, d, cur, d, 1, act, ff, stream);
                    break;
            case 3: matmul(L.w2, L.w28, nullptr, d, ff, act, ff, 1, up, d, y, stream); break;
            case 4: LB_CHECK(model->has_head(), "no lm_head on this stage");
                    matmul(model->output, model->output8, nullptr, V, d, cur, d, 1, logits, V, nullptr, stream); break;
            case 5: k::attention_decode(qkv, Kc, Vc, attn, state_dev, ctx_size, d, H, attn_scratch, stream); break;
            case 6: k::rms_norm(x, L.attention_norm, cur, d, 1, stream); break;
            case 7: matmul(L.w1, L.w18, nullptr, ff, d, cur, d, pf_n, act, ff, nullptr, stream); break;  // prefill GEMM
            default: LB_CHECK(false, "bench_kernel : unknown kernel id");
        }
    };
    const uint64_t T = (uint64_t)past + 1;
    auto wb = [&](uint64_t nw) { return model->q8() ? nw / 32 * 36 : nw * 4; };  // weight bytes
    switch (which) {  // algorithmic bytes: weights + activations in + out
        case 0: *bytes_per_launch = wb(3ull * d * d) + 4ull * (d + 3ull * d); break;
        case 1: *bytes_per_launch = wb((uint64_t)d * d) + 4ull * 3ull * d; break;
        case 2: *bytes_per_launch = wb(2ull * ff * d) + 4ull * (d + ff); break;
        case 3: *bytes_per_launch = wb((uint64_t)d * ff) + 4ull * (ff + 2ull * d); break;
        case 4: *bytes_per_launch = wb((uint64_t)V * d) + 4ull * (d + V); break;
        case 5: *bytes_per_launch = 4ull * (2ull * T * d + 2ull * d); break;
        case 7: *bytes_per_launch = 2ull * ff * d * pf_n; break;  // FLOPs (not bytes) of the GEMM
        default: *bytes_per_launch = 4ull * 3ull * d; break;
    }
    for (uint32_t i = 0; i < 3; i++) launch(i);  // warm-up
    LB_CUDA(cudaStreamSynchronize(stream));
    LB_CUDA(cudaEventRecord(ev0, stream));
    for (uint32_t i = 0; i < iters; i++) launch(i + 3);
    LB_CUDA(cudaEventRecord(ev1, stream));
    LB_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    LB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    return ms;
}

// Host-side twin of k::init_random (same integer recipe as llama.go_b200/synth.py).
static inline uint64_t splitmix64_host(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
void synth_fill_host(float *dst, uint64_t count, uint64_t seed, uint64_t tid, uint64_t start, float mean, double sigma) {
    const uint64_t base = seed * 0x9E3779B97F4A7C15ull + tid * 0xD1B54A32D192ED03ull;
    const float sscale = (float)(sigma / IH_STD);
    unsigned nt = std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    if (nt > 32) nt = 32;
    if (count < (1u << 16)) nt = 1;
    std::vector<std::thread> th;
    const uint64_t chunk = (count + nt - 1) / nt;
    for (unsigned t = 0; t < nt; t++) {
        uint64_t b = (uint64_t)t * chunk, e = b + chunk < count ? b + chunk : count;
        if (b >= e) break;
        th.emplace_back([=]() {
            for (uint64_t i = b; i < e; i++) {
                uint64_t h = splitmix64_host(base + start + i);
                int s = (int)(h & 0xFFFF) + (int)((h >> 16) & 0xFFFF) + (int)((h >> 32) & 0xFFFF) + (int)(h >> 48);
                volatile float tt = (float)(s - 131070) * sscale;  // one rounding, no FMA contraction
                dst[i] = mean + tt;
            }
        });
    }
    for (auto &x : th) x.join();
}

// ---------------------------------------------------------------------------------------------
// llama.Eval transcribed node for node onto the ml:: mirror (llama.go:211-426).  Every ml.* call
// below is the same call, with the same arguments, that the reference makes at the cited line.
void Context::eval_graph(const uint32_t *tokens, uint32_t N, uint32_t pastCount, float *logits_out) {
    using namespace ml;
    const HParams &hp = model->hp;
    LB_CHECK(model->has_embedding() && model->has_head(), "eval_graph : needs a single-stage model");
    LB_CHECK(model->f32(), "eval_graph : the pkg/ml op API is FP32 only (like the reference)");
    LB_CHECK(N >= 1 && (uint64_t)pastCount + N <= ctx_size, "Eval : pastCount + N exceeds the context size");
    LB_CUDA(cudaSetDevice(model->device));
    const uint32_t embdSize = hp.dim, layersCount = hp.layers, ctxSize = ctx_size, headsCount = hp.heads;
    const uint32_t vocabSize = hp.vocab, rotCount = hp.dim / hp.heads, ff = hp.ff();

    ml::Context mctx(model->device, stream);
    ml::Context *ctx0 = &mctx;
    Graph graph;
    auto weight = [&](float *p, uint32_t ne0, uint32_t ne1) {  // leaves created with ctx == nil in Go
        return NewTensor(ctx0, TYPE_F32, ne1 > 1 ? 2 : 1, ne0, ne1, 1, 1, p, (size_t)ne0 * ne1);
    };
    const size_t kvSize = (size_t)embdSize * layersCount * ctxSize;
    Tensor *kvK = NewTensor(ctx0, TYPE_F32, 1, (uint32_t)kvSize, 1, 1, 1, kv_k, kvSize);
    Tensor *kvV = NewTensor(ctx0, TYPE_F32, 1, (uint32_t)kvSize, 1, 1, 1, kv_v, kvSize);

    Tensor *embd = NewTensor1D(ctx0, TYPE_F32, N);  // :239-242 — ids as float32
    std::vector<float> idsf(N);
    for (uint32_t i = 0; i < N; i++) {
        LB_CHECK(tokens[i] < vocabSize, "Eval : token id out of range");
        idsf[i] = (float)tokens[i];
    }
    LB_CUDA(cudaMemcpyAsync(embd->data, idsf.data(), N * sizeof(float), cudaMemcpyHostToDevice, stream));
    LB_CUDA(cudaStreamSynchronize(stream));

    Tensor *inpL = GetRows(ctx0, weight(model->tok_embeddings, embdSize, vocabSize), embd);  // :244
    for (uint32_t il = 0; il < layersCount; il++) {
        const Layer &L = model->layers[il];
        Tensor *wq = weight(L.wqkv, embdSize, embdSize);
        Tensor *wk = weight(L.wqkv + (size_t)embdSize * embdSize, embdSize, embdSize);
        Tensor *wv = weight(L.wqkv + 2 * (size_t)embdSize * embdSize, embdSize, embdSize);
        Tensor *inpSA = inpL;
        Tensor *cur = RMSNorm(ctx0, inpL);                                              // :255
        Tensor *rep = Repeat(ctx0, weight(L.attention_norm, embdSize, 1), cur);         // :258
        cur = Mul(ctx0, rep, cur);                                                      // :259
        Tensor *Qcur = MulMat(ctx0, wq, cur);                                           // :263
        Tensor *Kcur = MulMat(ctx0, wk, cur);                                           // :264
        Tensor *Vcur = MulMat(ctx0, wv, cur);                                           // :265
        Tensor *kview = View1D(ctx0, kvK, N * embdSize, embdSize * (il * ctxSize + pastCount));  // :274
        Tensor *vview = View1D(ctx0, kvV, N * embdSize, embdSize * (il * ctxSize + pastCount));  // :275
        BuildForwardExpand(&graph, Copy(ctx0, Kcur, kview));                            // :277
        BuildForwardExpand(&graph, Copy(ctx0, Vcur, vview));                            // :278
        Tensor *Q = Permute(ctx0,
                            Rope(ctx0, Copy(ctx0, Qcur, NewTensor3D(ctx0, TYPE_F32, embdSize / headsCount, headsCount, N)),
                                 pastCount, rotCount, 0),
                            0, 2, 1, 3);                                                // :281-288
        Tensor *K = Permute(ctx0,
                            Rope(ctx0,
                                 Reshape3D(ctx0, View1D(ctx0, kvK, (pastCount + N) * embdSize, il * ctxSize * embdSize),
                                           embdSize / headsCount, headsCount, pastCount + N),
                                 pastCount, rotCount, 1),
                            0, 2, 1, 3);                                                // :290-297
        Tensor *KQ = MulMat(ctx0, K, Q);                                                // :300
        Tensor *KQScaled = Scale(ctx0, KQ, NewFP32(ctx0, (float)(1.0 / sqrt((double)embdSize / (double)headsCount))));  // :303-307
        Tensor *KQMasked = DiagMaskInf(ctx0, KQScaled, pastCount);                      // :310
        Tensor *KQSoftMax = SoftMax(ctx0, KQMasked);                                    // :313
        Tensor *VTrans = Copy(ctx0,
                              Permute(ctx0,
                                      Reshape3D(ctx0, View1D(ctx0, kvV, (pastCount + N) * embdSize, il * ctxSize * embdSize),
                                                embdSize / headsCount, headsCount, pastCount + N),
                                      1, 2, 0, 3),
                              NewTensor3D(ctx0, TYPE_F32, pastCount + N, embdSize / headsCount, headsCount));  // :315-322
        Tensor *KQV = MulMat(ctx0, VTrans, KQSoftMax);                                  // :325
        Tensor *KQVMerged = Permute(ctx0, KQV, 0, 2, 1, 3);                             // :328
        cur = Copy(ctx0, KQVMerged, NewTensor2D(ctx0, TYPE_F32, embdSize, N));          // :331-333
        cur = MulMat(ctx0, weight(L.wo, embdSize, embdSize), cur);                      // :336
        Tensor *inpFF = Add(ctx0, cur, inpSA);                                          // :340
        cur = RMSNorm(ctx0, inpFF);                                                     // :346
        cur = Mul(ctx0, Repeat(ctx0, weight(L.ffn_norm, embdSize, 1), cur), cur);       // :349-351
        Tensor *tmp = MulMat(ctx0, weight(L.w3, embdSize, ff), cur);                    // :354
        cur = MulMat(ctx0, weight(L.w1, embdSize, ff), cur);                            // :356
        cur = Silu(ctx0, cur);                                                          // :359
        cur = Mul(ctx0, cur, tmp);                                                      // :361
        cur = MulMat(ctx0, weight(L.w2, ff, embdSize), cur);                            // :363
        cur = Add(ctx0, cur, inpFF);                                                    // :366
        inpL = cur;                                                                     // :369
    }
    inpL = RMSNorm(ctx0, inpL);                                                         // :374
    inpL = Mul(ctx0, Repeat(ctx0, weight(model->norm, embdSize, 1), inpL), inpL);       // :377-379
    inpL = MulMat(ctx0, weight(model->output, embdSize, vocabSize), inpL);              // :384
    BuildForwardExpand(&graph, inpL);                                                   // :387
    GraphCompute(ctx0, &graph);                                                         // :389
    // :394-401 — row N-1 of the logits
    if (logits_out)
        LB_CUDA(cudaMemcpy(logits_out, inpL->data + (size_t)vocabSize * (N - 1), vocabSize * sizeof(float), cudaMemcpyDeviceToHost));
    last_n = N;
}

}  // namespace llama
}  // namespace lb
