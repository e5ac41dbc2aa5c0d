// pipeline.cpp — multi-GPU layer sharding (SURVEY.md §8e): one process per GPU, stage g owns layers
// [g*L/G, (g+1)*L/G) and the KV slabs of those layers; the only exchange is a point-to-point NCCL
// send/recv of the residual stream [dim] FP32 between consecutive stages (llama.go:369 `inpL`).
// No collective is invented: there is no all-reduce/all-gather anywhere on this path.
//
// NCCL is bound at run time (dlopen "libnccl.so.2": the copy torch already loaded if the host
// process imported torch, else the system one) so that libllamab200.so itself loads on machines
// without NCCL or a GPU.
#include <dlfcn.h>
#include <string.h>

#include <mutex>

#include "llama.hpp"

namespace lb {
namespace pipe {

// minimal NCCL ABI (nccl.h: ncclUniqueId is 128 opaque bytes; ncclFloat32 = 7, ncclUint32 = 3... see below)
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclUint32 = 3, ncclFloat32 = 7 };

struct Nccl {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
};
static Nccl g_nccl;
static std::mutex g_mu;
static ncclComm_t g_comm = nullptr;
static int g_rank = 0, g_world = 1, g_device = 0;

static void load_nccl() {
    if (g_nccl.h) return;
    const char *names[] = {"libnccl.so.2", "libnccl.so", nullptr};
    for (int i = 0; names[i] && !g_nccl.h; i++) g_nccl.h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    LB_CHECK(g_nccl.h != nullptr, std::string("cannot load NCCL: ") + dlerror());
#define LB_SYM(field, sym)                                              \
    g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(g_nccl.h, sym)); \
    LB_CHECK(g_nccl.field != nullptr, std::string("NCCL symbol missing: ") + sym)
    LB_SYM(GetUniqueId, "ncclGetUniqueId");
    LB_SYM(CommInitRank, "ncclCommInitRank");
    LB_SYM(CommDestroy, "ncclCommDestroy");
    LB_SYM(Send, "ncclSend");
    LB_SYM(Recv, "ncclRecv");
    LB_SYM(GroupStart, "ncclGroupStart");
    LB_SYM(GroupEnd, "ncclGroupEnd");
    LB_SYM(GetErrorString, "ncclGetErrorString");
    LB_SYM(GetVersion, "ncclGetVersion");
#undef LB_SYM
}
#define LB_NCCL(expr)                                                                                   \
    do {                                                                                                \
        ncclResult_t _r = (expr);                                                                       \
        if (_r != 0) throw lb::Error(std::string(#expr) + ": " + g_nccl.GetErrorString(_r));            \
    } while (0)

void unique_id(void *out128) {
    std::lock_guard<std::mutex> lk(g_mu);
    load_nccl();
    ncclUniqueId id;
    LB_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(out128, &id, 128);
}

void comm_init(const void *id128, int rank, int world, int device) {
    std::lock_guard<std::mutex> lk(g_mu);
    LB_CHECK(world >= 1 && rank >= 0 && rank < world, "comm_init: bad rank/world");
    load_nccl();
    LB_CHECK(g_comm == nullptr, "comm_init: communicator already initialised");
    LB_CUDA(cudaSetDevice(device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    LB_NCCL(g_nccl.CommInitRank(&g_comm, world, id, rank));
    g_rank = rank; g_world = world; g_device = device;
}

void comm_destroy() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_comm) { g_nccl.CommDestroy(g_comm); g_comm = nullptr; }
}

int nccl_version() {
    std::lock_guard<std::mutex> lk(g_mu);
    load_nccl();
    int v = 0;
    g_nccl.GetVersion(&v);
    return v;
}

// ---- fused stage hand-off over NVLink peer memory ---------------------------------------------------------------------
// Instead of ncclRecv -> stage kernels -> ncclSend per (step, sequence) slot (two extra kernels and a rendezvous per slot:
// ~60 us of a ~625 us slot at 8 GPUs, VERDICT r01), the stage's persistent kernel itself stores the residual into the next
// stage's buffer (peer-mapped by CUDA IPC; one process per GPU) and raises a flag there; the next stage's kernel — already
// streaming its weights — waits for that flag (kernels_ring.cu).  Back-pressure is a second flag going upstream.
// export: per context 2 x 64 bytes (cudaIpcMemHandle of x, of the flags);  import: the handles of the downstream stage's
// contexts (null on the last stage) and of the upstream stage's contexts (null on the first stage).
void p2p_export(llama::Context **ctxs, uint32_t n_seq, void *out) {
    LB_CHECK(ctxs && out && n_seq >= 1, "p2p_export: nil argument");
    char *o = static_cast<char *>(out);
    for (uint32_t s = 0; s < n_seq; s++) {
        llama::Context *c = ctxs[s];
        LB_CUDA(cudaSetDevice(c->model->device));
        if (!c->p2p_flags) c->p2p_flags = c->mem.dmalloc<uint32_t>(4);
        cudaIpcMemHandle_t hx, hf;
        LB_CUDA(cudaIpcGetMemHandle(&hx, c->x));
        LB_CUDA(cudaIpcGetMemHandle(&hf, c->p2p_flags));
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
        memcpy(o + (size_t)s * 128, &hx, 64);
        memcpy(o + (size_t)s * 128 + 64, &hf, 64);
    }
}

void p2p_import(llama::Context **ctxs, uint32_t n_seq, const void *down, const void *up) {
    LB_CHECK(ctxs && n_seq >= 1, "p2p_import: nil argument");
    for (uint32_t s = 0; s < n_seq; s++) {
        llama::Context *c = ctxs[s];
        LB_CHECK(!c->model->f16(), "p2p_import: the fused hand-off does not carry F16 weights (FP32 only)");
        LB_CHECK(c->p2p_flags != nullptr, "p2p_import: call p2p_export first");
        LB_CHECK(c->use_mega && !c->use_ring_q8, "p2p_import: the fused hand-off needs the FP32 decode megakernel (unsupported shape, Q8 weights or LB_NO_MEGA)");
        LB_CHECK(!c->stage_graph, "p2p_import: the stage graph is already captured");
        LB_CUDA(cudaSetDevice(c->model->device));
        cudaIpcMemHandle_t h;
        void *ptr = nullptr;
        if (down) {
            memcpy(&h, static_cast<const char *>(down) + (size_t)s * 128, 64);
            LB_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
            c->p2p_x_out = static_cast<float *>(ptr);
            memcpy(&h, static_cast<const char *>(down) + (size_t)s * 128 + 64, 64);
            LB_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
            c->p2p_flag_out = static_cast<uint32_t *>(ptr);
        }
        if (up) {
            memcpy(&h, static_cast<const char *>(up) + (size_t)s * 128 + 64, 64);
            LB_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
            c->p2p_ack_out = static_cast<uint32_t *>(ptr);
        }
        c->p2p_ready = true;
        // Capture the stage graph NOW, while no peer can be decoding yet (the caller's enable_p2p is collective and ends with
        // a barrier).  ensure_stage_graph starts with an eager warm-up launch that runs outside the flag protocol and, on every
        // stage but the first, overwrites this context's x with its own layer outputs: left to the first lb_pipeline_decode, it
        // clobbered the step-0 residual an already-running upstream stage had deposited there (2-GPU run r02s: 9e-3 logits
        // error on the 1 + 2 layer split, where stage 0 is the faster one).  The warm-up runs at the LAST cache position: the
        // K/V row it writes is rewritten by the real step that reaches it before anything reads it.
        c->state_host[0] = c->ctx_size - 1; c->state_host[1] = 0;
        LB_CUDA(cudaMemcpyAsync(c->state_dev, c->state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        c->ensure_stage_graph(c->stream);
        LB_CUDA(cudaStreamSynchronize(c->stream));
    }
}

void p2p_disable(llama::Context **ctxs, uint32_t n_seq) {
    for (uint32_t s = 0; s < n_seq; s++) {
        llama::Context *c = ctxs[s];
        if (c->stage_graph && c->p2p_ready) {   // captured with the hand-off (p2p_import): drop it, the next decode captures the NCCL variant
            LB_CUDA(cudaSetDevice(c->model->device));
            LB_CUDA(cudaStreamSynchronize(c->stream));
            cudaGraphExecDestroy(c->stage_graph);
            c->stage_graph = nullptr;
        }
        c->p2p_ready = false;
    }
}

// Steady-state pipelined decode.  `ctxs[s]` = this stage's context of in-flight sequence s (its own
// KV slabs and activations).  For step k = 0..steps-1 and sequence s = 0..S-1, in that order on ONE
// stream:   [recv residual from stage-1]  ->  this stage's layers (CUDA-graph replay)  ->
//           [send residual to stage+1].
// Tokens are teacher-forced: stage 0 holds tokens[s][k] (the sampler that would feed tokens back is
// host code outside this path, pkg/server/server.go:200-214).  The chain is feed-forward, so the
// blocking send/recv pairs cannot form a cycle.  Returns the CUDA-event time of the whole run on
// this rank's stream.
float pipeline_decode(llama::Context **ctxs, uint32_t S, const uint32_t *tokens, uint32_t steps, uint32_t past) {
    LB_CHECK(S >= 1 && steps >= 1 && ctxs != nullptr, "pipeline_decode: bad arguments");
    llama::Context *c0 = ctxs[0];
    llama::Model *m = c0->model;
    const uint32_t d = m->hp.dim;
    const bool first = m->has_embedding(), last = m->has_head();
    const int world = (first && last) ? 1 : g_world;
    const bool p2p = c0->p2p_ready;   // fused hand-off over peer memory: no NCCL call on the decode path
    if (world > 1 && !p2p) LB_CHECK(g_comm != nullptr, "pipeline_decode: call lb_comm_init first");
    LB_CHECK((uint64_t)past + steps <= c0->ctx_size, "pipeline_decode: past + steps exceeds the context size");
    LB_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = c0->stream;
    for (uint32_t s = 0; s < S; s++) {
        llama::Context *c = ctxs[s];
        LB_CHECK(c->model == m, "pipeline_decode: contexts must share the stage model");
        LB_CHECK(c->p2p_ready == p2p, "pipeline_decode: every context of the stage must use the same hand-off");
        LB_CHECK(steps <= c->tokens_cap, "pipeline_decode: too many steps");
        if (first) {
            LB_CHECK(tokens != nullptr, "pipeline_decode: stage 0 needs tokens");
            for (uint32_t k = 0; k < steps; k++) {
                LB_CHECK(tokens[(size_t)s * steps + k] < m->hp.vocab, "pipeline_decode: token id out of range");
                c->tokens_host[k] = tokens[(size_t)s * steps + k];
            }
            LB_CUDA(cudaMemcpyAsync(c->tokens_dev, c->tokens_host, steps * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        }
        c->state_host[0] = past; c->state_host[1] = 0;
        LB_CUDA(cudaMemcpyAsync(c->state_dev, c->state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        c->ensure_stage_graph(st);
    }
    LB_CUDA(cudaStreamSynchronize(st));
    LB_CUDA(cudaEventRecord(c0->ev0, st));
    for (uint32_t k = 0; k < steps; k++) {
        for (uint32_t s = 0; s < S; s++) {
            llama::Context *c = ctxs[s];
            if (!first && !p2p) LB_NCCL(g_nccl.Recv(c->x, d, ncclFloat32, g_rank - 1, g_comm, st));
            LB_CUDA(cudaGraphLaunch(c->stage_graph, st));
            count_launch(c->use_mega ? 2 : m->layers.size() * 8 + 4);
            if (!last && !p2p) LB_NCCL(g_nccl.Send(c->x, d, ncclFloat32, g_rank + 1, g_comm, st));
        }
    }
    LB_CUDA(cudaEventRecord(c0->ev1, st));
    LB_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    LB_CUDA(cudaEventElapsedTime(&ms, c0->ev0, c0->ev1));
    return ms;
}

// One pipelined pass of `n` tokens per sequence (prompt prefill): per sequence this rank receives
// the residual [n][dim], runs its layers eagerly (GEMM path for n > 8), sends it on.
void pipeline_prefill(llama::Context **ctxs, uint32_t S, const uint32_t *tokens, uint32_t n, uint32_t past) {
    LB_CHECK(S >= 1 && n >= 1 && ctxs != nullptr, "pipeline_prefill: bad arguments");
    llama::Context *c0 = ctxs[0];
    llama::Model *m = c0->model;
    const uint32_t d = m->hp.dim;
    const bool first = m->has_embedding(), last = m->has_head();
    const int world = (first && last) ? 1 : g_world;
    if (world > 1) LB_CHECK(g_comm != nullptr, "pipeline_prefill: call lb_comm_init first");
    LB_CHECK((uint64_t)past + n <= c0->ctx_size && n <= c0->max_batch, "pipeline_prefill: past + n exceeds the context size");
    LB_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = c0->stream;
    for (uint32_t s = 0; s < S; s++) {
        llama::Context *c = ctxs[s];
        LB_CHECK(c->model == m, "pipeline_prefill: contexts must share the stage model");
        if (first) {
            LB_CHECK(tokens != nullptr, "pipeline_prefill: stage 0 needs tokens");
            for (uint32_t i = 0; i < n; i++) {
                LB_CHECK(tokens[(size_t)s * n + i] < m->hp.vocab, "pipeline_prefill: token id out of range");
                c->tokens_host[i] = tokens[(size_t)s * n + i];
            }
            LB_CUDA(cudaMemcpyAsync(c->tokens_dev, c->tokens_host, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        }
        c->state_host[0] = past; c->state_host[1] = 0;
        LB_CUDA(cudaMemcpyAsync(c->state_dev, c->state_host, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        if (!first) LB_NCCL(g_nccl.Recv(c->x, (size_t)n * d, ncclFloat32, g_rank - 1, g_comm, st));
        c->forward_on(st, n);
        if (!last) LB_NCCL(g_nccl.Send(c->x, (size_t)n * d, ncclFloat32, g_rank + 1, g_comm, st));
        LB_CUDA(cudaStreamSynchronize(st));  // pinned staging buffers are reused by the next sequence
    }
}

}  // namespace pipe
}  // namespace lb
