/*
 * llamab200.h — C-ABI of the B200-native LLaMA forward-pass engine.
 *
 * Drop-in boundary for the hot path of gotzmann/llama.go: the exported Go API of
 * pkg/ml (Tensor, op constructors, Graph, GraphCompute) and pkg/llama (NewContext, Eval).
 * The reference has no FFI of its own (CGO_ENABLED=0, Makefile:25; the only foreign call is
 * the Go-asm stub vdot, pkg/ml/floats_avx.go:28), so these are the entry points a cgo shim
 * placed under pkg/ml and pkg/llama binds (INTEGRATION.md shows that shim).  Plain pointers
 * and sizes only; no torch, no C++ types.
 *
 * Conventions
 *   - Every function that can fail returns int: 0 = OK, non-zero = error; the message is in
 *     lb_last_error() (thread-local).  Constructors return NULL on error.  The reference's
 *     behaviour on the same conditions is print "[HALT] ..." + os.Exit(1) (e.g. ml.go:254-257,
 *     2116-2124); the Go shim maps a non-zero status back to that.
 *   - Host pointers are only read/written during the call and never retained (cgo rule).
 *   - lb_model is immutable after load and may be shared; each lb_context owns its KV cache
 *     and CUDA stream and is single-threaded, many may run concurrently ("pods",
 *     pkg/server/server.go:84-106).
 *   - There is NO CPU fallback: every entry point fails if no sm_100 device is usable.
 */
#ifndef LLAMAB200_H
#define LLAMAB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LB_API __attribute__((visibility("default")))

/* dtype codes = ml.DType (pkg/ml/ml.go:85-94) */
enum { LB_TYPE_F32 = 0, LB_TYPE_F16 = 1, LB_TYPE_Q4_0 = 2, LB_TYPE_Q4_1 = 3, LB_TYPE_I8 = 4,
       LB_TYPE_I16 = 5, LB_TYPE_I32 = 6,
       LB_TYPE_Q8_0 = 16 /* this repo's block format: 32 int8 + fp32 scale, see DESIGN.md */ };

typedef struct lb_model   lb_model;    /* = llama.Model   (pkg/llama/llama.go:181-193) */
typedef struct lb_context lb_context;  /* = llama.Context (pkg/llama/llama.go:83-88)   */
typedef struct lb_mlctx   lb_mlctx;    /* = ml.Context    (pkg/ml/ml.go:50-57)         */
typedef struct lb_tensor  lb_tensor;   /* = ml.Tensor     (pkg/ml/ml.go:180-203)       */
typedef struct lb_graph   lb_graph;    /* = ml.Graph      (pkg/ml/ml.go:31-45)         */
typedef struct lb_batch   lb_batch;    /* a set of up to 8 lb_contexts ("pods") decoded together */

/* HParams (pkg/llama/llama.go:149-158); ff is derived as in llama.go:761 */
typedef struct {
    uint32_t vocab, dim, mult, heads, layers;
} lb_hparams;

/* ---- library -------------------------------------------------------------------------- */
LB_API const char *lb_last_error(void);
LB_API int         lb_device_count(void);          /* usable sm_100 devices; <=0 => nothing works */
LB_API const char *lb_version(void);
LB_API uint64_t    lb_kernel_launches(void);       /* kernels launched by this library so far (process-wide) */

/* ---- model = llama.Model + LoadModel's tensor map (llama.go:712-976) ------------------ */
/* Layers [layer_begin, layer_end) live on `device`; the stage with layer_begin == 0 also owns
 * tok_embeddings, the stage with layer_end == layers also owns norm + output (SURVEY §8e).
 * weight_type: LB_TYPE_F32; LB_TYPE_F16 to hold every 2-D MulMat matrix (wq|wk|wv, wo, w1, w2, w3, output) as
 * IEEE binary16 — half the bytes, the same arithmetic on the widened values (needs dim and ff multiples of 32);
 * or LB_TYPE_Q8_0 to hold them block-quantised.  Norm vectors and tok_embeddings always stay FP32. */
LB_API lb_model *lb_model_create(const lb_hparams *hp, int device, uint32_t layer_begin,
                                 uint32_t layer_end, int weight_type);
LB_API void      lb_model_free(lb_model *m);
/* LoadModel (llama.go:712-976): a ggjt v1 file (F32 or F16 tensors) streamed straight into HBM through
 * pinned staging buffers; same magic/version/name/dtype checks as the reference.  layer_end = 0 means
 * "all layers"; hp_out (optional) receives the file's hyper-parameters. */
LB_API lb_model *lb_model_load_ggjt(const char *path, int device, uint32_t layer_begin, uint32_t layer_end,
                                    int weight_type, lb_hparams *hp_out);
/* name = ggjt tensor name (llama.go:826-861); dtype LB_TYPE_F32 or LB_TYPE_F16 (widened to FP32
 * like llama.go:938-941); tensors of layers this stage does not own are accepted and ignored.
 * Into an LB_TYPE_F16 model's matrices F16 data is stored byte for byte and F32 data is rounded to nearest
 * even (as numpy's astype(float16)); a finite value beyond +-65504 is an error.  The same holds for
 * lb_model_load_ggjt and lb_model_init_random. */
LB_API int       lb_model_set_tensor(lb_model *m, const char *name, int dtype, const void *host, size_t nbytes);
LB_API int       lb_model_get_tensor(lb_model *m, const char *name, float *host, size_t nelem); /* dequantised / widened to FP32 */
/* Synthetic weights generated on the device; bit-identical to llama.go_b200/synth.py. */
LB_API int       lb_model_init_random(lb_model *m, uint64_t seed);
LB_API uint64_t  lb_model_weight_bytes(const lb_model *m);   /* bytes one decoded token streams */
/* Host-side generator of the same synthetic weights (elements [start, start+count) of tensor
 * `tensor_id`), multi-threaded; used to write ggjt files for the reference binary quickly.
 * Pure host code: works without a GPU. */
LB_API int       lb_synth_fill_host(float *dst, uint64_t count, uint64_t seed, uint64_t tensor_id,
                                    uint64_t start, float mean, double sigma);
/* Micro-benchmark of one hot-path kernel for the roofline report: launches kernel `which`
 * (0 qkv gemv, 1 wo gemv+residual, 2 w1/w3 swiglu gemv, 3 w2 gemv+residual, 4 lm_head gemv,
 * 5 attention at `past`, 6 rmsnorm, 7 prefill GEMM w1 x min(512, ctx) tokens — bytes_out then holds its
 * FLOPs) `iters` times back to back on the context's stream, cycling
 * through the layers so the weights never sit in L2; ms_out = CUDA-event time of all launches,
 * bytes_out = algorithmic bytes of ONE launch.  F32 and Q8_0 models only (an F16 model is refused). */
LB_API int       lb_bench_kernel(lb_context *c, int which, uint32_t iters, uint32_t past, float *ms_out,
                                 uint64_t *bytes_out);

/* ---- context = llama.NewContext / ReleaseContext / Eval (llama.go:91-113, 211-426) ---- */
LB_API lb_context *lb_context_create(lb_model *m, uint32_t ctx_size);
LB_API void        lb_context_free(lb_context *c);
/* llama.Eval: evaluate `n` new tokens at position `past`; logits_out receives row n-1 ([vocab]).
 * Host buffers; H2D of the ids and D2H of the logits happen inside the call. */
LB_API int lb_eval(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out);
/* Same, but every row of logits ([n][vocab]) as the reference computes them (llama.go:384). */
LB_API int lb_eval_all_logits(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out);
/* The same forward pass built node for node with the op API below, exactly as llama.go:211-426
 * builds it, and run by lb_graph_compute (slow path; exists to prove the op API is a drop-in).
 * The op API is FP32 like the reference's: Q8_0 and F16 models are refused. */
LB_API int lb_eval_graph(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past, float *logits_out);
/* Device-resident decode: enqueue `steps` single-token evals starting at `past` with the given
 * tokens (teacher forcing), no host copies; used by bench.py for the kernel-only number.
 * ms_out (optional) = CUDA-event time of the whole batch of steps on the context's stream. */
LB_API int lb_decode_resident(lb_context *c, const uint32_t *tokens, uint32_t steps, uint32_t past, float *ms_out);
/* The generate loop of pkg/server.Do at temp -> 0 (server.go:153-237) with the sampler on the device
 * (SURVEY §8f-2): prompt eval, then `predict` x [repetition-penalised argmax (llama.go:500-527) ->
 * single-token eval], no host round trip per token.  out_tokens receives the `predict` generated ids. */
LB_API int lb_generate_greedy(lb_context *c, const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, float temp,
                              float repeat_penalty, uint32_t *out_tokens);
/* llama.SampleTopPTopK (pkg/llama/llama.go:455-707) on the device, on the logits of the context's last eval:
 * repetition penalty for the ids in last_n_tokens (membership only, :501-527), descending sort + top-k cut (:548-565),
 * softmax in f64 -> f32 (:579-599), top-p cut + renormalisation (:614-629), pick argmax p*p*f*f (:658-673).  The
 * reference seeds its generator with time.Now() (:655): `seed` replaces it (f_i from splitmix64(seed + i)).
 * cand_ids_out / cand_probs_out (optional, capacity top_k) receive the candidate set after both cuts. */
LB_API int lb_sample_top_p_top_k(lb_context *c, const uint32_t *last_n_tokens, uint32_t n_last, uint32_t top_k, float top_p,
                                 float temp, float repeat_penalty, uint64_t seed, uint32_t *cand_ids_out, float *cand_probs_out,
                                 uint32_t *n_cand_out, uint32_t *token_out);
/* The generate loop of pkg/server.Do (pkg/server/server.go:127-237): prompt consumed in batches of batch_size, the
 * context-swap rule when the context is full (:158-172, keep_count = Params.KeepCount), one device sample per token
 * (seed + token index).  out_tokens receives the `predict` sampled ids. */
LB_API int lb_generate(lb_context *c, const uint32_t *prompt, uint32_t n_prompt, uint32_t predict, uint32_t top_k, float top_p,
                       float temp, float repeat_penalty, uint32_t keep_count, uint32_t batch_size, uint64_t seed,
                       uint32_t *out_tokens);
/* The context-swap rule alone (server.go:165-172; main.go:190-200), pure host code: if *past_io + n_embd > ctx_size then
 * *past_io = keep_count and the last (past - keep_count) / 2 ids of `history` (oldest first) are put in front of embd.
 * Returns the new length written to embd_out (capacity cap), or -1 on error. */
LB_API int64_t lb_context_swap(uint32_t ctx_size, uint32_t keep_count, const uint32_t *history, uint32_t n_history,
                               uint32_t *past_io, const uint32_t *embd, uint32_t n_embd, uint32_t *embd_out, uint32_t cap);
LB_API int lb_context_read_logits(lb_context *c, float *logits_out);              /* last eval's row */
LB_API int lb_context_read_kv(lb_context *c, uint32_t layer, uint32_t t0, uint32_t nt, float *k_out, float *v_out);
LB_API int lb_context_read_hidden(lb_context *c, uint32_t n, float *hidden_out);  /* residual stream before final norm */
LB_API int lb_context_synchronize(lb_context *c);
/* profiling aid: 13 globaltimer (ns) stamps per layer of the last single-token megakernel launch
 * (CTA 0), valid when the context was created with LB_MEGA_TRACE=1 in the environment */
LB_API int lb_context_mega_trace(lb_context *c, uint64_t *out, uint32_t n);
/* pipeline stages (multi-GPU layer sharding, SURVEY §8e): run only this stage's layers.
 * hidden_in/out are DEVICE pointers to [n][dim] FP32 (NULL on the first/last stage). */
LB_API int lb_eval_stage(lb_context *c, const uint32_t *tokens, uint32_t n, uint32_t past,
                         const float *hidden_in_dev, float *hidden_out_dev, float *logits_out);
LB_API float *lb_context_hidden_buffer(lb_context *c);   /* device [max_batch][dim] scratch for hand-offs */
LB_API void  *lb_context_stream(lb_context *c);          /* cudaStream_t */
/* which kernels a single-token Eval of this context runs: "ring" (TMA-ring megakernel), "ring_f16" (the same with F16 weights),
   "mega" (register-fed megakernel), "ring_q8" (Q8_0 ring megakernel) or "perop" (one kernel per op) — measurement aid,
   no reference counterpart */
LB_API const char *lb_context_decode_path(lb_context *c);
/* work split / data layout of the ring megakernels, evaluated on the HOST by the same functions the kernels use (test aid, no
   GPU needed, no reference counterpart).  kind 0: FP32 ring, K = a -> out {chunks per row, floats per chunk};
   kind 1: Q8 ring, matrix [a x b], rows of work slot c -> out {r0, r1};  kind 2: Q8 decode plane, matrix [a x b], tile of row c ->
   out {first row, height, byte offset of the tile's first record (low, high)};  kind 3: pods ring, a rows, work slot c ->
   out {r0, r1, chunk index or 0xFFFFFFFF}.  Returns 0, or -1 for shapes the kernel does not take. */
LB_API int lb_layout_query(uint32_t kind, uint32_t a, uint32_t b, uint32_t c, uint32_t out[4]);

/* ---- tokenizer (SURVEY §8f-4): ml.Tokenize (pkg/ml/ml.go:2761-2848) on the host; works without a GPU ---- */
typedef struct lb_vocab lb_vocab;                                  /* = ml.Vocab (ml.go:2653-2657) */
LB_API lb_vocab *lb_vocab_create(uint32_t size);
LB_API void      lb_vocab_free(lb_vocab *v);
LB_API int       lb_vocab_set(lb_vocab *v, uint32_t id, const char *bytes, uint32_t len, float score);
/* returns the number of ids (may exceed cap; only min(count, cap) are written), or -1 on bad arguments */
LB_API int64_t   lb_tokenize(const lb_vocab *v, const char *text, uint32_t len, int bos, uint32_t *out, uint32_t cap);

/* ---- pod batching (SURVEY §8f-1): the reference runs --pods concurrent jobs, one llama.Context each, on one
 * shared Model (pkg/server/server.go:84-106,151-175).  Their single-token Evals are evaluated here as ONE
 * pass over the weights (B-column MulMat); every pod keeps its own KV cache and position. ---- */
LB_API lb_batch *lb_batch_create(lb_context **ctxs, uint32_t n);          /* 1..8 contexts of one model, same ctx size */
LB_API void      lb_batch_free(lb_batch *b);
/* one token per pod: tokens[n], pasts[n] (position of each pod's new token), logits_out [n][vocab]; synchronous */
LB_API int       lb_batch_eval(lb_batch *b, const uint32_t *tokens, const uint32_t *pasts, float *logits_out);
/* `steps` tokens per pod (tokens [n][steps], teacher-forced) enqueued back to back; ms_out = CUDA-event time */
LB_API int       lb_batch_decode_resident(lb_batch *b, const uint32_t *tokens, uint32_t steps, const uint32_t *pasts, float *ms_out);
LB_API int       lb_batch_read_logits(lb_batch *b, float *logits_out);    /* [n][vocab] of the last step */
/* profiling aid, like lb_context_mega_trace: 13 globaltimer stamps per layer of the last pod-batch step (LB_MEGA_TRACE=1) */
LB_API int       lb_batch_mega_trace(lb_batch *b, uint64_t *out, uint32_t n);

/* ---- multi-GPU layer sharding: one process per GPU, NCCL send/recv of the residual stream ----
 * rank r owns the stage created with lb_model_create(hp, dev, r*L/G, (r+1)*L/G).  NCCL is bound at
 * run time (dlopen), so the library itself loads without it. */
LB_API int  lb_comm_unique_id(void *out128);                 /* rank 0: ncclGetUniqueId (128 bytes) */
LB_API int  lb_comm_init(const void *id128, int rank, int world, int device);   /* ncclCommInitRank */
LB_API void lb_comm_destroy(void);
LB_API int  lb_nccl_version(void);
/* Fused stage hand-off over NVLink peer memory (one process per GPU): instead of ncclRecv / stage kernels / ncclSend per
 * (step, sequence) slot, the stage's persistent kernel stores the residual stream straight into the next stage's buffer
 * (CUDA IPC mapping) and raises a flag there, which the next stage's kernel waits for while it already streams its weights.
 * export: handles_out receives n x 128 bytes for this stage's n contexts; every rank exchanges them (any transport);
 * import: the bytes of the downstream stage (NULL on the last stage) and of the upstream stage (NULL on the first), before
 * the first lb_pipeline_decode.  Without import, lb_pipeline_decode uses NCCL send/recv as before; prefill always does.
 * import also captures the stage's CUDA graph (its warm-up launch must not run once a peer is decoding).  Caller's contract:
 * a barrier over all stages after import and after every lb_pipeline_prefill, before any stage calls lb_pipeline_decode —
 * prefill is outside the hand-off's flag protocol (llama.go_b200/pipeline.py does both barriers). */
LB_API int lb_pipeline_p2p_export(lb_context **ctxs, uint32_t n, void *handles_out);
LB_API int lb_pipeline_p2p_import(lb_context **ctxs, uint32_t n, const void *downstream_handles, const void *upstream_handles);   /* FP32 stages only: F16 is refused */
LB_API int lb_pipeline_p2p_disable(lb_context **ctxs, uint32_t n);   /* back to NCCL (e.g. another rank's import failed) */
/* Pipelined steady-state decode of `n_seq` in-flight sequences ("pods", server.go:84-106) for `steps`
 * tokens each, starting at position `past`: per (step, sequence) this rank receives the residual
 * [dim] from rank-1, runs its layers, sends it to rank+1; all on one stream, no host sync.  tokens
 * ([n_seq][steps], teacher-forced) are read on stage 0 only.  ms_out = CUDA-event time on this rank. */
LB_API int  lb_pipeline_decode(lb_context **ctxs, uint32_t n_seq, const uint32_t *tokens, uint32_t steps,
                               uint32_t past, float *ms_out);

/* One pipelined pass of n tokens per sequence (prompt prefill) through this rank's layers. */
LB_API int  lb_pipeline_prefill(lb_context **ctxs, uint32_t n_seq, const uint32_t *tokens, uint32_t n, uint32_t past);

/* ---- op-level mirror of pkg/ml -------------------------------------------------------- */
LB_API lb_mlctx  *lb_ml_new_context(int device);                   /* ml.NewContext (ml.go:59-74) */
LB_API void       lb_ml_release_context(lb_mlctx *ctx);            /* ReleaseContext (ml.go:77-80) */
LB_API lb_tensor *lb_new_tensor(lb_mlctx *ctx, int dtype, uint32_t dims, uint32_t ne0, uint32_t ne1,
                                uint32_t ne2, uint32_t ne3, const float *host_or_null); /* NewTensor ml.go:760 */
LB_API int        lb_tensor_write(lb_tensor *t, const float *host, size_t nelem);  /* = fill t.Data */
LB_API int        lb_tensor_read(lb_tensor *t, float *host, size_t nelem);         /* = read t.Data (backing store) */
LB_API int        lb_tensor_shape(const lb_tensor *t, uint32_t ne[4], uint32_t nb[4]); /* NB in bytes, ml.go:188 */
/* lazy op constructors, same arguments as the Go ctors (file:line in pkg/ml/ml.go) */
LB_API lb_tensor *lb_get_rows(lb_mlctx *, lb_tensor *a, lb_tensor *b);                 /* :528 */
LB_API lb_tensor *lb_rms_norm(lb_mlctx *, lb_tensor *a);                               /* :559 */
LB_API lb_tensor *lb_repeat(lb_mlctx *, lb_tensor *a, lb_tensor *b);                   /* :487 */
LB_API lb_tensor *lb_mul(lb_mlctx *, lb_tensor *a, lb_tensor *b);                      /* :241 */
LB_API lb_tensor *lb_add(lb_mlctx *, lb_tensor *a, lb_tensor *b);                      /* :347 */
LB_API lb_tensor *lb_mul_mat(lb_mlctx *, lb_tensor *a, lb_tensor *b);                  /* :295 */
LB_API lb_tensor *lb_view_1d(lb_mlctx *, lb_tensor *a, uint32_t ne0, uint32_t offset_floats); /* :601 */
LB_API lb_tensor *lb_cpy(lb_mlctx *, lb_tensor *a, lb_tensor *b);                      /* :733 */
LB_API lb_tensor *lb_rope(lb_mlctx *, lb_tensor *a, uint32_t past, uint32_t dims, uint32_t mode); /* :848 */
LB_API lb_tensor *lb_permute(lb_mlctx *, lb_tensor *a, uint32_t ax0, uint32_t ax1, uint32_t ax2, uint32_t ax3); /* :786 */
LB_API lb_tensor *lb_transpose(lb_mlctx *, lb_tensor *a);                              /* :1087 */
LB_API lb_tensor *lb_reshape_3d(lb_mlctx *, lb_tensor *a, uint32_t ne0, uint32_t ne1, uint32_t ne2); /* :882 */
LB_API lb_tensor *lb_new_f32(lb_mlctx *, float value);                                 /* :915 */
LB_API lb_tensor *lb_scale(lb_mlctx *, lb_tensor *a, lb_tensor *b);                    /* :959 */
LB_API lb_tensor *lb_diag_mask_inf(lb_mlctx *, lb_tensor *a, uint32_t past);           /* :968 */
LB_API lb_tensor *lb_soft_max(lb_mlctx *, lb_tensor *a);                               /* :993 */
LB_API lb_tensor *lb_silu(lb_mlctx *, lb_tensor *a);                                   /* :1041 */
/* graph */
LB_API lb_graph *lb_graph_new(void);
LB_API void      lb_graph_free(lb_graph *g);
LB_API int       lb_build_forward_expand(lb_graph *g, lb_tensor *t);                   /* :642 */
LB_API int       lb_graph_compute(lb_mlctx *ctx, lb_graph *g);                         /* :1411, synchronous */
LB_API uint32_t  lb_graph_nodes(const lb_graph *g);

#ifdef __cplusplus
}
#endif
#endif /* LLAMAB200_H */
