"""Python mirror of the reference's pkg/llama hot-path API (pkg/llama/llama.go:83-113, 211-426).

    model = llama.Model(hp); model.load(tensors) | model.init_random(seed) | llama.LoadModel(path)
    lctx  = llama.NewContext(model, ctx_size)
    llama.Eval(lctx, tokens, pastCount)      # fills lctx.Logits (row N-1), like the reference
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi, synth
from ._capi import HParamsC, LlamaB200Error, check, check_ptr, lib  # noqa: F401

_f32p = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)
LB_TYPE_F32, LB_TYPE_F16, LB_TYPE_Q8_0 = 0, 1, 16  # include/llamab200.h


class Model:
    """llama.Model (llama.go:181-193), device resident.  layer range = pipeline stage."""

    def __init__(self, hp: synth.HParams, device: int = 0, layer_begin: int = 0, layer_end: int | None = None,
                 weight_type: int = 0):
        _capi.require_gpu()
        self.hp = hp
        self.device = device
        self.layer_begin = layer_begin
        self.layer_end = hp.layers if layer_end is None else layer_end
        c = HParamsC(hp.vocab, hp.dim, hp.mult, hp.heads, hp.layers)
        self._h = check_ptr(lib().lb_model_create(C.byref(c), device, self.layer_begin, self.layer_end, weight_type))

    def set_tensor(self, name: str, arr: np.ndarray) -> None:
        if arr.dtype == np.float16:
            a, dt = np.ascontiguousarray(arr), 1
        else:
            a, dt = np.ascontiguousarray(arr, dtype=np.float32), 0
        check(lib().lb_model_set_tensor(self._h, name.encode(), dt, a.ctypes.data_as(C.c_void_p), a.nbytes))

    def get_tensor(self, name: str, shape) -> np.ndarray:
        out = np.empty(int(np.prod(shape)), np.float32)
        check(lib().lb_model_get_tensor(self._h, name.encode(), out.ctypes.data_as(_f32p), out.size))
        return out.reshape(shape)

    def load(self, tensors) -> "Model":
        for name, arr in tensors:
            self.set_tensor(name, arr)
        return self

    def init_random(self, seed: int) -> "Model":
        check(lib().lb_model_init_random(self._h, seed))
        return self

    @property
    def weight_bytes_per_token(self) -> int:
        return lib().lb_model_weight_bytes(self._h)

    def free(self):
        if self._h:
            lib().lb_model_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def LoadModel(fileName: str, device: int = 0, weight_type: int = LB_TYPE_F32, layer_begin: int = 0, layer_end: int = 0):
    """LoadModel (llama.go:712-976): ggjt v1 file -> Model, streamed into HBM by the native loader
    (csrc/loader.cpp).  Returns (vocab, model) like the reference; the vocab is read on the host."""
    _capi.require_gpu()
    c = HParamsC()
    h = check_ptr(lib().lb_model_load_ggjt(fileName.encode(), device, layer_begin, layer_end, weight_type, C.byref(c)))
    hp = synth.HParams(c.vocab, c.dim, c.mult, c.heads, c.layers)
    m = Model.__new__(Model)
    m.hp, m.device, m.layer_begin, m.layer_end, m._h = hp, device, layer_begin, layer_end or hp.layers, h
    vocab = synth.read_ggjt_vocab(fileName)
    return vocab, m


class Context:
    """llama.Context (llama.go:83-88): KV cache + Logits."""

    def __init__(self, model: Model, ctx_size: int):
        self.model = model
        self.ctx_size = ctx_size
        self._h = check_ptr(lib().lb_context_create(model._h, ctx_size))
        self.Logits = np.zeros(model.hp.vocab, np.float32)

    def ReleaseContext(self):
        if self._h:
            lib().lb_context_free(self._h)
            self._h = None

    def kv(self, layer: int, t0: int, nt: int):
        d = self.model.hp.dim
        k = np.empty((nt, d), np.float32)
        v = np.empty((nt, d), np.float32)
        check(lib().lb_context_read_kv(self._h, layer, t0, nt, k.ctypes.data_as(_f32p), v.ctypes.data_as(_f32p)))
        return k, v

    def hidden(self, n: int) -> np.ndarray:
        out = np.empty((n, self.model.hp.dim), np.float32)
        check(lib().lb_context_read_hidden(self._h, n, out.ctypes.data_as(_f32p)))
        return out

    def __del__(self):
        try:
            self.ReleaseContext()
        except Exception:
            pass


def NewContext(model: Model, ctx_size: int) -> Context:
    return Context(model, ctx_size)


def _toks(tokens):
    t = np.ascontiguousarray(tokens, dtype=np.uint32).reshape(-1)
    return t, t.ctypes.data_as(_u32p)


def Eval(lctx: Context, tokens, pastCount: int) -> np.ndarray:
    """llama.Eval (llama.go:211-426).  Fills and returns lctx.Logits."""
    t, p = _toks(tokens)
    check(lib().lb_eval(lctx._h, p, t.size, pastCount, lctx.Logits.ctypes.data_as(_f32p)))
    return lctx.Logits


def EvalAllLogits(lctx: Context, tokens, pastCount: int) -> np.ndarray:
    t, p = _toks(tokens)
    out = np.empty((t.size, lctx.model.hp.vocab), np.float32)
    check(lib().lb_eval_all_logits(lctx._h, p, t.size, pastCount, out.ctypes.data_as(_f32p)))
    lctx.Logits[:] = out[-1]
    return out


def EvalGraph(lctx: Context, tokens, pastCount: int) -> np.ndarray:
    """The same Eval, built node for node with the pkg/ml op API and run by GraphCompute."""
    t, p = _toks(tokens)
    check(lib().lb_eval_graph(lctx._h, p, t.size, pastCount, lctx.Logits.ctypes.data_as(_f32p)))
    return lctx.Logits


def DecodeResident(lctx: Context, tokens, pastCount: int) -> float:
    """Teacher-forced single-token evals enqueued back to back, no host copies; returns CUDA-event ms."""
    t, p = _toks(tokens)
    ms = C.c_float(0)
    check(lib().lb_decode_resident(lctx._h, p, t.size, pastCount, C.byref(ms)))
    return ms.value


def GenerateGreedy(lctx: Context, prompt_ids, predict: int, temp: float = 1e-6, repeat_penalty: float = 1.10):
    """pkg/server.Do's generate loop at temp -> 0 with the sampler on the device; returns the generated ids."""
    t, p = _toks(prompt_ids)
    out = np.zeros(predict, np.uint32)
    check(lib().lb_generate_greedy(lctx._h, p, t.size, predict, temp, repeat_penalty, out.ctypes.data_as(_u32p)))
    return out.tolist()


def SampleTopPTopK(lctx: Context, lastNTokens, topK: int = 40, topP: float = 0.95, temp: float = 0.8, repeatPenalty: float = 1.10,
                   seed: int = 0):
    """llama.SampleTopPTopK (llama.go:455-707) on the device, on the logits of lctx's last Eval.  Returns
    (token, candidate ids, candidate probabilities) — the candidate set after the top-k and top-p cuts."""
    t, p = _toks(lastNTokens)
    ids = np.zeros(topK, np.uint32)
    probs = np.zeros(topK, np.float32)
    n, tok = C.c_uint32(0), C.c_uint32(0)
    check(lib().lb_sample_top_p_top_k(lctx._h, p, t.size, topK, topP, temp, repeatPenalty, seed, ids.ctypes.data_as(_u32p),
                                      probs.ctypes.data_as(_f32p), C.byref(n), C.byref(tok)))
    return tok.value, ids[:n.value].copy(), probs[:n.value].copy()


def Generate(lctx: Context, prompt_ids, predict: int, topK: int = 40, topP: float = 0.95, temp: float = 0.8, repeatPenalty: float = 1.10,
             keepCount: int = 0, batchSize: int | None = None, seed: int = 0):
    """The generate loop of pkg/server.Do (server.go:127-237) incl. the context swap (:158-172); returns the sampled ids."""
    t, p = _toks(prompt_ids)
    out = np.zeros(predict, np.uint32)
    check(lib().lb_generate(lctx._h, p, t.size, predict, topK, topP, temp, repeatPenalty, keepCount,
                            batchSize if batchSize else lctx.ctx_size, seed, out.ctypes.data_as(_u32p)))
    return out.tolist()


def ContextSwap(ctxSize: int, keepCount: int, history, pastCount: int, embd):
    """The context-swap rule of server.Do (server.go:165-172): returns (new pastCount, new embd)."""
    h, hp_ = _toks(history)
    e, ep = _toks(embd)
    past = C.c_uint32(pastCount)
    out = np.zeros(h.size + e.size + 1, np.uint32)
    n = lib().lb_context_swap(ctxSize, keepCount, hp_, h.size, C.byref(past), ep, e.size, out.ctypes.data_as(_u32p), out.size)
    if n < 0:
        check(1)
    return past.value, out[:n].tolist()


class PodBatch:
    """Up to 8 llama.Contexts ("pods", pkg/server/server.go:84-106) of one Model decoded together: one
    pass over the weights per step for all of them (SURVEY §8f-1)."""

    def __init__(self, ctxs):
        self.ctxs = list(ctxs)
        self.vocab = self.ctxs[0].model.hp.vocab
        arr = (C.c_void_p * len(self.ctxs))(*[c._h for c in self.ctxs])
        self._h = check_ptr(lib().lb_batch_create(arr, len(self.ctxs)))

    def Eval(self, tokens, pasts) -> np.ndarray:
        """tokens[n], pasts[n] -> logits [n][vocab] (row b = llama.Eval(ctxs[b], [tokens[b]], pasts[b]))."""
        t, tp = _toks(tokens)
        p, pp = _toks(pasts)
        if t.size != len(self.ctxs) or p.size != len(self.ctxs):
            raise ValueError("PodBatch.Eval: need one token and one position per pod")
        out = np.empty((len(self.ctxs), self.vocab), np.float32)
        check(lib().lb_batch_eval(self._h, tp, pp, out.ctypes.data_as(_f32p)))
        return out

    def DecodeResident(self, tokens, pasts) -> float:
        t = np.ascontiguousarray(tokens, dtype=np.uint32)
        p, pp = _toks(pasts)
        if t.ndim != 2 or t.shape[0] != len(self.ctxs) or p.size != len(self.ctxs):
            raise ValueError("PodBatch.DecodeResident: tokens must be [pods][steps], pasts [pods]")
        ms = C.c_float(0)
        check(lib().lb_batch_decode_resident(self._h, t.ctypes.data_as(_u32p), t.shape[1], pp, C.byref(ms)))
        return ms.value

    def ReadLogits(self) -> np.ndarray:
        out = np.empty((len(self.ctxs), self.vocab), np.float32)
        check(lib().lb_batch_read_logits(self._h, out.ctypes.data_as(_f32p)))
        return out

    def _seeds(self, seeds, what):
        s = np.ascontiguousarray(range(len(self.ctxs)) if seeds is None else seeds, dtype=np.uint64).reshape(-1)
        if s.size != len(self.ctxs):
            raise ValueError(f"PodBatch.{what}: need one seed per pod")
        return s, s.ctypes.data_as(C.POINTER(C.c_uint64))

    def SampleTopPTopK(self, lastN, topK: int = 40, topP: float = 0.95, temp: float = 0.8, repeatPenalty: float = 1.10, seeds=None):
        """SampleTopPTopK for every pod on the batch's last logits (row b with lastN[b] and seeds[b], default b).  Returns
        (tokens [n], candidate ids per pod, candidate probabilities per pod), as llama.SampleTopPTopK does for one context."""
        n = len(self.ctxs)
        last = np.ascontiguousarray(lastN, dtype=np.uint32)
        if last.ndim != 2 or last.shape[0] != n:
            raise ValueError("PodBatch.SampleTopPTopK: lastN must be [pods][n_last]")
        s, sp = self._seeds(seeds, "SampleTopPTopK")
        ids = np.zeros((n, topK), np.uint32)
        probs = np.zeros((n, topK), np.float32)
        cnt = np.zeros(n, np.uint32)
        toks = np.zeros(n, np.uint32)
        check(lib().lb_batch_sample(self._h, last.ctypes.data_as(_u32p), last.shape[1], topK, topP, temp, repeatPenalty, sp,
                                    ids.ctypes.data_as(_u32p), probs.ctypes.data_as(_f32p), cnt.ctypes.data_as(_u32p),
                                    toks.ctypes.data_as(_u32p)))
        return toks.tolist(), [ids[b, :cnt[b]].copy() for b in range(n)], [probs[b, :cnt[b]].copy() for b in range(n)]

    def Generate(self, prompts, predict: int, topK: int = 40, topP: float = 0.95, temp: float = 0.8, repeatPenalty: float = 1.10,
                 keepCount: int = 0, batchSize: int | None = None, seeds=None, return_ms: bool = False):
        """llama.Generate for every pod at once (pkg/server.Do per job, server.go:127-237): prompts[b] on pod b with
        seeds[b] (default b).  Returns one list of `predict` ids per pod (and the decode phase's CUDA-event ms if
        return_ms)."""
        n = len(self.ctxs)
        if len(prompts) != n:
            raise ValueError("PodBatch.Generate: need one prompt per pod")
        lens = np.asarray([len(p) for p in prompts], np.uint32)
        cat = np.ascontiguousarray(np.concatenate([np.asarray(p, np.uint32).reshape(-1) for p in prompts]), dtype=np.uint32)
        s, sp = self._seeds(seeds, "Generate")
        out = np.zeros((n, predict), np.uint32)
        ms = C.c_float(0)
        check(lib().lb_batch_generate(self._h, cat.ctypes.data_as(_u32p), lens.ctypes.data_as(_u32p), predict, topK, topP, temp,
                                      repeatPenalty, keepCount, self.ctxs[0].ctx_size if batchSize is None else batchSize, sp,
                                      out.ctypes.data_as(_u32p), C.byref(ms)))
        toks = [row.tolist() for row in out]
        return (toks, ms.value) if return_ms else toks

    def free(self):
        if self._h:
            lib().lb_batch_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def ReadLogits(lctx: Context) -> np.ndarray:
    check(lib().lb_context_read_logits(lctx._h, lctx.Logits.ctypes.data_as(_f32p)))
    return lctx.Logits
