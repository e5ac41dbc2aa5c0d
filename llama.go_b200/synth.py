"""Synthetic LLaMA models: counter-based weight generator + ggjt v1 writer.

Every weight element is a pure function of (seed, tensor id, flat element index), so any
slice of any tensor can be regenerated bit-identically on the host (numpy, here) and on
the device (csrc/kernels/init_random.cu implements exactly the same integer recipe).  That
is what lets a 7B/13B/65B model be materialised directly in HBM (65B FP32 = 261 GB does not
fit host RAM) while layer-sliced copies of the same model stay checkable against the CPU
oracle.

Recipe (all integer arithmetic mod 2^64, then two FP32 roundings):
    h   = splitmix64(seed * 0x9E3779B97F4A7C15 + tensor_id * 0xD1B54A32D192ED03 + index)
    s   = sum of the four 16-bit fields of h            (Irwin-Hall, 0 .. 262140)
    t   = float32(s - 131070) * float32(sigma / IH_STD) (one rounding; |s-131070| < 2^18 is exact)
    val = float32(mean) + t                             (one rounding; no FMA)
Distributions (SURVEY.md §8d): matrices ~N(0, 1/in_features), norm vectors 1 + 0.1*N(0,1),
embeddings ~N(0,1).

File format: ggjt v1 as read by the reference loader (pkg/llama/llama.go:712-976) and
written by scripts/convert-pth-to-ggml.py:109-137,190-232.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass

import numpy as np

IH_STD = 37837.22539803592  # sqrt(4 * (65536**2 - 1) / 12): std of the sum of four uniform u16
GGJT_MAGIC = 0x67676A74
GGJT_VERSION = 1

_M1 = np.uint64(0x9E3779B97F4A7C15)
_M2 = np.uint64(0xD1B54A32D192ED03)
_S1 = np.uint64(0xBF58476D1CE4E5B9)
_S2 = np.uint64(0x94D049BB133111EB)


@dataclass(frozen=True)
class HParams:
    """HParams of the reference (pkg/llama/llama.go:149-158)."""
    vocab: int
    dim: int
    mult: int
    heads: int
    layers: int

    @property
    def ff(self) -> int:
        # pkg/llama/llama.go:761
        return ((2 * (4 * self.dim) // 3 + self.mult - 1) // self.mult) * self.mult

    @property
    def head_dim(self) -> int:
        return self.dim // self.heads


LLAMA_7B = HParams(32000, 4096, 256, 32, 32)
LLAMA_13B = HParams(32000, 5120, 256, 40, 40)
LLAMA_30B = HParams(32000, 6656, 256, 52, 60)
LLAMA_65B = HParams(32000, 8192, 256, 64, 80)

# per-layer tensor kinds; tensor_id = 16 * (layer + 1) + kind, globals use ids 1..3
_LAYER_KINDS = {
    "attention_norm.weight": 0,
    "attention.wq.weight": 1,
    "attention.wk.weight": 2,
    "attention.wv.weight": 3,
    "attention.wo.weight": 4,
    "ffn_norm.weight": 5,
    "feed_forward.w1.weight": 6,
    "feed_forward.w2.weight": 7,
    "feed_forward.w3.weight": 8,
}
_GLOBAL_IDS = {"tok_embeddings.weight": 1, "norm.weight": 2, "output.weight": 3}


def tensor_table(hp: HParams):
    """[(name, tensor_id, shape [out,in] or [n], mean, sigma)] in ggjt naming (llama.go:826-861)."""
    d, ff, V = hp.dim, hp.ff, hp.vocab
    rows = [
        ("tok_embeddings.weight", 1, (V, d), 0.0, 1.0),
        ("norm.weight", 2, (d,), 1.0, 0.1),
        ("output.weight", 3, (V, d), 0.0, d ** -0.5),
    ]
    for il in range(hp.layers):
        p = f"layers.{il}."
        base = 16 * (il + 1)
        rows += [
            (p + "attention_norm.weight", base + 0, (d,), 1.0, 0.1),
            (p + "attention.wq.weight", base + 1, (d, d), 0.0, d ** -0.5),
            (p + "attention.wk.weight", base + 2, (d, d), 0.0, d ** -0.5),
            (p + "attention.wv.weight", base + 3, (d, d), 0.0, d ** -0.5),
            (p + "attention.wo.weight", base + 4, (d, d), 0.0, d ** -0.5),
            (p + "ffn_norm.weight", base + 5, (d,), 1.0, 0.1),
            (p + "feed_forward.w1.weight", base + 6, (ff, d), 0.0, d ** -0.5),
            (p + "feed_forward.w2.weight", base + 7, (d, ff), 0.0, ff ** -0.5),
            (p + "feed_forward.w3.weight", base + 8, (ff, d), 0.0, d ** -0.5),
        ]
    return rows


def tensor_id(name: str) -> int:
    if name in _GLOBAL_IDS:
        return _GLOBAL_IDS[name]
    parts = name.split(".", 2)
    return 16 * (int(parts[1]) + 1) + _LAYER_KINDS[parts[2]]


def _splitmix64(x: np.ndarray) -> np.ndarray:
    z = x + _M1
    z = (z ^ (z >> np.uint64(30))) * _S1
    z = (z ^ (z >> np.uint64(27))) * _S2
    return z ^ (z >> np.uint64(31))


def synth_values(seed: int, tid: int, start: int, count: int, mean: float, sigma: float) -> np.ndarray:
    """Elements [start, start+count) of tensor `tid` as float32."""
    with np.errstate(over="ignore"):
        base = np.uint64(seed) * _M1 + np.uint64(tid) * _M2
        idx = np.arange(start, start + count, dtype=np.uint64)
        h = _splitmix64(base + idx)
    s = ((h & np.uint64(0xFFFF)) + ((h >> np.uint64(16)) & np.uint64(0xFFFF)) +
         ((h >> np.uint64(32)) & np.uint64(0xFFFF)) + (h >> np.uint64(48))).astype(np.int64)
    t = (s - 131070).astype(np.float32) * np.float32(sigma / IH_STD)
    return (np.float32(mean) + t).astype(np.float32)


def synth_values_fast(seed: int, tid: int, start: int, count: int, mean: float, sigma: float) -> np.ndarray:
    """Same values as synth_values(), produced by the multi-threaded host generator inside
    libllamab200.so (lb_synth_fill_host) — ~100x faster; needs the built library, not a GPU."""
    import ctypes as C
    from . import _capi
    out = np.empty(count, np.float32)
    _capi.check(_capi.lib().lb_synth_fill_host(out.ctypes.data_as(C.POINTER(C.c_float)), count, seed, tid, start,
                                                float(mean), float(sigma)))
    return out


def synth_model_fast(seed: int, hp: HParams):
    for name, tid, shape, mean, sigma in tensor_table(hp):
        yield name, synth_values_fast(seed, tid, 0, int(np.prod(shape)), mean, sigma).reshape(shape)


def synth_tensor(seed: int, name: str, hp: HParams) -> np.ndarray:
    for n, tid, shape, mean, sigma in tensor_table(hp):
        if n == name:
            cnt = int(np.prod(shape))
            return synth_values(seed, tid, 0, cnt, mean, sigma).reshape(shape)
    raise KeyError(name)


def synth_model(seed: int, hp: HParams):
    """Yield (name, float32 ndarray) for every tensor of the model."""
    for name, tid, shape, mean, sigma in tensor_table(hp):
        cnt = int(np.prod(shape))
        yield name, synth_values(seed, tid, 0, cnt, mean, sigma).reshape(shape)


# --------------------------------------------------------------------------- Q8_0 reference (numpy)
def quantize_q8(w: np.ndarray):
    """Q8_0 as defined in DESIGN.md §6 / csrc/kernels_q8.cu: blocks of 32 along the last axis,
    d = max|w| / 127 (FP32), q = rint(w / d) (FP32 divide, round-half-even) clamped to [-127, 127]."""
    w = np.ascontiguousarray(w, dtype=np.float32)
    assert w.shape[-1] % 32 == 0
    blocks = w.reshape(-1, 32)
    d = (np.abs(blocks).max(axis=1) / np.float32(127.0)).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(d[:, None] > 0, np.rint(blocks / d[:, None]), 0.0)
    q = np.clip(q, -127, 127).astype(np.int8)
    return q.reshape(w.shape), d.reshape(w.shape[:-1] + (w.shape[-1] // 32,))


def dequantize_q8(q: np.ndarray, d: np.ndarray) -> np.ndarray:
    return (q.astype(np.float32).reshape(-1, 32) * d.reshape(-1, 1).astype(np.float32)).astype(np.float32).reshape(q.shape)


Q8_MATRICES = ("attention.wq.weight", "attention.wk.weight", "attention.wv.weight", "attention.wo.weight",
               "feed_forward.w1.weight", "feed_forward.w2.weight", "feed_forward.w3.weight", "output.weight")


def is_q8_matrix(name: str) -> bool:
    """The MulMat weights that a Q8_0 model block-quantises (norm vectors and the embedding table stay FP32)."""
    return name.endswith(Q8_MATRICES)


# --------------------------------------------------------------------------- F16 weights
def round_f16(w: np.ndarray) -> np.ndarray:
    """What an LB_TYPE_F16 model holds for an FP32 matrix, widened back: binary16 round-to-nearest-even."""
    return np.asarray(w, np.float32).astype(np.float16).astype(np.float32)


def synth_model_f16(seed: int, hp: HParams):
    """synth_model() as an LB_TYPE_F16 model holds it: the MulMat matrices (is_q8_matrix) rounded to binary16 and
    widened back, norm vectors and the embedding table untouched.  The oracle's input for F16 models."""
    for name, arr in synth_model(seed, hp):
        yield name, round_f16(arr) if is_q8_matrix(name) else arr


# --------------------------------------------------------------------------- vocab
def byte_vocab(vocab_size: int):
    """Synthetic vocab under which the reference tokenizer (pkg/ml/ml.go:2761-2848) maps every
    prompt byte b to id b+3 and never merges: NO single characters and no 2-symbol
    concatenations are in the vocab, so every symbol takes the byte fallback `id = byte + 3`
    (ml.go:2827-2833).  A CLI prompt of k ASCII bytes becomes exactly k+3 tokens: BOS(1) + two
    spaces + bytes (SURVEY.md §8d).  Token strings are `w<id>;` — printable, free of spaces,
    newlines and '%' — because the reference CLI trims ' ' and '\n' from the job output at the
    end (server.go:244) while main.go:137-147 prints it incrementally by length with
    fmt.Printf(diff); any of those characters would corrupt the printed stream."""
    toks = []
    for i in range(vocab_size):
        if i == 0:
            toks.append(b"<unk>")
        elif i in (1, 2):
            toks.append(b"")
        else:
            toks.append(b"w%d;" % i)
    return toks


def merge_vocab(vocab_size: int):
    """A vocab WITH merges, to exercise ml.Tokenize's bigram queue (ml.go:2739-2821): ids 3.. hold
    pieces and their scores (ties included); the rest is filled like byte_vocab().  No piece contains a
    space, newline or '%', so the CLI's printed stream stays intact (see byte_vocab)."""
    pieces = [(b"he", -1.0), (b"ll", -2.0), (b"hell", -3.0), (b"hello", -2.5), (b"lo", -2.0), (b"wo", -4.0), (b"rl", -4.0),
              (b"wor", -5.0), (b"ld", -3.5), (b"world", -1.5), (b"th", -0.5), (b"the", -0.75), (b"el", -2.0), (b"or", -4.0),
              (b"h", -9.0), (b"e", -9.0), (b"l", -9.0), (b"o", -9.0), (b"helloworld", -0.1), (b"ow", -6.0)]
    toks, scores = byte_vocab(vocab_size), [0.0] * vocab_size
    for i, (p, sc) in enumerate(pieces):
        toks[3 + i] = p
        scores[3 + i] = sc
    return toks, scores


def prompt_token_ids(prompt: bytes):
    """Token ids the reference produces for `--prompt <prompt>` with byte_vocab():
    main.go:129 prepends one space, server.go:120 another, Tokenize adds BOS."""
    return [1] + [b + 3 for b in (b"  " + prompt)]


# --------------------------------------------------------------------------- ggjt writer
def write_ggjt(path: str, hp: HParams, tensors, vocab=None, f16: bool = False, scores=None) -> None:
    """Write a ggjt v1 file.  `tensors` = iterable of (name, ndarray[out,in] or [n])."""
    vocab = vocab if vocab is not None else byte_vocab(hp.vocab)
    with open(path, "wb") as f:
        f.write(struct.pack("<9I", GGJT_MAGIC, GGJT_VERSION, hp.vocab, hp.dim, hp.mult, hp.heads,
                            hp.layers, hp.dim // hp.heads, 1 if f16 else 0))
        for i, tok in enumerate(vocab):
            f.write(struct.pack("<I", len(tok)))
            f.write(tok)
            f.write(struct.pack("<f", 0.0 if scores is None else float(scores[i])))
        for name, arr in tensors:
            arr = np.ascontiguousarray(arr)
            nb = name.encode()
            use_f16 = f16 and arr.ndim == 2
            f.write(struct.pack("<3I", arr.ndim, len(nb), 1 if use_f16 else 0))
            for d in reversed(arr.shape):  # dims are written reversed: ne[0] = in_features
                f.write(struct.pack("<I", d))
            f.write(nb)
            pad = (-f.tell()) % 32
            f.write(b"\0" * pad)
            arr.astype("<f2" if use_f16 else "<f4").tofile(f)


def read_ggjt_vocab(path: str):
    """Only the vocab section of a ggjt v1 file: list of token byte strings."""
    with open(path, "rb") as f:
        magic, ver, V = struct.unpack("<3I", f.read(12))
        if magic != GGJT_MAGIC or ver != GGJT_VERSION:
            raise ValueError("not a ggjt v1 file")
        f.read(24)
        vocab = []
        for _ in range(V):
            (ln,) = struct.unpack("<I", f.read(4))
            vocab.append(f.read(ln))
            f.read(4)
        return vocab


def read_ggjt(path: str):
    """Minimal reader (host-side loader for tests): returns (HParams, vocab, {name: ndarray})."""
    with open(path, "rb") as f:
        magic, ver, V, dim, mult, heads, layers, _rot, _ft = struct.unpack("<9I", f.read(36))
        if magic != GGJT_MAGIC or ver != GGJT_VERSION:
            raise ValueError("not a ggjt v1 file")
        hp = HParams(V, dim, mult, heads, layers)
        vocab = []
        for _ in range(V):
            (ln,) = struct.unpack("<I", f.read(4))
            vocab.append(f.read(ln))
            f.read(4)
        tensors = {}
        while True:
            hdr = f.read(12)
            if len(hdr) < 12:
                break
            nd, nl, dt = struct.unpack("<3I", hdr)
            if nd < 1 or nd > 2:
                break
            ne = struct.unpack("<%dI" % nd, f.read(4 * nd))
            name = f.read(nl).decode()
            f.seek((-f.tell()) % 32, 1)
            cnt = int(np.prod(ne))
            if dt == 1:
                arr = np.fromfile(f, dtype="<f2", count=cnt).astype(np.float32)
            else:
                arr = np.fromfile(f, dtype="<f4", count=cnt)
            tensors[name] = arr.reshape(tuple(reversed(ne)))
        return hp, vocab, tensors
