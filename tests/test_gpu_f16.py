"""LB_TYPE_F16 weights: every MulMat matrix held in HBM as IEEE binary16, vectors and the embedding table FP32.

The parity target is the reference's FP32 path on the widened weights (it widens F16 tensors at load, llama.go:938-941):
the oracle on synth.synth_model_f16().  The decode ring and the per-op GEMV read each F16 weight where the FP32 kernels read
the FP32 one and issue the same FMAs in the same order, so they must equal an FP32 model holding the widened weights bit for bit."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN, load_case
from test_gpu_eval import assert_logits_close
from test_gpu_longctx import oracle_prefill

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    import llama_go_b200  # noqa: F401
    from llama_go_b200 import llama
    return llama


def _path(L, lctx):
    return L.lib().lb_context_decode_path(lctx._h).decode()


def _pair(L, synth, hp, seed):
    """(F16 model of synth_model(seed), FP32 model of the same weights widened from binary16)"""
    m16 = L.Model(hp, weight_type=L.LB_TYPE_F16).load(synth.synth_model(seed, hp))
    m32 = L.Model(hp).load(synth.synth_model_f16(seed, hp))
    return m16, m32


# ---- 1. storage ------------------------------------------------------------------------------------------------
def test_f16_storage_rounds_like_numpy(L, synth):
    hp = synth.HParams(320, 128, 32, 4, 2)
    tensors = dict(synth.synth_model(3, hp))
    w = tensors["layers.0.attention.wq.weight"].copy()
    w[0, :8] = [65504.0, -65504.0, 65519.0, 6.1e-5, 5.96e-8, 2.98e-8, 1e-9, 0.0]   # max, rounds-to-max, subnormals, underflow
    w[1, :4] = [1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, -(1.0 + 2.0 ** -11), 2049.0]   # exact ties: to even
    tensors["layers.0.attention.wq.weight"] = w
    model = L.Model(hp, weight_type=L.LB_TYPE_F16).load(tensors.items())
    for name, arr in tensors.items():
        got = model.get_tensor(name, arr.shape)
        exp = arr.astype(np.float16).astype(np.float32) if synth.is_q8_matrix(name) else arr
        np.testing.assert_array_equal(got, exp, err_msg=name)
    # F16 host data is stored byte for byte (and widened into the FP32 vectors / embedding table)
    h = {n: a.astype(np.float16) for n, a in synth.synth_model(4, hp)}
    for n, a in h.items():
        model.set_tensor(n, a)
    for n, a in h.items():
        np.testing.assert_array_equal(model.get_tensor(n, a.shape), a.astype(np.float32), err_msg=n)
    # device-side synthetic weights = the host recipe, rounded
    rnd = L.Model(hp, weight_type=L.LB_TYPE_F16).init_random(5)
    for n, a in synth.synth_model_f16(5, hp):
        np.testing.assert_array_equal(rnd.get_tensor(n, a.shape), a, err_msg=n)
    # a finite value that would round to inf is refused, not stored
    for bad in (65520.0, -7.0e4, 3.0e38):
        w2 = w.copy()
        w2[5, 7] = bad
        with pytest.raises(L.LlamaB200Error, match="F16 range"):
            model.set_tensor("layers.0.attention.wq.weight", w2)
    assert L.Model(synth.LLAMA_7B, weight_type=L.LB_TYPE_F16).weight_bytes_per_token == 13215236096
    with pytest.raises(L.LlamaB200Error):
        L.Model(synth.HParams(64, 48, 16, 2, 1), weight_type=L.LB_TYPE_F16)   # dim not a multiple of 32


# ---- 2. the decode ring is bit-identical to the FP32 ring on the widened weights ----------------------------------
@pytest.mark.parametrize("case", ["tiny", "hd128", "wide3h", "7b_T400"])
def test_f16_ring_bit_identical_to_f32_ring_on_widened_weights(L, synth, case):
    if case == "7b_T400":
        hp, seed, ctx = synth.HParams(2048, 4096, 256, 32, 2), 0, 512
        ids = np.random.RandomState(1).randint(3, hp.vocab, size=401).astype(np.uint32)
    else:
        rec, g = load_case(case)
        hp, seed, ctx = synth.HParams(*rec["hparams"]), rec["seed"], rec["context"]
        ids = np.concatenate([g["prompt_ids"], g["gen_ids"][:6]]).astype(np.uint32)
    m16, m32 = _pair(L, synth, hp, seed)
    c16, c32 = L.NewContext(m16, ctx), L.NewContext(m32, ctx)
    assert _path(L, c16) == "ring_f16" and _path(L, c32) == "ring"
    # every token through the ring (a prompt eval would go through the GEMMs, whose summation order differs)
    L.DecodeResident(c16, ids[:-1], 0)
    L.DecodeResident(c32, ids[:-1], 0)
    assert np.array_equal(L.ReadLogits(c16), L.ReadLogits(c32))
    a = L.Eval(c16, [int(ids[-1])], len(ids) - 1).copy()
    b = L.Eval(c32, [int(ids[-1])], len(ids) - 1).copy()
    assert np.array_equal(a, b)
    k16, v16 = c16.kv(hp.layers - 1, 0, len(ids))
    k32, v32 = c32.kv(hp.layers - 1, 0, len(ids))
    assert np.array_equal(k16, k32) and np.array_equal(v16, v32)


# ---- 3. against the oracle on the golden cases -------------------------------------------------------------------
@pytest.mark.parametrize("case", ["tiny", "hd128", "wide3h", "long"])
def test_f16_eval_matches_oracle_on_widened_weights(L, synth, oracle, case, monkeypatch):
    rec, g = load_case(case)
    hp = synth.HParams(*rec["hparams"])
    m16, m32 = _pair(L, synth, hp, rec["seed"])
    om = oracle.OracleModel(hp).load(synth.synth_model_f16(rec["seed"], hp))
    ids = g["prompt_ids"]
    # prompt, every row: the F16 tcgen05 GEMM
    c16 = L.NewContext(m16, rec["context"])
    oc = oracle.OracleContext(om, rec["context"])
    got = L.EvalAllLogits(c16, ids, 0)
    _, ref = oc.eval(ids, 0, all_logits=True)
    kernel_err = assert_logits_close(got, ref, what=f"{case} F16 prefill")
    f32 = L.EvalAllLogits(L.NewContext(m32, rec["context"]), ids, 0)
    assert np.abs(got - f32).max() <= 1e-5 * np.abs(f32).max()
    # 6 decode steps (first eager, then CUDA-graph replay): the ring where the shape allows, else gemv_f16
    past, refs = len(ids), []
    for tok in g["gen_ids"][:6]:
        got = L.Eval(c16, [int(tok)], past).copy()
        ref = oc.eval([int(tok)], past)
        refs.append(ref)
        kernel_err = max(kernel_err, assert_logits_close(got, ref, what=f"{case} F16 decode past {past}"))
        past += 1
    # the rounding moves the logits by far more than the kernel error: the comparison can tell F16 from FP32
    assert np.abs(refs[-1] - g["step_logits"][6]).max() > 10 * kernel_err * np.abs(refs[-1]).max()
    # a short prompt (N <= 8) goes through gemv_f16 (multi-column); equal to the FP32 GEMV on the widened weights
    got = L.Eval(L.NewContext(m16, rec["context"]), ids[:5], 0).copy()
    assert_logits_close(got, oracle.OracleContext(om, rec["context"]).eval(ids[:5], 0), what=f"{case} F16 5-token prompt")
    assert np.array_equal(got, L.Eval(L.NewContext(m32, rec["context"]), ids[:5], 0))
    # LB_NO_MEGA=1: per-op decode through gemv_f16 / gemv_f16_swiglu
    monkeypatch.setenv("LB_NO_MEGA", "1")
    c = L.NewContext(m16, rec["context"])
    assert _path(L, c) == "perop"
    L.Eval(c, ids, 0)
    past = len(ids)
    for tok, ref in zip(g["gen_ids"][:6], refs):
        assert_logits_close(L.Eval(c, [int(tok)], past), ref, what=f"{case} F16 per-op decode past {past}")
        past += 1


# ---- 4. the operating shapes -------------------------------------------------------------------------------------
SHAPED = [
    ("7B",  (2048, 4096, 256, 32, 2), 512, 400),
    ("13B", (2048, 5120, 256, 40, 1), 512, 480),
    ("65B", (2048, 8192, 256, 64, 1), 2048, 1900),
]
_SHAPED_REF = {}


@pytest.mark.parametrize("path", ["ring_f16", "perop"])
@pytest.mark.parametrize("name,dims,ctx,T", SHAPED, ids=[s[0] for s in SHAPED])
def test_f16_shaped_layers_at_operating_T_against_oracle(L, synth, oracle, name, dims, ctx, T, path, monkeypatch):
    if path == "perop":
        monkeypatch.setenv("LB_NO_MEGA", "1")
    else:
        monkeypatch.delenv("LB_NO_MEGA", raising=False)
    hp = synth.HParams(*dims)
    model = L.Model(hp, weight_type=L.LB_TYPE_F16).init_random(0)
    rs = np.random.RandomState(7)
    ids = rs.randint(3, hp.vocab, size=T).astype(np.uint32)
    gen = rs.randint(3, hp.vocab, size=4).astype(np.uint32)
    if name not in _SHAPED_REF:
        tensors = [(n, synth.round_f16(a) if synth.is_q8_matrix(n) else a) for n, a in synth.synth_model_fast(0, hp)]
        oracle.set_dot_mode(True)
        try:
            oc = oracle.OracleContext(oracle.OracleModel(hp).load(tensors), ctx)
            _SHAPED_REF[name] = (oracle_prefill(oc, ids), [oc.eval([int(t)], T + i) for i, t in enumerate(gen)])
        finally:
            oracle.set_dot_mode(False)
    ref_prefill, ref_steps = _SHAPED_REF[name]
    lctx = L.NewContext(model, ctx)
    assert _path(L, lctx) == path
    e0 = assert_logits_close(L.Eval(lctx, ids, 0).copy(), ref_prefill, what=f"{name}-shape F16 prefill T={T}")
    for i, t in enumerate(gen):
        e1 = assert_logits_close(L.Eval(lctx, [int(t)], T + i).copy(), ref_steps[i], what=f"{name}-shape F16 {path} decode past {T + i}")
    print(f"[{name}-shaped F16 {path}, ctx {ctx}] prefill rel err {e0:.3e}, decode rel err {e1:.3e}")


# ---- 5. pods -----------------------------------------------------------------------------------------------------
def test_f16_pod_batch_matches_solo_decodes_and_oracle(L, synth, oracle):
    rec, g = load_case("hd128")
    hp = synth.HParams(*rec["hparams"])
    model = L.Model(hp, weight_type=L.LB_TYPE_F16).load(synth.synth_model(rec["seed"], hp))
    om = oracle.OracleModel(hp).load(synth.synth_model_f16(rec["seed"], hp))
    ids = [int(t) for t in g["prompt_ids"]]
    gen = [int(t) for t in g["gen_ids"][:-1]]
    B = 4
    pods, solo, orc = [], [], []
    for b in range(B):
        pc, sc, oc = L.NewContext(model, rec["context"]), L.NewContext(model, rec["context"]), oracle.OracleContext(om, rec["context"])
        for c in (pc, sc):
            L.Eval(c, ids, 0)
            for i in range(b):
                L.Eval(c, [gen[i]], len(ids) + i)
        oc.eval(ids, 0)
        for i in range(b):
            oc.eval([gen[i]], len(ids) + i)
        pods.append(pc); solo.append(sc); orc.append(oc)
    batch = L.PodBatch(pods)
    for step in range(3):
        toks = [gen[b + step] for b in range(B)]
        pasts = [len(ids) + b + step for b in range(B)]
        got = batch.Eval(toks, pasts)
        for b in range(B):
            ref_solo = L.Eval(solo[b], [toks[b]], pasts[b])
            assert np.abs(got[b] - ref_solo).max() <= 2e-5 * np.abs(ref_solo).max()
            assert_logits_close(got[b], orc[b].eval([toks[b]], pasts[b]), what=f"F16 pod {b} step {step}")


# ---- 6. the reference binary's streams on an F16 ggjt file -------------------------------------------------------
@pytest.mark.parametrize("case", ["tiny", "hd128"])
def test_f16_ggjt_file_generates_reference_stream(L, synth, case):
    import json
    with open(os.path.join(GOLDEN, "refbin_f16.json")) as f:
        rec = json.load(f)[case]
    hp = synth.HParams(*rec["hparams"])
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "m.bin")
        synth.write_ggjt(path, hp, synth.synth_model(rec["seed"], hp), synth.byte_vocab(hp.vocab), f16=True)
        for wt in (L.LB_TYPE_F16, L.LB_TYPE_F32):
            _, model = L.LoadModel(path, weight_type=wt)
            lctx = L.NewContext(model, rec["context"])
            assert L.GenerateGreedy(lctx, rec["prompt_ids"], rec["predict"]) == rec["oracle_tokens"], wt
        # the loader stores the file's F16 bytes as they are
        _, model = L.LoadModel(path, weight_type=L.LB_TYPE_F16)
        _, _, widened = synth.read_ggjt(path)
        for n, a in widened.items():
            np.testing.assert_array_equal(model.get_tensor(n, a.shape), a, err_msg=n)


# ---- 7. refusals ---------------------------------------------------------------------------------------------------
def test_f16_refusals_leave_the_process_usable(L, synth, oracle):
    rec, g = load_case("tiny")
    hp = synth.HParams(*rec["hparams"])
    model = L.Model(hp, weight_type=L.LB_TYPE_F16).load(synth.synth_model(rec["seed"], hp))
    lctx = L.NewContext(model, rec["context"])
    ids = g["prompt_ids"]
    with pytest.raises(L.LlamaB200Error, match="FP32 only"):
        L.EvalGraph(lctx, ids, 0)
    ms, nb = C.c_float(0), C.c_uint64(0)
    with pytest.raises(L.LlamaB200Error, match="F32 and Q8_0"):
        L.check(L.lib().lb_bench_kernel(lctx._h, 0, 4, 0, C.byref(ms), C.byref(nb)))
    arr = (C.c_void_p * 1)(lctx._h)
    with pytest.raises(L.LlamaB200Error, match="F16"):
        L.check(L.lib().lb_pipeline_p2p_import(arr, 1, None, None))
    ref = oracle.OracleContext(oracle.OracleModel(hp).load(synth.synth_model_f16(rec["seed"], hp)), rec["context"]).eval(ids, 0)
    assert_logits_close(L.Eval(lctx, ids, 0), ref, what="eval after the refusals")
