"""Pins the oracle on F16 input to the reference itself (tests/golden/refbin_f16.json, tools/gen_golden.py f16).

The reference widens F16 tensors to FP32 at load (pkg/llama/llama.go:938-941), so its greedy stream on an F16 ggjt file is
the FP32 computation on the widened weights.  The fixture holds what its binary printed (scalar and --avx) for the tiny and
hd128 models written with F16 matrices; the oracle on the widened weights must reproduce both streams.  The GPU side
(tests/test_gpu_f16.py) checks LB_TYPE_F16 models against the same fixture."""
import hashlib
import json
import os
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN


def _fixture(case):
    with open(os.path.join(GOLDEN, "refbin_f16.json")) as f:
        return json.load(f)[case]


@pytest.mark.parametrize("case", ["tiny", "hd128"])
def test_oracle_reproduces_reference_binary_on_f16_file(oracle, synth, case):
    from oracle import refbin
    rec = _fixture(case)
    hp = synth.HParams(*rec["hparams"])
    vocab = synth.byte_vocab(hp.vocab)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "m.bin")
        synth.write_ggjt(path, hp, synth.synth_model(rec["seed"], hp), vocab, f16=True)
        with open(path, "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == rec["ggjt_sha256"]
        _, _, widened = synth.read_ggjt(path)
    # what the F16 file holds: every 2-D tensor rounded to binary16 (matrices and the embedding table), vectors FP32
    for name, arr in synth.synth_model(rec["seed"], hp):
        exp = synth.round_f16(arr) if arr.ndim == 2 else arr
        np.testing.assert_array_equal(widened[name], exp, err_msg=name)
    tensors = [(n, widened[n]) for n, *_ in synth.tensor_table(hp)]
    for mode in ("scalar", "avx"):
        oracle.set_dot_mode(mode == "avx")
        try:
            c = oracle.OracleContext(oracle.OracleModel(hp).load(tensors), rec["context"])
            toks = oracle.greedy_stream(c, rec["prompt_ids"], rec["predict"], rec["context"])
        finally:
            oracle.set_dot_mode(False)
        expected = refbin.expected_text(vocab, rec["prompt_ids"], toks)
        assert refbin.same_stream(bytes.fromhex(rec["runs"][mode]["text_hex"]), expected), mode
        assert toks == rec["oracle_tokens"], mode
        assert rec["runs"][mode]["evals"] == rec["predict"]


def test_synth_f16_helper_rounds_only_the_matrices(synth):
    hp = synth.HParams(512, 64, 32, 2, 2)
    for (name, a), (name16, b) in zip(synth.synth_model(7, hp), synth.synth_model_f16(7, hp)):
        assert name == name16
        if synth.is_q8_matrix(name):
            np.testing.assert_array_equal(b, a.astype(np.float16).astype(np.float32), err_msg=name)
            assert not np.array_equal(a, b)
        else:
            np.testing.assert_array_equal(b, a, err_msg=name)   # vectors and the embedding table stay FP32
