#!/usr/bin/env python
"""Generate the committed fixtures under tests/golden/.

Runs ONLY in the build container (needs /root/reference via oracle/_ref):
  1. refbin_<case>.json — output of the REFERENCE ITSELF: the greedy text the reference's
     prebuilt binary prints for a synthetic ggjt model (scalar and --avx), plus the model
     recipe (hparams, seed, prompt).  tests/test_oracle_vs_refbin.py re-derives the same text
     from the CPU restatement (oracle/) and requires equality — this is what pins the oracle.
  2. logits_<case>.npz — teacher-forced logits of the pinned oracle for the same models
     (prompt eval + decode steps, scalar dot order), the golden vectors the GPU path is
     compared against on the GPU box (where /root/reference does not exist).

Usage: python tools/gen_golden.py [case ...]            # refbin_<case>.json, logits_<case>.npz
       python tools/gen_golden.py swap|threads2|vdot    # refbin_swap.json, refbin_threads2.json, vdot_ref.npz
       python tools/gen_golden.py f16                   # refbin_f16.json

refbin_f16.json pins F16 input (the format LLaMA ggjt checkpoints most often come in): the reference binary's scalar and
--avx greedy streams on the tiny and hd128 models written with F16 matrices, the SHA-256 of those files, and the oracle's
tokens on the widened weights.  LB_TYPE_F16 models (the MulMat matrices held as binary16) are checked against it on the GPU.
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import llama_go_b200  # noqa: E402,F401
from llama_go_b200 import synth  # noqa: E402
from oracle import oracle as O, refbin  # noqa: E402

CASES = [
    # name, (vocab, dim, mult, heads, layers), seed, prompt, context, predict
    ("tiny", (512, 64, 32, 2, 2), 7, "hello world, this is a test", 128, 24),
    ("hd128", (1024, 256, 64, 2, 3), 11, "The quick brown fox jumps over", 128, 24),
    ("wide3h", (768, 384, 128, 3, 2), 23, "abcde", 64, 16),  # 8-token prompt: the --avx edge (T>=8)
    ("long", (512, 128, 32, 4, 2), 5, "x" * 61, 160, 40),    # 64-token prompt, T up to 104
    # vocab WITH merges: pins ml.Tokenize (csrc/tokenizer.cpp) to the reference through the generated stream
    ("merges", (512, 64, 32, 2, 2), 13, "hello world the hell helloworld lower", 128, 16),
]


def main():
    O.build()
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    only = set(sys.argv[1:])
    for name, hpt, seed, prompt, context, predict in CASES:
        if only and name not in only:
            continue
        hp = synth.HParams(*hpt)
        scores = None
        if name == "merges":
            from llama_go_b200 import ml
            vocab, scores = synth.merge_vocab(hp.vocab)
            # main.go:129 and server.go:120 each prepend one space; Tokenize adds BOS
            ids = ml.Tokenize(ml.Vocab(vocab, scores), b"  " + prompt.encode(), True)
        else:
            vocab = synth.byte_vocab(hp.vocab)
            ids = synth.prompt_token_ids(prompt.encode())
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "m.bin")
            synth.write_ggjt(path, hp, synth.synth_model(seed, hp), vocab, scores=scores)
            rec = {"hparams": list(hpt), "seed": seed, "prompt": prompt, "prompt_ids": ids,
                   "context": context, "predict": predict, "runs": {}}
            for mode, threads, avx in (("scalar", 1, False), ("avx", 4, True)):
                r = refbin.run(path, prompt, predict, context, threads, avx)
                rec["runs"][mode] = {"threads": threads, "text_hex": r["text"].hex()}
                print(f"[{name}/{mode}] binary text len {len(r['text'])}")
        # oracle streams (scalar order) + margins, and teacher-forced golden logits
        O.set_dot_mode(False)
        m = O.OracleModel(hp).load(synth.synth_model(seed, hp))
        c = O.OracleContext(m, context)
        toks, logits, margins = O.greedy_stream(c, ids, predict, context, return_logits=True)
        rec["oracle_tokens"] = toks
        rec["min_margin"] = min(margins)
        for mode in rec["runs"]:
            exp = refbin.expected_text(vocab, ids, toks)
            got = bytes.fromhex(rec["runs"][mode]["text_hex"])
            ok = refbin.same_stream(got, exp)
            print(f"[{name}/{mode}] oracle == binary: {ok}  (min margin {min(margins):.4g})")
            if not ok:
                print(got); print(exp)
                raise SystemExit(f"oracle does not reproduce the reference binary on case {name}/{mode}")
        with open(os.path.join(out_dir, f"refbin_{name}.json"), "w") as f:
            json.dump(rec, f, indent=1)
        # teacher-forced: prompt eval with all rows, then each generated token
        c2 = O.OracleContext(m, context)
        last, allrows, hid = c2.eval(ids, 0, all_logits=True, hidden=True)
        k, v = c2.kv()
        np.savez_compressed(
            os.path.join(out_dir, f"logits_{name}.npz"),
            prompt_ids=np.asarray(ids, np.uint32), gen_ids=np.asarray(toks, np.uint32),
            prompt_all_logits=allrows, prompt_hidden=hid, step_logits=logits,
            k_after_prompt=k[:, :len(ids)].copy(), v_after_prompt=v[:, :len(ids)].copy())
    print("done")


if __name__ == "__main__" and not {"swap", "threads2", "vdot", "f16"} & set(sys.argv[1:]):
    main()


def gen_swap():
    """refbin_swap.json — the reference binary run PAST its context (context 40, 30-token prompt, predict 40): the
    context-swap rule of server.go:158-172 fires three times.  Pins oracle.generate_stream (and through it
    lb_generate / lb_context_swap)."""
    O.build()
    hpt, seed, prompt, context, predict = (512, 64, 32, 2, 2), 7, "hello world, this is a test", 40, 40
    hp = synth.HParams(*hpt)
    vocab = synth.byte_vocab(hp.vocab)
    ids = synth.prompt_token_ids(prompt.encode())
    rec = {"hparams": list(hpt), "seed": seed, "prompt": prompt, "prompt_ids": ids, "context": context, "predict": predict, "runs": {}}
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "m.bin")
        synth.write_ggjt(path, hp, synth.synth_model(seed, hp), vocab)
        for mode, avx, thr in (("scalar", False, 1), ("avx", True, 4)):
            r = refbin.run(path, prompt, predict, context, thr, avx, port=18190)
            rec["runs"][mode] = {"text_hex": r["text"].hex(), "evals": len(r["eval_ms"])}
    m = O.OracleModel(hp).load(synth.synth_model(seed, hp))
    toks = O.generate_stream(O.OracleContext(m, context), ids, predict, context)
    exp = refbin.expected_text(vocab, ids, toks)
    for mode in rec["runs"]:
        assert refbin.same_stream(bytes.fromhex(rec["runs"][mode]["text_hex"]), exp), mode
    rec["oracle_tokens"] = toks
    with open(os.path.join(ROOT, "tests", "golden", "refbin_swap.json"), "w") as f:
        json.dump(rec, f)
    print("swap:", len(toks), "tokens")


if __name__ == "__main__" and "swap" in sys.argv[1:]:
    gen_swap()


def gen_threads2():
    """refbin_threads2.json — the reference binary (--avx, 2 threads) on the ggjt files synth.write_ggjt makes for the tiny
    and hd128 cases: the file's SHA-256, the printed stream and the number of evals it timed.  Pins the ggjt writer and
    the oracle's --avx stream to a third thread count."""
    O.build()
    out = {}
    for name in ("tiny", "hd128"):
        with open(os.path.join(ROOT, "tests", "golden", f"refbin_{name}.json")) as f:
            rec = json.load(f)
        hp = synth.HParams(*rec["hparams"])
        vocab = synth.byte_vocab(hp.vocab)
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "m.bin")
            synth.write_ggjt(path, hp, synth.synth_model(rec["seed"], hp), vocab)
            with open(path, "rb") as f:
                sha = hashlib.sha256(f.read()).hexdigest()
            r = refbin.run(path, rec["prompt"], rec["predict"], rec["context"], 2, True, port=18181)
        exp = refbin.expected_text(vocab, rec["prompt_ids"], rec["oracle_tokens"])
        assert refbin.same_stream(r["text"], exp), name
        out[name] = {"threads": 2, "avx": True, "ggjt_sha256": sha, "text_hex": r["text"].hex(), "evals": len(r["eval_ms"])}
        print(f"[{name}/threads2] binary text len {len(r['text'])}, {len(r['eval_ms'])} evals")
    with open(os.path.join(ROOT, "tests", "golden", "refbin_threads2.json"), "w") as f:
        json.dump(out, f, indent=1)


def gen_vdot():
    """vdot_ref.npz — _mm256_dot of the reference's utils/floats_avx.c, compiled as-is (oracle/_ref/libvdot_ref.so), on
    seeded vectors of the lengths that exercise its 8-lane body and scalar tail.  Pins the oracle's --avx dot order."""
    import ctypes as C
    O.build()
    L = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libvdot_ref.so"))
    fp = C.POINTER(C.c_float)
    L._mm256_dot.argtypes = [fp, fp, C.c_int64, fp]
    rng = np.random.default_rng(0)
    ns = [8, 9, 15, 16, 128, 131, 4096, 11008]
    a = rng.standard_normal(sum(ns)).astype(np.float32)
    b = rng.standard_normal(sum(ns)).astype(np.float32)
    dots, off = [], 0
    for n in ns:
        ret = C.c_float(0)
        L._mm256_dot(a[off:].ctypes.data_as(fp), b[off:].ctypes.data_as(fp), n, C.byref(ret))
        dots.append(ret.value)
        off += n
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "vdot_ref.npz"), n=np.asarray(ns, np.int64), a=a, b=b,
                        dot=np.asarray(dots, np.float32))


if __name__ == "__main__" and "threads2" in sys.argv[1:]:
    gen_threads2()
if __name__ == "__main__" and "vdot" in sys.argv[1:]:
    gen_vdot()


def gen_f16():
    """refbin_f16.json — the reference binary (scalar, and --avx at 4 threads) on the ggjt files synth.write_ggjt(f16=True) makes for
    the tiny and hd128 cases (every 2-D tensor stored as F16, which the reference widens at load): the files' SHA-256, the printed
    streams, and the oracle's stream on the widened weights.  The F16 rounding must move the logits measurably against the FP32
    fixtures (logits_<case>.npz), or the pin could not tell F16 input apart from FP32."""
    O.build()
    out = {}
    for name in ("tiny", "hd128"):
        with open(os.path.join(ROOT, "tests", "golden", f"refbin_{name}.json")) as f:
            base = json.load(f)
        g = np.load(os.path.join(ROOT, "tests", "golden", f"logits_{name}.npz"))
        hp = synth.HParams(*base["hparams"])
        vocab = synth.byte_vocab(hp.vocab)
        ids = base["prompt_ids"]
        rec = {k: base[k] for k in ("hparams", "seed", "prompt", "prompt_ids", "context", "predict")}
        rec["runs"] = {}
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "m.bin")
            synth.write_ggjt(path, hp, synth.synth_model(base["seed"], hp), vocab, f16=True)
            with open(path, "rb") as f:
                rec["ggjt_sha256"] = hashlib.sha256(f.read()).hexdigest()
            for mode, threads, avx in (("scalar", 1, False), ("avx", 4, True)):
                r = refbin.run(path, base["prompt"], base["predict"], base["context"], threads, avx, port=18183)
                rec["runs"][mode] = {"threads": threads, "text_hex": r["text"].hex(), "evals": len(r["eval_ms"])}
            _, _, widened = synth.read_ggjt(path)
        tensors = [(n, widened[n]) for n, *_ in synth.tensor_table(hp)]
        for mode in ("scalar", "avx"):
            O.set_dot_mode(mode == "avx")
            try:
                c = O.OracleContext(O.OracleModel(hp).load(tensors), base["context"])
                toks, logits, margins = O.greedy_stream(c, ids, base["predict"], base["context"], return_logits=True)
            finally:
                O.set_dot_mode(False)
            exp = refbin.expected_text(vocab, ids, toks)
            assert refbin.same_stream(bytes.fromhex(rec["runs"][mode]["text_hex"]), exp), (name, mode)
            if mode == "scalar":
                rec["oracle_tokens"] = toks
                rec["min_margin"] = min(margins)
                shift = float(np.abs(logits[0] - g["step_logits"][0]).max() / np.abs(g["step_logits"][0]).max())
            else:
                assert toks == rec["oracle_tokens"], name
        # a pin that cannot tell F16 from FP32 pins nothing: the rounding must move the prompt logits far beyond summation noise
        assert shift > 1e-4, (name, shift)
        rec["prompt_logit_shift_vs_f32"] = shift
        rec["differs_from_f32_stream"] = rec["oracle_tokens"] != base["oracle_tokens"]
        out[name] = rec
        print(f"[{name}/f16] streams pinned, prompt logits moved {shift:.3e} (relative) by the F16 rounding")
    with open(os.path.join(ROOT, "tests", "golden", "refbin_f16.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__" and "f16" in sys.argv[1:]:
    gen_f16()
