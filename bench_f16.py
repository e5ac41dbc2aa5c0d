#!/usr/bin/env python
"""F16 weights (LB_TYPE_F16) against FP32 on one B200: decode, prefill, and a 65B model on one GPU.  Prints one JSON line.

  * decode, LLaMA-7B at context 512: an FP32 model and an F16 model of the same seed, the FP32 one holding the F16
    weights widened back (per-tensor lb_model_get_tensor -> lb_model_set_tensor), so both compute the same function.
    Both get the same 384-token prompt through the decode path, then teacher-forced DecodeResident windows alternate
    FP32 / F16 / FP32 / F16.  Reported: tok/s of each, the F16 window's share of the HBM roofline (weight bytes + KV
    bytes per token over MEASURED_PEAKS.json hbm_gbs, or the named fallback), and the largest logit difference between
    the two models after the last window (the decode ring computes bit-identical logits: expected 0).
  * prefill of the same 384 tokens (lb_eval, synchronous): FP32 vs F16, alternating, median of the repeats.
  * LLaMA-65B, F16, context 2048 on one GPU: decode tok/s at T ~ 1024 and the device memory in use.

Usage: python bench_f16.py [--steps 120] [--warmup 8] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import llama_go_b200  # noqa: E402,F401
from llama_go_b200 import _capi, llama, synth  # noqa: E402

PROMPT_LEN = 384


def smi(query):
    out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader,nounits", "-i", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, check=True).stdout
    return [v.strip() for v in out.strip().splitlines()[0].split(",")]


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback: 6.65 TB/s, not measured on this card"


def kv_bytes(hp, T):
    return 2 * hp.layers * T * hp.dim * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=120)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    K, W = args.steps, args.warmup
    assert PROMPT_LEN + W + K <= 512, "a decode window must fit context 512"
    _capi.require_gpu()
    lib = _capi.lib()
    name, power_limit, max_sm = smi("name,power.limit,clocks.max.sm")
    peak, peak_src = measured_peak()
    hp = synth.LLAMA_7B
    rs = np.random.RandomState(0)
    prompt = rs.randint(3, hp.vocab, size=PROMPT_LEN).astype(np.uint32)
    gen = rs.randint(3, hp.vocab, size=W + K).astype(np.uint32)

    # ---- models: F16 of seed 0, and FP32 holding the same weights widened
    m16 = llama.Model(hp, weight_type=llama.LB_TYPE_F16).init_random(0)
    m32 = llama.Model(hp).init_random(0)
    for tname, _tid, shape, _m, _s in synth.tensor_table(hp):
        if synth.is_q8_matrix(tname):
            m32.set_tensor(tname, m16.get_tensor(tname, shape))
    ctx = {"f32": llama.NewContext(m32, 512), "f16": llama.NewContext(m16, 512)}
    paths = {k: lib.lb_context_decode_path(c._h).decode() for k, c in ctx.items()}

    # ---- decode: the prompt through the decode path on both, then alternating windows at T ~ 400; every window
    #      decodes the same tokens at the same positions (teacher-forced, the KV rows are rewritten with the same values)
    for c in ctx.values():
        llama.DecodeResident(c, prompt, 0)
    rates = {"f32": [], "f16": []}
    for k in ("f32", "f16", "f32", "f16"):
        llama.DecodeResident(ctx[k], gen[:W], PROMPT_LEN)
        ms = llama.DecodeResident(ctx[k], gen[W:], PROMPT_LEN + W)
        rates[k].append(K / (ms / 1e3))
    lg32, lg16 = llama.ReadLogits(ctx["f32"]).copy(), llama.ReadLogits(ctx["f16"]).copy()
    max_diff = float(np.abs(lg32 - lg16).max())
    T_mid = PROMPT_LEN + W + K / 2.0
    bytes16 = m16.weight_bytes_per_token + kv_bytes(hp, T_mid)
    bytes32 = m32.weight_bytes_per_token + kv_bytes(hp, T_mid)
    tok16, tok32 = max(rates["f16"]), max(rates["f32"])
    decode = {
        "model": "LLaMA-7B synthetic (seed 0), context 512, teacher-forced DecodeResident windows of %d steps after %d warm-up, T %d..%d"
                 % (K, W, PROMPT_LEN + W, PROMPT_LEN + W + K),
        "f32_tok_s": [round(r, 1) for r in rates["f32"]], "f16_tok_s": [round(r, 1) for r in rates["f16"]],
        "f16_over_f32": round(tok16 / tok32, 3), "decode_path": paths,
        "f16_bytes_per_token": int(bytes16), "f32_bytes_per_token": int(bytes32),
        "f16_roofline": {"peak_gbs": peak, "peak_source": peak_src, "achieved_gbs": round(bytes16 * tok16 / 1e9, 1),
                         "frac": round(bytes16 * tok16 / 1e9 / peak, 4), "roofline_tok_s": round(peak * 1e9 / bytes16, 1)},
        "max_abs_logit_diff_f16_vs_widened_f32": max_diff,
    }

    # ---- prefill: 384 tokens, synchronous lb_eval (tcgen05 GEMMs), alternating
    pf = {"f32": [], "f16": []}
    pctx = {"f32": llama.NewContext(m32, 512), "f16": llama.NewContext(m16, 512)}
    for k in ("f32", "f16"):
        llama.Eval(pctx[k], prompt, 0)                  # warm-up (kernel attributes, tensor maps)
    for _ in range(5):
        for k in ("f32", "f16"):
            lib.lb_context_synchronize(pctx[k]._h)
            t0 = time.perf_counter()
            llama.Eval(pctx[k], prompt, 0)
            pf[k].append((time.perf_counter() - t0) * 1e3)
    prefill = {"tokens": PROMPT_LEN, "f32_ms": round(float(np.median(pf["f32"])), 2), "f16_ms": round(float(np.median(pf["f16"])), 2),
               "f32_ms_all": [round(v, 2) for v in pf["f32"]], "f16_ms_all": [round(v, 2) for v in pf["f16"]]}
    prefill["f16_over_f32_speed"] = round(prefill["f32_ms"] / prefill["f16_ms"], 3)
    for c in list(ctx.values()) + list(pctx.values()):
        c.ReleaseContext()
    m16.free(); m32.free()

    # ---- 65B F16 on one GPU, context 2048, decode at T ~ 1024
    hp65 = synth.LLAMA_65B
    t0 = time.time()
    m65 = llama.Model(hp65, weight_type=llama.LB_TYPE_F16).init_random(0)
    c65 = llama.NewContext(m65, 2048)
    p65 = rs.randint(3, hp65.vocab, size=1000).astype(np.uint32)
    g65 = rs.randint(3, hp65.vocab, size=8 + 48).astype(np.uint32)
    llama.Eval(c65, p65, 0)
    setup_s = time.time() - t0
    llama.DecodeResident(c65, g65[:8], 1000)
    ms65 = llama.DecodeResident(c65, g65[8:], 1008)
    lg65 = llama.ReadLogits(c65)
    mem_used, mem_total = smi("memory.used,memory.total")
    tok65 = 48 / (ms65 / 1e3)
    b65 = m65.weight_bytes_per_token + kv_bytes(hp65, 1032)
    big = {"model": "LLaMA-65B synthetic (seed 0), F16, context 2048, 1000-token prompt, 48 decode steps at T 1008..1056",
           "decode_path": lib.lb_context_decode_path(c65._h).decode(), "tok_s": round(tok65, 2),
           "weight_bytes_per_token": int(m65.weight_bytes_per_token), "roofline_frac": round(b65 * tok65 / 1e9 / peak, 4),
           "device_memory_used_mib": int(mem_used), "device_memory_total_mib": int(mem_total),
           "logits_finite": bool(np.isfinite(lg65).all()), "setup_s": round(setup_s, 1)}
    c65.ReleaseContext(); m65.free()

    rec = {"bench": "f16_weights", "gpu": name, "power_limit_w": float(power_limit), "max_sm_clock_mhz": int(max_sm),
           "decode_7b": decode, "prefill_7b": prefill, "llama_65b_f16_one_gpu": big,
           "targets": {"f16_decode_ge_1p7x_f32": tok16 >= 1.7 * tok32, "f16_prefill_no_slower": prefill["f16_ms"] <= prefill["f32_ms"] * 1.02,
                       "65b_f16_runs_on_one_gpu": big["logits_finite"]}}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_f16.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
