#!/usr/bin/env python
"""Pod-batched generation (lb_batch_generate) on one B200: LLaMA-7B FP32 (init_random), 8 pods at context 512.  Prints one
JSON line.

  * workload i:  128-token prompts, predict 256 — no context swap;
  * workload ii: 384-token prompts, predict 512 — every pod swaps (keep 0) twice.

For each: the aggregate generated tok/s over the decode phase (8 x predict ids over lb_batch_generate's decode_ms_out,
CUDA events from the first batched sample to the last, swaps included), and teacher-forced lb_batch_decode_resident
tok/s on the same pods over the same positions (8 x steps over its CUDA-event time; workload ii runs it as the three
windows the generate loop's swaps leave: 384 +128, 256 +256, 256 +127) — the upper bound — and their ratio.  Runs
alternate generate / resident; each figure is the median over --reps.  Then one solo lb_generate on one context of
the same model, the path without pods: (predict - 1) / (wall(predict) - wall(1)), host clock around synchronous calls.

Usage: python bench_pods_generate.py [--reps 3] [--out DIR]
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

B, CTX = 8, 512
SAMPLING = dict(topK=40, topP=0.95, temp=0.8, repeatPenalty=1.10)


def smi(query):
    out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader,nounits", "-i", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, check=True).stdout
    return [v.strip() for v in out.strip().splitlines()[0].split(",")]


def resident_windows(n_prompt, predict, keep=0):
    """(past, steps) windows of the pod steps the generate loop runs: a window ends where the pending id would land at
    the context's end, and the swap restarts it at keep + (ctx - keep) // 2."""
    wins, past, left = [], n_prompt, predict - 1
    while left:
        if past == CTX:
            past = keep + (CTX - keep) // 2
        n = min(left, CTX - past)
        wins.append((past, n))
        past += n
        left -= n
    return wins


def workload(pb, rs, vocab, n_prompt, predict, reps):
    prompts = [rs.randint(3, vocab, size=n_prompt).tolist() for _ in range(B)]
    seeds = [1 + b for b in range(B)]
    wins = resident_windows(n_prompt, predict)
    pb.Generate(prompts, predict, seeds=seeds, **SAMPLING)   # warm-up: graph capture, sampler attributes
    gen_ms, res_ms, streams = [], [], None
    for _ in range(reps):
        streams, ms = pb.Generate(prompts, predict, seeds=seeds, return_ms=True, **SAMPLING)
        gen_ms.append(ms)
        t = 0.0
        for past, n in wins:
            toks = rs.randint(3, vocab, size=(B, n)).astype(np.uint32)
            t += pb.DecodeResident(toks, [past] * B)
        res_ms.append(t)
    steps = sum(n for _, n in wins)
    g, r = float(np.median(gen_ms)), float(np.median(res_ms))
    gen_tps, res_tps = B * predict / (g / 1e3), B * steps / (r / 1e3)
    assert all(len(s) == predict and max(s) < vocab for s in streams)
    return dict(prompt=n_prompt, predict=predict, swaps_per_pod=len(wins) - 1, decode_ms=round(g, 2),
                generated_tok_s=round(gen_tps, 1), resident_windows=wins, resident_ms=round(r, 2), resident_tok_s=round(res_tps, 1),
                ratio=round(gen_tps / res_tps, 4), gen_ms_all=[round(x, 2) for x in gen_ms], resident_ms_all=[round(x, 2) for x in res_ms],
                distinct_streams=len({tuple(s) for s in streams}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _capi.require_gpu()
    name, power_limit = smi("name,power.limit")
    hp = synth.LLAMA_7B
    model = llama.Model(hp).init_random(0)
    pods = [llama.NewContext(model, CTX) for _ in range(B)]
    pb = llama.PodBatch(pods)
    rs = np.random.RandomState(0)
    res = dict(metric="pods_generate", model="LLaMA-7B FP32 (init_random)", pods=B, context=CTX, sampling=SAMPLING,
               gpu=name, power_limit_w=power_limit)
    res["i"] = workload(pb, rs, hp.vocab, 128, 256, args.reps)
    res["ii"] = workload(pb, rs, hp.vocab, 384, 512, args.reps)

    solo = llama.NewContext(model, CTX)
    prompt = rs.randint(3, hp.vocab, size=128).tolist()
    llama.Generate(solo, prompt, 8, seed=1, **SAMPLING)   # warm-up
    walls = {}
    for predict in (1, 256):
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            llama.Generate(solo, prompt, predict, seed=1, **SAMPLING)
            ts.append(time.perf_counter() - t0)
        walls[predict] = float(np.median(ts))
    solo_tps = 255 / (walls[256] - walls[1])
    res["solo_lb_generate"] = dict(prompt=128, predict=256, tok_s=round(solo_tps, 1))
    res["i"]["vs_solo"] = round(res["i"]["generated_tok_s"] / solo_tps, 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_pods_generate.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
