#!/usr/bin/env python
"""bench.py — LLaMA-7B FP32 decode tokens/sec on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): LLaMA-7B FP32, context 512, predict 128 — a 384-token
synthetic prompt is prefilled (untimed setup), then single-token decode steps are timed.
A "step" = one decoded token per in-flight sequence (N sequences at N GPUs, see DESIGN.md §multi-GPU).
  value : whole-job decode tokens/s, tokens/KV/weights resident in HBM, K CUDA-graph replays timed
          with CUDA events on the engine's stream (lb_decode_resident).  Every timed region is exactly K steps.
  e2e   : the same K steps through the public API lb_eval() with HOST buffers: token id H2D and
          128 KB logits D2H inside the timed region, one synchronous call per token.
  roofline    : dominant kernel = the decode megakernel (one launch per token): algorithmic bytes of a token
                (SURVEY §8d) / CUDA-event time per replay vs the measured HBM peak; on the per-op paths
                (Q8 weights, LB_NO_MEGA=1) the w1/w3 SwiGLU GEMV.
  cpu_baseline: the reference's own binary (--avx, all host threads) on a bounded sample.
--impl reference times the reference's own CPU implementation (oracle/_ref/llama-go-linux).
Weights (26.4 GB/token) are far larger than L2 (126 MB): no flush needed between iterations.
--dump-outputs DIR writes the logits of the last timed step of every measured decode path to DIR/<name>.npy
(float32), so that two builds run with the same arguments (same seeded inputs) can be compared output for output.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "LLaMA-7B FP32 decode tokens/sec"
MODELS = {"7b": "LLAMA_7B", "13b": "LLAMA_13B", "30b": "LLAMA_30B", "65b": "LLAMA_65B"}


def metric_name(model):
    return METRIC.replace("7B", model.upper())
UNIT = "tokens/s"
PROMPT_LEN = 384
CTX = 512


def rank_world():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)      # a measurement that raises before stop() must not leave it running
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# --------------------------------------------------------------------------------------------- reference arm
def _scratch_dir(need_bytes):
    for d in ("/dev/shm", tempfile.gettempdir()):
        try:
            if shutil.disk_usage(d).free > need_bytes * 1.2:
                return tempfile.mkdtemp(prefix="lb_ref_", dir=d)
        except Exception:
            continue
    return tempfile.mkdtemp(prefix="lb_ref_")


def _mem_available_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


REF_STREAM_PATH = os.path.join(tempfile.gettempdir(), "lb_reference_stream_7b.json")


def _ref_modules():
    """synth.py (pure Python: hyper-parameters, tensor table, ggjt writer) loaded WITHOUT the product package's
    ctypes binding, and the oracle wrapper whose liboracle.so generates the synthetic weights — the reference
    arm never maps libllamab200.so."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_lb_synth_only", os.path.join(ROOT, "llama.go_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec)
    sys.modules["_lb_synth_only"] = synth   # dataclasses looks the module up while the class is being built
    spec.loader.exec_module(synth)
    from oracle import oracle as O
    O.build()
    return synth, O


def _save_reference_stream(r, hp, prompt, predict, context):
    """Leave the binary's greedy stream on the full model where the GPU arm (run right after this one on the
    same box) can pick it up and compare it with lb_generate_greedy (BASELINE.md §4 item 5)."""
    try:
        with open(REF_STREAM_PATH, "w") as f:
            json.dump({"model": "7b", "seed": 0, "prompt": prompt, "predict": predict, "context": context,
                       "text_hex": r["text"].hex(), "when": time.time()}, f)
    except Exception as e:
        sys.stderr.write(f"[bench] could not save the reference stream: {e}\n")


def reference_cpu_decode_full(steps, warmup, threads=None):
    """The reference binary on the FULL LLaMA-7B FP32 model (26.9 GB ggjt file in a RAM-backed scratch
    dir, same synthetic weights as the GPU arm): 8-token prompt, then warmup+steps single-token decodes;
    tok/s = steps / sum(EVAL_TIME of the timed decodes).  Needs ~60 GB of host RAM; only used when the box has it."""
    synth, O = _ref_modules()
    from oracle import refbin
    threads = threads or os.cpu_count() or 1
    hp = synth.LLAMA_7B
    predict = warmup + steps + 1
    context = 8 + predict + 8
    td = _scratch_dir(28e9)
    try:
        path = os.path.join(td, "llama7b.bin")
        synth.write_ggjt(path, hp, O.synth_model(0, hp, synth.tensor_table(hp)))
        r = refbin.run(path, "abcde", predict, context, threads, True, port=18097, timeout=3000)
    finally:
        shutil.rmtree(td, ignore_errors=True)
    _save_reference_stream(r, hp, "abcde", predict, context)
    dec = r["eval_ms"][1:][warmup:warmup + steps]
    if len(dec) < max(1, steps // 2):
        raise RuntimeError("reference binary produced no timing report:\n" + r["raw"][-2000:].decode("utf-8", "replace"))
    ms = float(np.mean(dec))
    return {"tok_s": 1000.0 / ms, "ms_per_token": ms, "kind": "reference", "cores": threads,
            "sample": (f"reference binary --avx --threads {threads} on the FULL LLaMA-7B FP32 synthetic model: 8-token prompt, "
                       f"{len(dec)} single-token decodes timed after {warmup} warm-up (mean {ms:.0f} ms/token, past 8..{8 + warmup + steps})")}


def reference_cpu_decode(steps, warmup, threads=None):
    """Time the reference's own CPU path on this box's host cores.

    Bounded sample: the reference binary (--avx, all host threads) decodes `warmup+steps` tokens on
    LLaMA-7B-SHAPED models with 2 and with 4 layers (same dims/heads/ff/vocab, same synthetic
    weights as the GPU arm's seed 0); per-token time is linear in the layer count
    (t = t_head + L * t_layer, BASELINE.md §2), so the full 32-layer figure is extrapolated from the
    two measurements.  Falls back to the C oracle (kind "port") if the binary is not in oracle/_ref.
    """
    synth, O = _ref_modules()
    from oracle import refbin
    threads = threads or os.cpu_count() or 1
    dims = (32000, 4096, 256, 32)
    prompt = "abcde"                       # BOS + 2 spaces + 5 bytes = 8 tokens (>= 8 for --avx, SURVEY §8c)
    n_prompt = 8
    predict = warmup + steps + 1           # 1 prompt eval + (predict-1) single-token evals
    context = n_prompt + predict + 8
    per_token_ms = {}
    if refbin.available():
        kind = "reference"
        td = _scratch_dir(4.4e9 + 2.8e9)
        try:
            hp4 = synth.HParams(*dims, 4)
            tensors4 = list(O.synth_model(0, hp4, synth.tensor_table(hp4)))
            for L in (2, 4):
                hp = synth.HParams(*dims, L)
                names = {n for n, *_ in synth.tensor_table(hp)}
                path = os.path.join(td, f"m{L}.bin")
                synth.write_ggjt(path, hp, [(n, a) for n, a in tensors4 if n in names])
                r = refbin.run(path, prompt, predict, context, threads, True, port=18090 + L, timeout=3000)
                dec = r["eval_ms"][1:][warmup:warmup + steps]
                if len(dec) < max(1, steps // 2):
                    raise RuntimeError("reference binary produced no timing report:\n" + r["raw"][-2000:].decode("utf-8", "replace"))
                per_token_ms[L] = float(np.mean(dec))
                os.unlink(path)
        finally:
            shutil.rmtree(td, ignore_errors=True)
    else:
        kind = "port"
        O.set_dot_mode(True); O.set_threads(threads)
        for L in (2, 4):
            hp = synth.HParams(*dims, L)
            om = O.OracleModel(hp).load(O.synth_model(0, hp, synth.tensor_table(hp)))
            oc = O.OracleContext(om, context)
            oc.eval(synth.prompt_token_ids(prompt.encode()), 0)
            ts = []
            for i in range(min(warmup + steps, 12)):
                t0 = time.perf_counter(); oc.eval([5 + i], n_prompt + i); ts.append((time.perf_counter() - t0) * 1e3)
            per_token_ms[L] = float(np.mean(ts[min(warmup, len(ts) - 1):]))
        O.set_dot_mode(False)
    t_layer = (per_token_ms[4] - per_token_ms[2]) / 2.0
    t_head = per_token_ms[2] - 2.0 * t_layer
    t_full = t_head + 32.0 * t_layer
    return {
        "tok_s": 1000.0 / t_full, "ms_per_token": t_full, "kind": kind, "cores": threads,
        "sample": (f"reference binary --avx --threads {threads}: {steps} single-token decodes (after {warmup} warm-up) on "
                   f"7B-shaped 2-layer ({per_token_ms[2]:.1f} ms/token) and 4-layer ({per_token_ms[4]:.1f} ms/token) "
                   f"models, extrapolated to 32 layers as t_head + 32*t_layer ({t_head:.1f} + 32*{t_layer:.2f} ms)"),
    }


def run_reference(args):
    rank, world, _ = rank_world()
    if rank != 0:
        return
    from oracle import refbin
    full_ok = refbin.available() and _mem_available_gb() > 100 and args.steps <= 160
    r = None
    if full_ok:
        try:
            r = reference_cpu_decode_full(args.steps, args.warmup)       # measured on the whole model
        except Exception as e:
            sys.stderr.write(f"[bench] full-model reference run failed ({e}); falling back to layer slices\n")
    if r is None:
        r = reference_cpu_decode(args.steps, args.warmup)                # bounded sample, extrapolated
    line = {
        "impl": "reference", "metric": METRIC, "value": r["tok_s"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_token"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "LLaMA-7B FP32 single-sequence decode (reference CPU path, --avx)", "l2": "inputs>L2"},
        "cpu_baseline": {"value": r["tok_s"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["tok_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- our arm
DECODE_PATHS = {"ring": "persistent cooperative megakernel fed by a TMA ring (kernels_ring.cu)",
                "mega": "persistent cooperative megakernel, register-fed (kernels_mega.cu)",
                "ring_q8": "persistent cooperative Q8_0 megakernel on a TMA ring, int8 tensor cores (kernels_ring_q8.cu)",
                "perop": "per-op kernels + PDL"}
MEGA_KERNELS = {"ring": "decode_ring_kernel", "mega": "decode_mega_kernel", "ring_q8": "decode_ring_q8_kernel"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_traffic(name):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f).get(name)
    except Exception:
        return None


def compare_with_reference_stream(llama, synth, model):
    """If `--impl reference` ran on this box just before (the driver runs it first), it left the reference
    binary's greedy token stream on the FULL 7B model in REF_STREAM_PATH: generate the same stream with
    lb_generate_greedy (device sampler, same prompt ids, same temp 1e-6 / penalty 1.1) and compare the printed
    text.  The CLI can drop the final token(s) (main.go:137-147 poll race), hence prefix-with-80%-coverage."""
    try:
        with open(REF_STREAM_PATH) as f:
            rec = json.load(f)
        if time.time() - rec["when"] > 6 * 3600 or rec["model"] != "7b" or rec["seed"] != 0:
            return None
        ids = synth.prompt_token_ids(rec["prompt"].encode())
        c = llama.NewContext(model, rec["context"])
        toks = llama.GenerateGreedy(c, ids, rec["predict"])
        vocab = synth.byte_vocab(model.hp.vocab)
        exp = b"".join(vocab[i] for i in toks).strip(b"\n ")
        got = bytes.fromhex(rec["text_hex"])
        ok = len(got) > 0 and (got == exp or (exp.startswith(got) and len(got) >= 0.8 * len(exp)))
        n_match = 0
        for t in toks:
            piece = vocab[t]
            if got[:len(piece)] != piece:
                break
            got = got[len(piece):]
            n_match += 1
        return {"equal": bool(ok), "tokens_compared": n_match, "tokens_generated": len(toks),
                "what": "reference binary --avx greedy stream on the full 7B synthetic model vs lb_generate_greedy"}
    except FileNotFoundError:
        return None
    except Exception as e:
        return {"equal": None, "error": str(e)}


def measure_decode(llama, lib, hp, q8, ctx_size, K, W, sampler=None):
    """One single-GPU decode measurement: model (device RNG, seed 0) + context, prompt prefill, `value` (device
    resident, CUDA events) and `e2e` (lb_eval with host buffers).  Returns a dict that keeps model/lctx alive."""
    t_setup = time.time()
    model = llama.Model(hp, weight_type=llama.LB_TYPE_Q8_0 if q8 else llama.LB_TYPE_F32).init_random(0)
    lctx = llama.NewContext(model, ctx_size)
    rs = np.random.RandomState(0)
    prompt = rs.randint(3, hp.vocab, size=PROMPT_LEN).astype(np.uint32)
    gen = rs.randint(3, hp.vocab, size=W + K).astype(np.uint32)
    llama.Eval(lctx, prompt, 0)                         # prefill (setup, untimed; first call also sets kernel attributes)
    t_setup = time.time() - t_setup
    lib.lb_context_synchronize(lctx._h)
    t0 = time.perf_counter()
    llama.Eval(lctx, prompt, 0)                         # the same prefill again, timed: synchronous call, host buffers
    prefill_s = time.perf_counter() - t0

    # ---- value: device-resident decode, CUDA events on the engine's stream
    llama.DecodeResident(lctx, gen[:max(W, 1)], PROMPT_LEN)    # warm-up (also captures the CUDA graph)
    llama.DecodeResident(lctx, gen[:max(W, 1)], PROMPT_LEN)
    lib.lb_context_synchronize(lctx._h)
    if sampler:
        sampler.start()
    l0 = lib.lb_kernel_launches()
    ms = llama.DecodeResident(lctx, gen[W:W + K], PROMPT_LEN + W)
    lib.lb_context_synchronize(lctx._h)
    launches = lib.lb_kernel_launches() - l0
    value = K / (ms / 1e3)
    logits = llama.ReadLogits(lctx).copy()              # the last timed step's row, before e2e overwrites it

    # ---- e2e: public API, host buffers, one synchronous lb_eval per token
    for i in range(W):
        llama.Eval(lctx, gen[i:i + 1], PROMPT_LEN + i)
    lib.lb_context_synchronize(lctx._h)
    t0 = time.perf_counter()
    for i in range(K):
        llama.Eval(lctx, gen[W + i:W + i + 1], PROMPT_LEN + W + i)
    lib.lb_context_synchronize(lctx._h)
    e2e = K / (time.perf_counter() - t0)
    clocks = sampler.stop() if sampler else None
    T_mid = PROMPT_LEN + W + K / 2.0
    bytes_per_token = model.weight_bytes_per_token + 2 * hp.layers * T_mid * hp.dim * 4 + 2 * hp.layers * hp.dim * 4 + 4 * hp.vocab
    return {"model": model, "lctx": lctx, "value": value, "ms": ms, "e2e": e2e, "launches": int(launches), "clocks": clocks,
            "decode_path": DECODE_PATHS.get(lib.lb_context_decode_path(lctx._h).decode(), "?"),
            "logits": logits, "setup_s": t_setup, "bytes_per_token": int(bytes_per_token),
            "prefill": {"tokens": PROMPT_LEN, "ms": round(prefill_s * 1e3, 2), "tok_s": round(PROMPT_LEN / prefill_s, 1),
                        "what": "lb_eval of the %d-token prompt (host buffers, synchronous; tcgen05 3xTF32 GEMMs + prefill attention)" % PROMPT_LEN}}


def sub_record(r, peak, what, K, W, extra=None):
    gbs = r["bytes_per_token"] * r["value"] / 1e9
    rec = {"workload": what, "decode_path": r.get("decode_path"), "value": r["value"], "unit": UNIT, "ms_per_step": r["ms"] / K, "steps": K, "warmup": W,
           "e2e": r["e2e"], "gpu_launches": r["launches"], "clocks": r["clocks"], "prefill": r["prefill"],
           "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(gbs / peak, 4),
                        "bytes_per_step": r["bytes_per_token"], "roofline_tok_s": round(peak * 1e9 / r["bytes_per_token"], 1)}}
    if extra:
        rec.update(extra)
    return rec


def measure_pods(llama, lib, hp, B, ctx_size, K, W, sampler=None):
    """B pods of one model decoded in one pass over the weights per step (SURVEY 8f-1): aggregate tokens/s."""
    model = llama.Model(hp).init_random(0)
    rs = np.random.RandomState(0)
    pods = [llama.NewContext(model, ctx_size) for _ in range(B)]
    for c in pods:
        llama.Eval(c, rs.randint(3, hp.vocab, size=PROMPT_LEN).astype(np.uint32), 0)
    gen = rs.randint(3, hp.vocab, size=(B, 2 * W + 2 * K)).astype(np.uint32)
    batch = llama.PodBatch(pods)
    batch.DecodeResident(gen[:, :W], [PROMPT_LEN] * B)
    batch.DecodeResident(gen[:, :W], [PROMPT_LEN] * B)
    if sampler:
        sampler.start()
    l0 = lib.lb_kernel_launches()
    ms = batch.DecodeResident(gen[:, W:W + K], [PROMPT_LEN + W] * B)
    launches = lib.lb_kernel_launches() - l0
    value = B * K / (ms / 1e3)
    logits = batch.ReadLogits()                         # [B][vocab] of the last timed step, before e2e overwrites it
    for i in range(W):
        batch.Eval(gen[:, W + K + i], [PROMPT_LEN + W + K + i] * B)
    t0 = time.perf_counter()
    for i in range(K):
        batch.Eval(gen[:, 2 * W + K + i], [PROMPT_LEN + 2 * W + K + i] * B)
    e2e = B * K / (time.perf_counter() - t0)
    clocks = sampler.stop() if sampler else None
    T_mid = PROMPT_LEN + W + K / 2.0
    bytes_per_step = model.weight_bytes_per_token + B * (2 * hp.layers * T_mid * hp.dim * 4 + 2 * hp.layers * hp.dim * 4 + 4 * hp.vocab)
    mega = os.environ.get("LB_NO_MEGA_PODS") is None
    return {"value": value, "ms": ms, "e2e": e2e, "launches": int(launches), "clocks": clocks, "logits": logits,
            "bytes_per_step": int(bytes_per_step), "B": B,
            "decode_path": ("pod-batch megakernel: one persistent launch per step, B-column MulMat on mma.sync tf32 (3xTF32)" if mega
                            else "per-op kernels, B-column GEMV, CUDA-graph replay")}


def pods_record(r, peak, peak_src, what, K, W):
    gbs = r["bytes_per_step"] * (r["value"] / r["B"]) / 1e9
    return {"workload": what, "value": r["value"], "unit": UNIT, "ms_per_step": r["ms"] / K, "steps": K, "warmup": W,
            "sequences_in_flight": r["B"], "e2e": r["e2e"], "gpu_launches": r["launches"], "clocks": r["clocks"],
            "decode_path": r["decode_path"],
            "roofline": {"bound": "hbm", "kernel": "whole step", "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(gbs / peak, 4), "bytes_per_step": r["bytes_per_step"], "peak_source": peak_src,
                         "roofline_tok_s": round(r["B"] * peak * 1e9 / r["bytes_per_step"], 1),
                         "note": "bytes per step = weights once + %d x (KV read/write + logits)" % r["B"]}}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one float32 .npy per measured decode path, the logits its last timed step computed."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float32))


def release(*objs):
    import gc
    for o in objs:
        for name in ("free", "ReleaseContext"):
            f = getattr(o, name, None)
            if f:
                try:
                    f()
                except Exception:
                    pass
    gc.collect()


def run_single_gpu(args):
    import ctypes as C
    import llama_go_b200  # noqa: F401
    from llama_go_b200 import _capi, llama, synth
    _capi.require_gpu()
    lib = _capi.lib()
    hp = getattr(synth, MODELS[args.model])
    K, W = args.steps, args.warmup
    q8 = args.weights == "q8"
    ctx_size = max(args.context or (1024 if q8 else CTX), PROMPT_LEN + 2 * W + K + 1)   # config 3 (Q8) is quoted at context 1024
    sampler = ClockSampler(0)
    r = measure_decode(llama, lib, hp, q8, ctx_size, K, W, sampler)
    model, lctx, value, ms, e2e, launches, clocks = r["model"], r["lctx"], r["value"], r["ms"], r["e2e"], r["launches"], r["clocks"]
    t_setup, prefill_rec = r["setup_s"], r["prefill"]
    outputs = {"logits": r["logits"]}

    # ---- roofline of the dominant kernel + per-kernel table (live CUDA-event timing)
    peak, peak_src = measured_peak()
    if q8:
        args.no_cpu_baseline = True   # the reference has no quantised path to time
    names = {0: "gemv qkv [12288x4096]", 1: "gemv wo+res [4096x4096]", 2: "gemv_swiglu w1,w3 [2x11008x4096]",
             3: "gemv w2+res [4096x11008]", 4: "gemv lm_head [32000x4096]", 5: "attention T=%d" % (PROMPT_LEN + W + K // 2),
             6: "rmsnorm [4096]"}
    kern = {}
    for which in range(7):
        msk, by = C.c_float(0), C.c_uint64(0)
        _capi.check(lib.lb_bench_kernel(lctx._h, which, 64, PROMPT_LEN + W + K // 2, C.byref(msk), C.byref(by)))
        us = msk.value * 1e3 / 64
        kern[names[which]] = {"us": round(us, 2), "bytes": by.value, "GB/s": round(by.value / us / 1e3, 1)}
    msk, fl = C.c_float(0), C.c_uint64(0)
    _capi.check(lib.lb_bench_kernel(lctx._h, 7, 16, 0, C.byref(msk), C.byref(fl)))
    prefill_gemm = {"what": "w1 [11008x4096] x %d tokens, %s" % (min(512, ctx_size), "tcgen05 kind::tf32 3xTF32, Q8_0 dequant fused in the smem stage, TMA + TMEM" if q8 else "tcgen05 kind::tf32, 3xTF32 split, TMA + TMEM"),
                    "us": round(msk.value * 1e3 / 16, 1), "fp32_equiv_TFLOPs": round(fl.value / (msk.value / 16 * 1e-3) / 1e12, 1),
                    "tensor_TFLOPs_issued": round(3 * fl.value / (msk.value / 16 * 1e-3) / 1e12, 1)}
    dom = kern[names[2]]
    bytes_per_token = r["bytes_per_token"]
    step_gbs = bytes_per_token * value / 1e9

    path = lib.lb_context_decode_path(lctx._h).decode()
    mega = path in MEGA_KERNELS      # one persistent launch per token: the whole step is the dominant kernel
    ref_stream = compare_with_reference_stream(llama, synth, model) if (args.model == "7b" and not q8) else None

    # ---- the other single-GPU BASELINE configurations, same process, weights freed in between (VERDICT r01 #4)
    configs = None
    if args.model == "7b" and not q8 and not args.no_configs:
        configs = {}
        release(lctx, model)
        lctx = model = r = None
        try:
            rq = measure_decode(llama, lib, synth.LLAMA_7B, True, max(1024, PROMPT_LEN + 2 * W + K + 1), K, W, ClockSampler(0))
            outputs["q8_7b_ctx1024_logits"] = rq["logits"]
            configs["q8_7b_ctx1024"] = sub_record(rq, peak, "BASELINE config 3: LLaMA-7B INT8 block-quant (Q8_0) decode, context 1024, %d-token prompt" % PROMPT_LEN, K, W,
                                                  {"dtype": "q8_0 weights x f32 activations"})
            release(rq["lctx"], rq["model"])
            rq = None
        except Exception as e:
            configs["q8_7b_ctx1024"] = {"error": str(e)}
        try:
            rp = measure_pods(llama, lib, synth.LLAMA_7B, 8, max(CTX, PROMPT_LEN + 2 * W + 2 * K + 2), K, W, ClockSampler(0))
            outputs["pods8_logits"] = rp["logits"]
            configs["pods8"] = pods_record(rp, peak, peak_src, "LLaMA-7B FP32, 8 pods (independent sequences, server.go:84-106) batched per weight pass, "
                                           "context 512, %d-token prompts" % PROMPT_LEN, K, W)
            rp = None
            release()
        except Exception as e:
            configs["pods8"] = {"error": str(e)}
        try:
            r13 = measure_decode(llama, lib, synth.LLAMA_13B, False, max(CTX, PROMPT_LEN + 2 * W + K + 1), K, W, ClockSampler(0))
            outputs["llama13b_1gpu_logits"] = r13["logits"]
            configs["llama13b_1gpu"] = sub_record(r13, peak, "LLaMA-13B FP32 single-sequence decode on 1 GPU, context 512 (BASELINE config 4's model, unsharded)", K, W,
                                                  {"dtype": "f32"})
            release(r13["lctx"], r13["model"])
            r13 = None
        except Exception as e:
            configs["llama13b_1gpu"] = {"error": str(e)}

    cpu = None
    if not args.no_cpu_baseline:
        try:
            rc = reference_cpu_decode(steps=12, warmup=2)
            cpu = {"value": rc["tok_s"], "unit": UNIT, "cores": rc["cores"], "kind": rc["kind"], "sample": rc["sample"]}
        except Exception as e:  # the baseline is reported, never the target; do not lose the GPU number
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e}"}

    wbytes = bytes_per_token - (2 * hp.layers * (PROMPT_LEN + W + K / 2.0) * hp.dim * 4 + 2 * hp.layers * hp.dim * 4 + 4 * hp.vocab)
    line = {
        "metric": metric_name(args.model) if not q8 else "LLaMA-%s INT8 block-quant (Q8_0) decode tokens/sec" % args.model.upper(), "value": value, "unit": UNIT,
        "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if not q8 else "q8_0 weights x f32 activations", "data": "synthetic",
        "config": {"workload": "LLaMA-%s %s single-sequence decode, context %d, %d-token prompt prefilled, past %d..%d"
                               % (args.model.upper(), "Q8_0" if q8 else "FP32", ctx_size, PROMPT_LEN, PROMPT_LEN + W, PROMPT_LEN + W + K),
                   "weights": "random-init (device RNG, seed 0) %.1f GB" % (wbytes / 1e9), "kv_cache": "fp32 in HBM",
                   "sequences_in_flight": 1, "parallelism": "single GPU", "l2": "inputs>L2 (%.1f GB weights per step)" % (wbytes / 1e9),
                   "decode_path": DECODE_PATHS.get(path, path) + ", CUDA-graph replay",
                   "timed_regions": "1 region of exactly %d steps (CUDA events)" % K,
                   "setup_s": round(t_setup, 1)},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 4 + 8, "d2h_bytes_per_step": 4 * hp.vocab,
                "api": "lb_eval (C-ABI, host buffers, synchronous)"},
        "gpu_launches": int(launches),
        "roofline": ({"bound": "hbm", "kernel": "%s (whole token: 32 layers + lm_head in one persistent launch)" % MEGA_KERNELS.get(path, path),
                      "achieved": round(step_gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(step_gbs / peak, 4),
                      "traffic": kernel_traffic(MEGA_KERNELS.get(path, path)), "peak_source": peak_src,
                      "bytes_per_launch": int(bytes_per_token), "us_per_launch": round(ms / K * 1e3, 1),
                      "note": "algorithmic bytes of one token (SURVEY 8d: weights + KV read/write + logits) / CUDA-event time per graph replay "
                              "(memset + megakernel + 1-thread state advance)"}
                     if mega else
                     {"bound": "hbm", "kernel": ("gemv_q8 (w1,w3 SwiGLU)" if q8 else "gemv_swiglu_kernel (w1,w3)"),
                      "achieved": dom["GB/s"], "peak": peak,
                      "unit": "GB/s", "frac": round(dom["GB/s"] / peak, 4),
                      "traffic": kernel_traffic("gemv_q8_db_kernel_swiglu" if q8 else "gemv_swiglu_kernel"),
                      "peak_source": peak_src, "bytes_per_launch": dom["bytes"], "us_per_launch": dom["us"]}),
        "step_roofline": {"bytes_per_token": int(bytes_per_token), "achieved_GBs": round(step_gbs, 1),
                          "frac": round(step_gbs / peak, 4), "roofline_tok_s": round(peak * 1e9 / bytes_per_token, 1)},
        "prefill": prefill_rec,
        "per_op_kernels": kern,
        "prefill_gemm": prefill_gemm,
        "cpu_baseline": cpu,
        "reference_stream": ref_stream,
        "configs": configs,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)


def run_pods(args):
    """Extra (non-headline) measurement, SURVEY §8f-1: B pods of LLaMA-7B FP32 decoded in one pass over the weights."""
    import llama_go_b200  # noqa: F401
    from llama_go_b200 import _capi, llama, synth
    _capi.require_gpu()
    lib = _capi.lib()
    hp = getattr(synth, MODELS[args.model])
    K, W, B = args.steps, args.warmup, args.pods
    ctx_size = max(args.context or CTX, PROMPT_LEN + 2 * W + 2 * K + 2)
    r = measure_pods(llama, lib, hp, B, ctx_size, K, W, ClockSampler(0))
    peak, peak_src = measured_peak()
    rec = pods_record(r, peak, peak_src, "LLaMA-%s FP32, %d independent sequences (pods), one token each per step, context %d, %d-token prompts"
                      % (args.model.upper(), B, ctx_size, PROMPT_LEN), K, W)
    line = {"metric": "LLaMA-%s FP32 decode tokens/sec, aggregate over %d pods batched per weight pass" % (args.model.upper(), B),
            "value": rec["value"], "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": rec["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": rec["workload"], "sequences_in_flight": B, "l2": "inputs>L2", "decode_path": rec["decode_path"]},
            "clocks": rec["clocks"],
            "e2e": {"value": rec["e2e"], "unit": UNIT, "h2d_bytes_per_step": 8 * B + 8, "d2h_bytes_per_step": 4 * hp.vocab * B,
                    "api": "lb_batch_eval (host buffers, synchronous)"},
            "gpu_launches": rec["gpu_launches"], "roofline": dict(rec["roofline"], traffic=None), "cpu_baseline": None}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": r["logits"]})
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra BASELINE configurations appended to the headline line")
    ap.add_argument("--weights", default="f32", choices=["f32", "q8"], help="q8 = BASELINE config 3 (not the headline metric)")
    ap.add_argument("--model", default="7b", choices=sorted(MODELS), help="default 7b = the headline metric; 13b/65b = BASELINE configs 4-5")
    ap.add_argument("--context", type=int, default=0, help="override the context size (BASELINE config 5 uses 2048)")
    ap.add_argument("--pods", type=int, default=1, help="extra measurement: B pods (1..8) batched per weight pass on one GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the logits of the last timed step of each measured path to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world, _ = rank_world()
    if args.dump_outputs and (args.impl == "reference" or world > 1 or args.gpus > 1):
        ap.error("--dump-outputs is available for the single-GPU arms of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if world > 1 or args.gpus > 1:
        from bench_pipeline import run_pipeline   # layer-sharded multi-GPU arm
        return run_pipeline(args)
    if args.pods > 1:
        return run_pods(args)
    return run_single_gpu(args)


if __name__ == "__main__":
    main()
