"""Pod-batched generation: pkg/server.Do's loop (server.go:127-237) for up to 8 jobs at once (PodBatch.Generate,
lb_batch_generate) with the sampler on the device (PodBatch.SampleTopPTopK, lb_batch_sample).

The loop is restated here step by step in Python against four callables — a per-pod prompt eval, one batch step, one
batch sample and the context-swap rule — with the swap planning of pods.cpp: a pod whose pending token would land at
past == ctx re-evaluates the swap prefix (which ends with the pending id itself) at keep, and the next batch step then
evaluates the pending id.  CPU: driven by the oracle, it reproduces the reference binary's stream through the swaps.
GPU: driven by Eval / PodBatch.Eval / the samplers, it equals PodBatch.Generate token for token."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_case


def load_swap():
    with open(os.path.join(GOLDEN, "refbin_swap.json")) as f:
        return json.load(f)


def pods_loop(prompts, predict, ctx, keep, batch, prompt_eval, first_sample, step, batch_sample, context_swap):
    """server.Do for len(prompts) pods.  prompt_eval(b, ids, past) evaluates ids on pod b's own context;
    first_sample(rings) -> one id per pod on those contexts' last logits; step(tokens, pasts) evaluates one token per pod
    at its own position; batch_sample(rings, produced) -> one id per pod on the step's logits (seed offset = produced).
    rings = each pod's last-ctx ids, oldest first.  Returns (ids per pod, per pod the decode steps at which it swapped)."""
    B = len(prompts)
    rings = [[0] * ctx for _ in range(B)]        # container/ring of CtxSize, zero-filled (server.go:127-138)
    pasts, swaps = [0] * B, [[] for _ in range(B)]
    for b in range(B):                           # prompt phase: Context::generate until its first sample
        embd, consumed = [], 0
        while True:
            if embd:
                pasts[b], embd = context_swap(ctx, keep, rings[b], pasts[b], embd)
                prompt_eval(b, embd, pasts[b])
            pasts[b] += len(embd)
            embd = []
            if consumed == len(prompts[b]):
                break
            while consumed < len(prompts[b]) and len(embd) < batch:
                embd.append(int(prompts[b][consumed]))
                rings[b] = rings[b][1:] + [int(prompts[b][consumed])]
                consumed += 1
    out = [[int(t)] for t in first_sample(rings)]
    for b in range(B):
        rings[b] = rings[b][1:] + [out[b][0]]
    for produced in range(1, predict):           # the last sampled id is never evaluated
        for b in range(B):
            if pasts[b] == ctx:                  # server.go:165-172 with embd = [pending]
                new_past, embd = context_swap(ctx, keep, rings[b], pasts[b], [out[b][-1]])
                assert embd[-1] == out[b][-1] and (len(embd) == 1 or embd[-2] == out[b][-1])   # the prefix ends with it too
                if len(embd) > 1:
                    prompt_eval(b, embd[:-1], new_past)
                pasts[b] = new_past + len(embd) - 1
                swaps[b].append(produced)
        step([o[-1] for o in out], list(pasts))
        pasts = [p + 1 for p in pasts]
        for b, t in enumerate(batch_sample(rings, produced)):
            rings[b] = rings[b][1:] + [int(t)]
            out[b].append(int(t))
    return out, swaps


def oracle_pods(oracle, octxs, prompts, predict, ctx, keep, batch, top_k, top_p, temp, penalty, seeds):
    logits = [None] * len(octxs)

    def prompt_eval(b, ids, past):
        logits[b] = octxs[b].eval(ids, past)

    def sample(rings, produced):
        res = []
        for b, ring in enumerate(rings):
            ids, probs = oracle.sample_candidates(logits[b], ring, top_k, top_p, temp, penalty)
            res.append(oracle.sample_pick(ids, probs, seeds[b] + produced))
        return res

    def step(tokens, pasts):
        for b, (t, p) in enumerate(zip(tokens, pasts)):
            logits[b] = octxs[b].eval([t], p)

    return pods_loop(prompts, predict, ctx, keep, batch, prompt_eval, lambda rings: sample(rings, 0), step, sample,
                     oracle.context_swap)


def test_pods_loop_restatement_on_the_oracle_reproduces_the_reference_stream_through_swaps(oracle, synth):
    """3 pods on refbin_swap's prompt (30 ids, context 40, 40 generated ids: two swaps each) at temp 1e-6: every pod
    gives the oracle's (= the reference binary's) stream, although each swap is evaluated as prefix + one batch step."""
    rec = load_swap()
    hp = synth.HParams(*rec["hparams"])
    m = oracle.OracleModel(hp).load(synth.synth_model(rec["seed"], hp))
    octxs = [oracle.OracleContext(m, rec["context"]) for _ in range(3)]
    toks, swaps = oracle_pods(oracle, octxs, [rec["prompt_ids"]] * 3, rec["predict"], rec["context"], 0, rec["context"], 40, 0.95,
                              1e-6, 1.10, [3, 4, 5])
    for b in range(3):
        assert toks[b] == rec["oracle_tokens"], b
    assert [len(s) for s in swaps] == [2, 2, 2]


# ----------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def L():
    import llama_go_b200  # noqa: F401
    from llama_go_b200 import llama
    return llama


def engine_pods(L, model, ctx, prompts, predict, keep, batch, top_k, top_p, temp, penalty, seeds):
    """The restatement driven by the engine: L.Eval on its own contexts, PodBatch.Eval for the steps,
    L.SampleTopPTopK for each pod's first id and PodBatch.SampleTopPTopK afterwards."""
    from oracle import oracle as O
    ctxs = [L.NewContext(model, ctx) for _ in prompts]
    pb = L.PodBatch(ctxs)

    def first_sample(rings):
        return [L.SampleTopPTopK(ctxs[b], rings[b], top_k, top_p, temp, penalty, seeds[b])[0] for b in range(len(ctxs))]

    def batch_sample(rings, produced):
        return pb.SampleTopPTopK(np.asarray(rings, np.uint32), top_k, top_p, temp, penalty, [s + produced for s in seeds])[0]

    return pods_loop(prompts, predict, ctx, keep, batch, lambda b, ids, past: L.Eval(ctxs[b], ids, past), first_sample,
                     lambda toks, pasts: pb.Eval(toks, pasts), batch_sample, O.context_swap)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 3, 8])
def test_pods_generate_reproduces_reference_binary_through_swaps(L, synth, B):
    from oracle import refbin
    rec = load_swap()
    hp = synth.HParams(*rec["hparams"])
    model = L.Model(hp).load(synth.synth_model(rec["seed"], hp))
    pb = L.PodBatch([L.NewContext(model, rec["context"]) for _ in range(B)])
    toks = pb.Generate([rec["prompt_ids"]] * B, rec["predict"], 40, 0.95, 1e-6, 1.10, 0, rec["context"], seeds=list(range(3, 3 + B)))
    vocab = synth.byte_vocab(hp.vocab)
    for b in range(B):
        assert toks[b] == rec["oracle_tokens"], b
        for mode in ("scalar", "avx"):
            assert refbin.same_stream(bytes.fromhex(rec["runs"][mode]["text_hex"]), refbin.expected_text(vocab, rec["prompt_ids"], toks[b]))


def _staggered(L, model, ctx, prompts, predict, keep, seeds):
    B = len(prompts)
    pb = L.PodBatch([L.NewContext(model, ctx) for _ in range(B)])
    got = pb.Generate(prompts, predict, 40, 0.95, 0.8, 1.10, keep, None, seeds=seeds)
    want, swaps = engine_pods(L, model, ctx, prompts, predict, keep, ctx, 40, 0.95, 0.8, 1.10, seeds)
    assert min(len(s) for s in swaps) >= 2 and len({s[0] for s in swaps}) == B   # every pod swaps, each at its own step
    for b in range(B):
        first = next((i for i, (x, y) in enumerate(zip(got[b], want[b])) if x != y), None)
        assert first is None, f"pod {b}: streams part at id {first} of {predict} (swaps at {swaps[b]})"
    assert len({tuple(t) for t in got}) == B          # different prompts and seeds: different streams
    return swaps


@pytest.mark.gpu
def test_pods_generate_equals_the_step_restatement_7b_shaped_ring_pods(L, synth):
    """LLaMA-7B layer shapes (2 layers, vocab 2048), context 512, 8 pods with prompts of 400 + 3b ids: the pod step is
    the TMA-ring pods megakernel.  Temp 0.8, top-k 40, top-p 0.95, keep 24, per-pod seeds; every pod swaps twice, at
    steps that differ between pods."""
    hp = synth.HParams(2048, 4096, 256, 32, 2)
    model = L.Model(hp).init_random(0)
    rs = np.random.RandomState(5)
    prompts = [rs.randint(3, hp.vocab, size=400 + 3 * b).tolist() for b in range(8)]
    swaps = _staggered(L, model, 512, prompts, 380, 24, [1000 + 17 * b for b in range(8)])
    print(f"[7B-shaped pods generate] swap steps per pod {swaps}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tiny", "hd128"])
@pytest.mark.parametrize("wt", ["f16", "q8_0"])
def test_pods_generate_equals_the_step_restatement_perop_f16_q8(L, synth, case, wt):
    """The golden models with F16 and Q8_0 weights (the per-op B-column pod kernels), context 64, 5 pods with prompts of
    20 + 3b ids, keep 4: every pod swaps at least twice."""
    rec, g = load_case(case)
    hp = synth.HParams(*rec["hparams"])
    model = L.Model(hp, weight_type=L.LB_TYPE_F16 if wt == "f16" else L.LB_TYPE_Q8_0).load(synth.synth_model(rec["seed"], hp))
    base = [int(t) for t in g["prompt_ids"]] + [int(t) for t in g["gen_ids"]]
    prompts = [base[b:b + 20 + 3 * b] for b in range(5)]
    _staggered(L, model, 64, prompts, 110, 4, [7 * b + 1 for b in range(5)])


@pytest.mark.gpu
@pytest.mark.parametrize("top_k,top_p,temp,penalty", [(40, 0.95, 0.8, 1.1), (1, 0.95, 0.8, 1.1), (200, 0.5, 1.3, 1.0),
                                                      (40, 0.95, 1e-6, 1.1), (512, 0.999, 2.0, 1.3)])
def test_batched_sampler_candidate_sets_match_oracle(L, oracle, synth, top_k, top_p, temp, penalty):
    rec = load_swap()
    hp = synth.HParams(*rec["hparams"])
    model = L.Model(hp).load(synth.synth_model(rec["seed"], hp))
    ids = rec["prompt_ids"]
    pods = [L.NewContext(model, 64) for _ in range(8)]
    for c in pods:
        L.Eval(c, ids, 0)
    pb = L.PodBatch(pods)
    logits = pb.Eval([ids[b] for b in range(8)], [len(ids)] * 8)
    rs = np.random.RandomState(2)
    rings = np.asarray([[0] * (10 + b) + rs.randint(0, hp.vocab, size=54 - b).tolist() for b in range(8)], np.uint32)
    for seed in (0, 12345):
        seeds = [seed + 101 * b for b in range(8)]
        toks, cids, cprobs = pb.SampleTopPTopK(rings, top_k, top_p, temp, penalty, seeds)
        for b in range(8):
            rids, rprobs = oracle.sample_candidates(logits[b], rings[b], top_k, top_p, temp, penalty)
            np.testing.assert_array_equal(cids[b], rids)                        # index work: exact
            np.testing.assert_allclose(cprobs[b], rprobs, rtol=3e-7, atol=0)    # f64 exp of two libms, then identical FP32 steps
            assert toks[b] == oracle.sample_pick(rids, rprobs, seeds[b]) or not np.array_equal(cprobs[b], rprobs)
            assert toks[b] in cids[b].tolist()


@pytest.mark.gpu
def test_pods_generate_refusals_leave_the_batch_usable_and_repeat_exactly(L, synth):
    rec, g = load_case("tiny")
    hp = synth.HParams(*rec["hparams"])
    ctx = rec["context"]
    model = L.Model(hp).load(synth.synth_model(rec["seed"], hp))
    ids = [int(t) for t in g["prompt_ids"]]
    gen = [int(t) for t in g["gen_ids"]]
    pods = [L.NewContext(model, ctx) for _ in range(4)]
    for c in pods:
        L.Eval(c, ids, 0)
    pb = L.PodBatch(pods)
    good = [ids] * 4
    bad_calls = [
        dict(prompts=[ids, ids, [], ids]),                            # an empty prompt
        dict(prompts=[ids, ids + [hp.vocab], ids, ids]),              # an id out of range
        dict(topK=0), dict(topK=hp.vocab + 1),                        # top_k outside 1..vocab
        dict(temp=0.0), dict(temp=-1.0),
        dict(keepCount=ctx), dict(keepCount=ctx + 5),                 # keep_count >= ctx_size
        dict(batchSize=0),
    ]
    for kw in bad_calls:
        args = dict(prompts=good, predict=8)
        args.update(kw)
        with pytest.raises(L.LlamaB200Error):
            pb.Generate(args.pop("prompts"), args.pop("predict"), **args)
    with pytest.raises(ValueError):
        pb.Generate([ids] * 3, 8)                                      # lengths do not match the pods
    with pytest.raises(ValueError):
        pb.Generate(good, 8, seeds=[1, 2])
    # nothing ran: the pods' caches still hold the prompt, the batch step gives the golden logits
    got = pb.Eval([gen[0]] * 4, [len(ids)] * 4)
    ref = g["step_logits"][1]
    for row in got:
        assert np.abs(row - ref).max() <= 1e-3 * np.abs(ref).max()
    a = pb.Generate([ids, ids[:10], ids[5:], ids], 50, seeds=[9, 8, 7, 9])
    b = pb.Generate([ids, ids[:10], ids[5:], ids], 50, seeds=[9, 8, 7, 9])
    assert a == b and all(len(t) == 50 for t in a)
    assert a[0] == a[3]                                               # same prompt and seed: same stream
    c = pb.Generate([ids, ids[:10], ids[5:], ids], 50, seeds=[9, 8, 7, 5])
    assert c[:3] == a[:3] and c[3] != a[3]                            # another seed changes that pod only
