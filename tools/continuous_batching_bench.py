"""Continuous batching (serve()) against lockstep generate() over consecutive groups of B, for both batched decoders, on
the tiny random-init fp16 Llama of tools/batched_sam_only_bench.py: B = 64 slots, max_cache_len 2048, N = 512 seeded
requests (copy_mix prompts of 64-1024 tokens, max_new_tokens log-uniform in [16, 512]).

Per arm: wall seconds of one pass (host clock, ending in a device synchronise; every graph was captured by an untimed
warm-up pass of the same arm), requests/s, output tokens/s, decode steps, host syncs and live slot-steps / (B x steps).
The lockstep arm runs each group to its longest limit and keeps every request's first `limit` tokens; its live
slot-steps are those before a request reached its own limit.  Before the timed passes, both arms run with the same
weights in fp32 and their outputs must be equal.  In fp16 the two arms batch the prompts differently (prefill
sub-batches vs groups, other key-length buckets), so logits can differ in the last bits; every fp16 request whose
outputs differ is reported with the position where they part and the fp16 / fp32 top-2 logits of a plain forward over
the common prefix there.  A separate instrumented serve() pass splits the admission cost with CUDA events around its
three parts: the sub-batch LM prefill, the drafters' masked reset + prompt ingestion, and the slot state.
    python tools/continuous_batching_bench.py [--out profiles/r04_continuous_batching.json]
(GPU box, from the repo root; prints one JSON line and writes it to --out)"""
import argparse
import copy
import json
import math
import os
import sys
import time

sys.path.insert(0, "sam-decoding_b200")
import numpy as np
import torch
from transformers import LlamaConfig, LlamaForCausalLM
from samd_b200 import engine as E, synth
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
from batched_sam_only_bench import gpu_info

B, MAX_LEN, N, T_SO = 64, 2048, 512, 40


def workload():
    rng = np.random.default_rng(2024)
    lens = rng.integers(64, 1025, size=N)
    limits = np.exp(rng.uniform(math.log(16), math.log(512), size=N)).round().astype(int).tolist()
    prompts = [synth.copy_mix(int(n), 96, 40000 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    return prompts, limits


def r03_corpus(lm, dtype):
    """The static corpus of tools/batched_sam_only_bench.py: 64-token pieces of the LM's greedy continuations of that
    bench's prompts, and unrelated copy_mix documents."""
    prompts = [synth.copy_mix(192 + (i % 5) * 16, 96, 900 + i, p_copy=0.7).tolist() for i in range(B)]
    cont, _ = BatchedSamOnlyDecoder(lm, B, MAX_LEN, max_predicts=T_SO, alpha=4.0, dtype=dtype).generate(prompts, 128)
    docs = [c[i % 16:i % 16 + 64] for i, c in enumerate(cont)] + [synth.copy_mix(2000, 96, 5000 + k, p_copy=0.7).tolist()
                                                                  for k in range(8)]
    return E.StaticSamDevice.build(docs, synth.EOS, with_counts=True), sum(map(len, docs))


def run_serve(dec, prompts, limits):
    out = {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i, tokens, _ in dec.serve(prompts, limits):
        out[i] = tokens
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    st = dec.serve_stats
    return [out[i] for i in range(len(prompts))], dt, st["steps_run"], st["host_syncs"], st["live_slot_steps"]


def run_lockstep(dec, prompts, limits):
    out, steps, syncs, live = [], 0, 0, 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for g in range(0, len(prompts), B):
        lim = limits[g:g + B]
        toks, st = dec.generate(prompts[g:g + B], max(lim))
        out += [t[:l] for t, l in zip(toks, lim)]
        steps, syncs = steps + st["steps_run"], syncs + st["host_syncs"]
        for acc, l in zip(st["accept_lengths"], lim):        # steps until the request had its own `limit` tokens
            live += int(np.searchsorted(np.cumsum(acc), l) + 1)
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0, steps, syncs, live


def admission_split(dec, prompts, limits):
    """One serve() pass with CUDA events around the three parts of every admission."""
    parts = ("_prefill_slots", "_ingest", "_set_slots")
    ev = {p: [] for p in parts}
    longest = []

    def timed(name, fn):
        def call(*a):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a)
            e.record()
            ev[name].append((s, e))
            if name == "_prefill_slots":
                longest.append(a[0].shape[1])
            return r
        return call

    for p in parts:
        setattr(dec, p, timed(p, getattr(dec, p)))
    try:
        for _ in dec.serve(prompts, limits):
            pass
        torch.cuda.synchronize()
    finally:
        for p in parts:
            delattr(dec, p)
    ms = {p: np.array([s.elapsed_time(e) for s, e in ev[p]]) for p in parts}
    ing, lg = ms["_ingest"], np.array(longest, dtype=np.float64)
    slope, icept = np.polyfit(lg, ing * 1e3, 1) if len(lg) > 1 else (float("nan"), float("nan"))
    names = {"_prefill_slots": "lm_prefill", "_ingest": "reset_and_ingest", "_set_slots": "slot_state"}
    return {"admission_calls": len(lg), "requests": dec.serve_stats["admissions"],
            **{names[p]: {"total_ms": float(v.sum()), "mean_ms": float(v.mean()), "max_ms": float(v.max())}
               for p, v in ms.items()},
            "reset_and_ingest_vs_longest_prompt": {"us_per_token": float(slope), "us_at_0": float(icept),
                                                   "note": "least-squares line of each call's reset + ingestion time "
                                                           "against the longest prompt it admitted"}}


@torch.inference_mode()
def divergence(lm, lm32, prompt, a, b):
    """Where two outputs of one prompt part: the position, each arm's token, and the top-2 logits of a plain forward over
    the common prefix in fp16 and with the same weights in fp32."""
    d = next((k for k, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
    ids = torch.as_tensor([prompt + a[:d]]).cuda()
    top = {}
    for tag, m in (("fp16", lm), ("fp32", lm32)):
        v, t = m(input_ids=ids).logits[0, -1].float().topk(2)
        top[tag] = {"top2": t.tolist(), "margin": float(v[0] - v[1])}
    return {"position": d, "serve": a[d] if d < len(a) else None, "lockstep": b[d] if d < len(b) else None, **top}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_continuous_batching.json")
    args = ap.parse_args()
    name, power = gpu_info()
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=4, max_position_embeddings=4096)
    dtype = torch.float16
    lm = LlamaForCausalLM(cfg).cuda().to(dtype).eval()
    prompts, limits = workload()
    static, corpus_tokens = r03_corpus(lm, dtype)
    decoders = {
        "samd": lambda: BatchedSamdDecoder(lm, B, MAX_LEN, n_predicts=8, len_bias=5, len_threshold=3, dtype=dtype),
        "sam_only": lambda: BatchedSamOnlyDecoder(lm, B, MAX_LEN, max_predicts=T_SO, alpha=4.0, K=8, len_bias=5,
                                                  static=static, dtype=dtype),
    }
    lm32 = copy.deepcopy(lm).float()                          # the same weights in fp32: the exact output check
    decoders32 = {
        "samd": lambda: BatchedSamdDecoder(lm32, B, MAX_LEN, n_predicts=8, len_bias=5, len_threshold=3, dtype=torch.float32),
        "sam_only": lambda: BatchedSamOnlyDecoder(lm32, B, MAX_LEN, max_predicts=T_SO, alpha=4.0, K=8, len_bias=5,
                                                  static=static, dtype=torch.float32),
    }
    n_out = sum(limits)
    res = {}
    for flavour, make in decoders.items():
        dec32 = decoders32[flavour]()
        outs32 = [fn(dec32, prompts, limits)[0] for fn in (run_serve, run_lockstep)]
        diff32 = [i for i, (a, b) in enumerate(zip(*outs32)) if a != b]
        assert not diff32, f"{flavour}: fp32 serve and lockstep outputs differ for requests {diff32[:16]}"
        del dec32
        dec = make()
        arms = {}
        for arm, fn in (("serve", run_serve), ("lockstep", run_lockstep)):
            fn(dec, prompts, limits)                          # warm-up: graph capture for every bucket the arm reaches
            arms[arm] = fn(dec, prompts, limits)
        diff = [i for i, (a, b) in enumerate(zip(arms["serve"][0], arms["lockstep"][0])) if a != b]
        r = {"outputs_equal_fp32": True, "fp16_requests_equal": N - len(diff),
             "fp16_divergences": {str(i): divergence(lm, lm32, prompts[i], arms["serve"][0][i], arms["lockstep"][0][i])
                                  for i in diff}}
        for arm, (out, dt, steps, syncs, live) in arms.items():
            r[arm] = {"seconds": dt, "requests_per_s": N / dt, "output_tokens": sum(map(len, out)),
                      "output_tokens_per_s": sum(map(len, out)) / dt, "steps": steps, "host_syncs": syncs,
                      "live_slot_steps": live, "utilisation": live / (B * steps)}
        r["speedup"] = r["lockstep"]["seconds"] / r["serve"]["seconds"]
        r["admission"] = admission_split(dec, prompts, limits)
        r["admission"]["share_of_serve_seconds"] = sum(r["admission"][k]["total_ms"] for k in
                                                       ("lm_prefill", "reset_and_ingest", "slot_state")) / 1e3 / r["serve"]["seconds"]
        res[flavour] = r
        del dec
    line = json.dumps({
        "gpu": name, "power_limit": power,
        "workload": f"B={B} slots, max_cache_len {MAX_LEN}, N={N} requests: copy_mix prompts of 64-1024 tokens (V=96, "
                    f"p_copy 0.7), max_new_tokens log-uniform in [16, 512] ({n_out} tokens in all), seeded; tiny Llama "
                    "(2 layers, d=128, V=96) fp16; samd: sequence mode, n_predicts 8, len_bias 5, len_threshold 3; "
                    f"sam_only: max_predicts {T_SO}, alpha 4, K 8, len_bias 5, the r03 static corpus ({corpus_tokens} "
                    "tokens, with counts)",
        "method": "serve() over all N requests vs generate() over consecutive groups of B (each group to its longest "
                  "limit, outputs cut to each request's limit); one untimed warm-up pass per arm, then one timed pass "
                  "(host clock ending in a device synchronise); outputs compared first: exactly, with the same weights "
                  "in fp32, and request by request in fp16 (fp16_divergences: where they part, top-2 logits of a plain "
                  "forward there); admission split from a separate "
                  "serve() pass with CUDA events around each part (device time from its first to its last launch, host "
                  "launch gaps included)",
        **res})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
