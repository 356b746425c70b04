"""Prefix reuse (max_prefixes, add_prefix) in serve(): the same requests served without a pool and with their shared heads
registered, for both batched decoders, on the tiny random-init fp16 Llama of tools/continuous_batching_bench.py: B = 64
slots, max_cache_len 2048, N = 512 seeded requests.  Each request is one of 8 heads of 512-1536 tokens plus a 32-256 token
suffix, except about 10 % that have a head of the same length that is not registered; max_new_tokens log-uniform in
[16, 512], cut so that prompt + limit + one step fits the cache.  Serving traffic with a shared system prompt, few-shot
block or document looks like this; how much of admission a pool removes depends on the share of the prompt the head is.

Per arm: wall seconds of one pass (host clock, ending in a device synchronise, after an untimed warm-up pass that captured
every graph), requests/s, decode steps, and a separate instrumented pass that splits the admission cost with CUDA events
around each of its parts (KV copy, drafter reset / clone, LM prefill, ingestion, slot state).  Before the timed passes
the two arms run with the same weights in fp32 and must give identical outputs; in fp16 the arms batch different rows
into the LM (whole prompts vs suffixes over copied rows), so near-ties can round differently: every fp16 divergence is
reported with the fp16 / fp32 top-2 logits of a plain forward where the outputs part.

Kernel lines: samd_kv_copy_rows on a Llama-7B-shaped KV (32 layers x K and V, 32 heads, dh 128, fp16; 16 pairs x 1024
rows) in bytes/s against a device-to-device copy of the same bytes, and samd_dyn_clone per request at max_tokens 16384
against samd_dyn_reset + ingestion of the same 1024-token prefix.
    python tools/prefix_cache_bench.py [--out profiles/r05_prefix_cache.json]
(GPU box, from the repo root; prints one JSON line and writes it to --out)"""
import argparse
import copy
import json
import math
import os
import sys
import time

sys.path.insert(0, "sam-decoding_b200")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch
from transformers import LlamaConfig, LlamaForCausalLM
from samd_b200 import _cabi as K, engine as E, synth
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
from batched_sam_only_bench import gpu_info
from continuous_batching_bench import divergence, r03_corpus

B, MAX_LEN, N, T_SO, N_HEADS = 64, 2048, 512, 40, 8


def workload():
    rng = np.random.default_rng(2025)
    heads = [synth.copy_mix(int(rng.integers(512, 1537)), 96, 60000 + k, p_copy=0.7).tolist() for k in range(N_HEADS)]
    prompts, registered = [], 0
    for i in range(N):
        k = int(rng.integers(N_HEADS))
        suffix = synth.copy_mix(int(rng.integers(32, 257)), 96, 70000 + i, p_copy=0.7).tolist()
        if rng.random() < 0.1:                                 # a head nobody registered, of the same length
            head = synth.copy_mix(len(heads[k]), 96, 80000 + i, p_copy=0.7).tolist()
        else:
            head, registered = heads[k], registered + 1
        prompts.append(head + suffix)
    limits = np.exp(rng.uniform(math.log(16), math.log(512), size=N)).round().astype(int)
    limits = [int(min(l, MAX_LEN - len(p) - T_SO - 1)) for l, p in zip(limits, prompts)]
    return heads, prompts, limits, registered


def run_serve(dec, prompts, limits):
    out = {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i, tokens, _ in dec.serve(prompts, limits):
        out[i] = tokens
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return [out[i] for i in range(len(prompts))], dt, dict(dec.serve_stats)


PARTS = {"_copy_prefix_kv": "kv_copy", "_clone_drafters": "reset_and_clone", "_prefill_slots": "lm_prefill",
         "_ingest": "reset_and_ingest", "_ingest_suffixes": "ingest", "_set_slots": "slot_state"}


def admission_split(dec, prompts, limits):
    """One serve() pass with CUDA events around every admission part (device time from its first to its last launch,
    host launch gaps included)."""
    ev = {p: [] for p in PARTS}

    def timed(name, fn):
        def call(*a, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **kw)
            e.record()
            ev[name].append((s, e))
            return r
        return call

    for p in PARTS:
        setattr(dec, p, timed(p, getattr(dec, p)))
    try:
        for _ in dec.serve(prompts, limits):
            pass
        torch.cuda.synchronize()
    finally:
        for p in PARTS:
            delattr(dec, p)
    return {PARTS[p]: {"calls": len(v), "total_ms": float(sum(s.elapsed_time(e) for s, e in v))} for p, v in ev.items() if v}


def time_events(fn, reps):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps * 1e3                         # us per call


def kv_copy_line():
    """samd_kv_copy_rows, 16 pairs x 1024 rows of a Llama-7B KV (n_kv 64, 32 heads, dh 128, fp16), against the copy peak:
    torch's device-to-device copy of the same number of bytes, contiguous."""
    n_kv, H, D, L, P, R = 64, 32, 128, 1024, 16, 1024
    pool = torch.randn(n_kv, P, H, L, D, dtype=torch.float16, device="cuda")
    cache = torch.zeros(n_kv, 2 * P, H, L, D, dtype=torch.float16, device="cuda")
    dst_row = torch.arange(P, 2 * P, dtype=torch.int32, device="cuda")
    src_row = torch.arange(P, dtype=torch.int32, device="cuda")
    n_rows = torch.full((P,), R, dtype=torch.int32, device="cuda")
    dt, st = E.kv_table(list(cache), "cuda"), E.kv_table(list(pool), "cuda")
    us = time_events(lambda: E.kv_copy_rows(dt, st, dst_row, src_row, n_rows), 10)
    torch.cuda.synchronize()
    assert torch.equal(cache[:, P:], pool)
    nbytes = n_kv * P * H * R * D * 2
    flat_src, flat_dst = pool.view(-1), cache.view(-1)[:pool.numel()]
    us_peak = time_events(lambda: flat_dst.copy_(flat_src), 10)
    del pool, cache
    torch.cuda.empty_cache()
    gbs, peak = 2 * nbytes / us / 1e3, 2 * nbytes / us_peak / 1e3
    return {"shape": f"n_kv {n_kv}, {H} heads, dh {D}, fp16; {P} pairs x {R} rows ({nbytes / 1e9:.2f} GB copied)",
            "us": us, "GB_per_s_read_plus_write": gbs, "copy_peak_GB_per_s": peak, "share_of_copy_peak": gbs / peak}


def clone_line():
    """samd_dyn_clone per request at max_tokens 16384 (64 pairs in one launch, and one pair) against the masked
    samd_dyn_reset + one samd_step ingesting the same 1024-token prefix (64 requests)."""
    R, cap, n = 64, 16384, 1024
    pool, dst = E.DynSamBatch(R, cap), E.DynSamBatch(R, cap)
    pe, de = (E.DraftEngine(d, None, K.FLAVOUR_SAMD, n_predicts=8) for d in (pool, dst))
    toks = torch.as_tensor(np.stack([synth.copy_mix(n, 32000, 90000 + r, p_copy=0.6) for r in range(R)]).astype(np.int32)).cuda()
    pe.step(toks, None, None)
    idx = torch.arange(R, dtype=torch.int32, device="cuda")
    us64 = time_events(lambda: dst.clone_from(pool, idx, idx), 20)
    us1 = time_events(lambda: dst.clone_from(pool, idx[:1], idx[:1]), 20)
    mask = torch.ones(R, dtype=torch.uint8, device="cuda")
    us_rebuild = time_events(lambda: (de.reset(mask), de.step(toks, None, None)), 20)
    torch.cuda.synchronize()
    assert np.array_equal(pool.meta()[:, :8], dst.meta()[:, :8])
    return {"max_tokens": cap, "prefix_tokens": n, "requests": R, "clone_us_per_request_64_pairs": us64 / R,
            "clone_us_one_pair": us1, "reset_plus_ingest_us_per_request_64": us_rebuild / R,
            "clone_launch_us_64_pairs": us64, "reset_plus_ingest_us_64": us_rebuild}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r05_prefix_cache.json")
    args = ap.parse_args()
    name, power = gpu_info()
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=4, max_position_embeddings=4096)
    dtype = torch.float16
    lm = LlamaForCausalLM(cfg).cuda().to(dtype).eval()
    lm32 = copy.deepcopy(lm).float()
    heads, prompts, limits, registered = workload()
    static, corpus_tokens = r03_corpus(lm, dtype)

    def make(model, dt, flavour, pool):
        kw = dict(dtype=dt, max_prefixes=N_HEADS if pool else 0)
        if flavour == "samd":
            dec = BatchedSamdDecoder(model, B, MAX_LEN, n_predicts=8, len_bias=5, len_threshold=3, **kw)
        else:
            dec = BatchedSamOnlyDecoder(model, B, MAX_LEN, max_predicts=T_SO, alpha=4.0, K=8, len_bias=5, static=static, **kw)
        for h in heads if pool else ():
            dec.add_prefix(h)
        return dec

    res = {}
    for flavour in ("samd", "sam_only"):
        outs32 = [run_serve(make(lm32, torch.float32, flavour, pool), prompts, limits)[0] for pool in (False, True)]
        diff32 = [i for i, (a, b) in enumerate(zip(*outs32)) if a != b]
        assert not diff32, f"{flavour}: fp32 outputs with and without the pool differ for requests {diff32[:16]}"
        arms, r = {}, {"outputs_equal_fp32": True}
        for arm, pool in (("no_pool", False), ("pool", True)):
            dec = make(lm, dtype, flavour, pool)
            run_serve(dec, prompts, limits)                    # warm-up: every graph the arm reaches is captured
            out, dt, st = arms[arm] = run_serve(dec, prompts, limits)
            split = admission_split(dec, prompts, limits)
            adm_ms = sum(v["total_ms"] for v in split.values())
            r[arm] = {"seconds": dt, "requests_per_s": N / dt, "output_tokens_per_s": sum(map(len, out)) / dt,
                      "steps": st["steps_run"], "host_syncs": st["host_syncs"], "admissions": st["admissions"],
                      **{k: st[k] for k in ("prefix_hits", "prefix_tokens") if k in st},
                      "admission": {**split, "total_ms": adm_ms, "share_of_serve_seconds": adm_ms / 1e3 / dt}}
            del dec
        diffs = {}
        for i, (a, b) in enumerate(zip(arms["pool"][0], arms["no_pool"][0])):
            if a != b:
                d = divergence(lm, lm32, prompts[i], a, b)
                d["pool"], d["no_pool"] = d.pop("serve"), d.pop("lockstep")
                diffs[str(i)] = d
        r["fp16_requests_equal"], r["fp16_divergences"] = N - len(diffs), diffs
        r["speedup"] = r["no_pool"]["seconds"] / r["pool"]["seconds"]
        res[flavour] = r
    del static
    torch.cuda.empty_cache()
    line = json.dumps({
        "gpu": name, "power_limit": power,
        "workload": f"B={B} slots, max_cache_len {MAX_LEN}, N={N} requests: one of {N_HEADS} copy_mix heads of 512-1536 "
                    f"tokens + a 32-256 token suffix (V=96, p_copy 0.7), {N - registered} of them with an unregistered "
                    f"head of the same length instead; max_new_tokens log-uniform in [16, 512] cut to the cache "
                    f"({sum(limits)} tokens in all), seeded; tiny Llama (2 layers, d=128, V=96) fp16; samd: sequence "
                    f"mode, n_predicts 8, len_bias 5, len_threshold 3; sam_only: max_predicts {T_SO}, alpha 4, K 8, "
                    f"len_bias 5, the r03 static corpus ({corpus_tokens} tokens, with counts)",
        "method": "serve() over all N requests by a decoder without a pool and by one with the 8 heads registered "
                  "(add_prefix, untimed); one untimed warm-up pass per arm, then one timed pass (host clock ending in a "
                  "device synchronise); outputs compared first: exactly with the same weights in fp32, request by request "
                  "in fp16; admission split from a separate pass with CUDA events around each part; kernel lines with "
                  "CUDA events over repeated launches after one warm-up launch",
        **res, "samd_kv_copy_rows": kv_copy_line(), "samd_dyn_clone": clone_line()})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
