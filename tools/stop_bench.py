"""Stop sequences, measured two ways.

1. serve() on the r04 workload (tools/continuous_batching_bench.py: B = 64 slots, N = 512 requests with copy_mix prompts
   of 64-1024 tokens and max_new_tokens log-uniform in [16, 512], the tiny fp16 Llama, the r03 static corpus for sam_only),
   for both decoders, greedy, with three arms: stop=None; 16 sequences of 16 ids that never occur (the cost of the extra
   launch per step); and one sequence planted at a random point of each request's unstopped output (4 ids ending there,
   seeded).  Every arm runs one untimed warm-up pass (graph capture), then ROUNDS timed passes with the arms alternating
   inside each round (host clock ending in a device synchronise); the median pass is reported beside all of them, with
   the steps, live slot-steps and output tokens, and the planted arm's savings against None.  The never arm's outputs
   are compared with None's, the planted arm's with None's cut at the earliest match.
2. samd_stop_match alone at B in {64, 256}, width in {16, 40, 128}: every request with 16 sequences of 16 ids, a full
   candidate row and 40 history tokens, nothing matching (every pair compared in full: the most work a launch does); a
   CUDA graph of 20 launches, CUDA events per replay, median of 30 replays / 20.  samd_verify_compact (greedy, no KV
   move) at the same B and T, V = 32000 bf16, timed the same way, stands beside it.
    python tools/stop_bench.py [--out profiles/r08_stop_sequences.json]
(GPU box, from the repo root; prints one JSON line and writes it to --out)"""
import argparse
import json
import os
import statistics
import sys
import time

sys.path.insert(0, "sam-decoding_b200")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch
from transformers import LlamaConfig, LlamaForCausalLM
from samd_b200 import engine as E
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder, StopSequences
from batched_sam_only_bench import gpu_info
from continuous_batching_bench import B, MAX_LEN, N, T_SO, r03_corpus, workload

ROUNDS = 3
V_TINY = 96


def run_serve(dec, prompts, limits, stop):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = {i: (tokens, info) for i, tokens, info in dec.serve(prompts, limits, stop=stop)}
    torch.cuda.synchronize()
    return time.perf_counter() - t0, got, dict(dec.serve_stats)


def earliest(u, seqs):
    """Length of u cut after the earliest end of any of seqs (matched within u), or len(u)."""
    for e in range(len(u)):
        for s in seqs:
            if e + 1 >= len(s) and u[e + 1 - len(s):e + 1] == s:
                return e + 1
    return len(u)


def serve_arms():
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=V_TINY, hidden_size=128, intermediate_size=256, num_hidden_layers=2,
                      num_attention_heads=4, num_key_value_heads=4, max_position_embeddings=4096)
    dtype = torch.float16
    lm = LlamaForCausalLM(cfg).cuda().to(dtype).eval()
    prompts, limits = workload()
    static, _ = r03_corpus(lm, dtype)
    makers = {
        "samd": lambda: BatchedSamdDecoder(lm, B, MAX_LEN, n_predicts=8, len_bias=5, len_threshold=3, dtype=dtype),
        "sam_only": lambda: BatchedSamOnlyDecoder(lm, B, MAX_LEN, max_predicts=T_SO, alpha=4.0, K=8, len_bias=5,
                                                  static=static, dtype=dtype),
    }
    res = {}
    for flavour, make in makers.items():
        dec = make()
        none = run_serve(dec, prompts, limits, None)
        # never: 16 x 16 ids the outputs do not contain (checked); planted: 4 ids ending at a random point
        seen = {t for i in range(N) for t in none[1][i][0]}
        absent = [t for t in range(V_TINY) if t not in seen] or [0]
        never = StopSequences([[absent[0]] * 15 + [absent[(j + 1) % len(absent)]] for j in range(16)])
        rng = np.random.default_rng(8)
        planted, want = [], []
        for i in range(N):
            u = none[1][i][0]
            e = int(rng.integers(0, len(u)))
            seq = [u[max(0, e - 3):e + 1]]
            planted.append(StopSequences(seq))
            want.append(u[:earliest(u, seq)])
        arms = {"none": None, "never_16x16": never, "planted": planted}
        warm = {"none": none}
        warm.update({arm: run_serve(dec, prompts, limits, ss) for arm, ss in arms.items() if arm != "none"})
        outs = {arm: w[1] for arm, w in warm.items()}
        never_same = all(outs["never_16x16"][i][0] == outs["none"][i][0] and
                         outs["never_16x16"][i][1]["accept_lengths"] == outs["none"][i][1]["accept_lengths"]
                         for i in range(N))
        # each planted output ends at the earliest match in its own tokens; it equals None's output cut there unless
        # the fp16 greedy tokens diverged first (a stopped request changes its neighbours' batch and key-length bucket)
        own_cut = all(earliest(outs["planted"][i][0], planted[i].sequences) == len(outs["planted"][i][0]) for i in range(N))
        planted_cut = sum(outs["planted"][i][0] == want[i] for i in range(N))
        secs = {arm: [] for arm in arms}
        for _ in range(ROUNDS):
            for arm, ss in arms.items():
                secs[arm].append(run_serve(dec, prompts, limits, ss)[0])
        r = {"never_equals_none": never_same, "planted_ends_at_own_earliest_match": own_cut,
             "planted_requests_equal_to_cut_none": planted_cut,
             "planted_finish_reasons": {k: sum(outs["planted"][i][1]["finish_reason"] == k for i in range(N))
                                        for k in ("stop", "length", "cache")}}
        for arm in arms:
            st = warm[arm][2]
            tokens = sum(len(outs[arm][i][0]) for i in range(N))
            r[arm] = {"seconds_median": statistics.median(secs[arm]), "seconds_all": secs[arm], "steps": st["steps_run"],
                      "output_tokens": tokens, "live_slot_steps": st["live_slot_steps"],
                      "vs_none": statistics.median(secs[arm]) / statistics.median(secs["none"])}
        p, n0 = r["planted"], r["none"]
        r["planted_saved"] = {"seconds": n0["seconds_median"] - p["seconds_median"], "steps": n0["steps"] - p["steps"],
                              "live_slot_steps": n0["live_slot_steps"] - p["live_slot_steps"],
                              "output_tokens": n0["output_tokens"] - p["output_tokens"]}
        res[flavour] = r
        del dec
    return res


def kernel_times():
    out = {}
    S, L = 16, 16
    for Bk in (64, 256):
        for W in (16, 40, 128):
            dev = "cuda"
            tokens = torch.randint(1, 1000, (Bk, W), dtype=torch.int32, device=dev)
            count = torch.full((Bk,), W, dtype=torch.int32, device=dev)
            hist = torch.randint(1, 1000, (Bk, 64), dtype=torch.int32, device=dev)
            hist_len = torch.full((Bk,), 40, dtype=torch.int32, device=dev)
            stop_tok = torch.randint(1, 1000, (Bk, S, L), dtype=torch.int32, device=dev)
            stop_tok[:, :, 15] = 5000                            # never present: every comparison runs to the last id
            stop_tok[:, :, :15] = tokens[:, :1, None]            # the first 15 ids all equal one repeated candidate...
            tokens[:] = tokens[:, :1]                            # ...so every pair compares all 16 ids
            stop_len = torch.full((Bk, S), L, dtype=torch.int32, device=dev)
            oc, oh = torch.empty_like(count), torch.empty_like(count)
            fn = lambda: E.match_stops(tokens, count, hist, hist_len, stop_tok, stop_len, out_count=oc, out_hit=oh)
            fn()
            assert int(oh.max()) == -1
            hist[:] = tokens[:, :1]
            V = 32000
            g = torch.Generator(device=dev).manual_seed(Bk * W)
            logits = (torch.randn(Bk, W, V, generator=g, device=dev) * 2.0).to(torch.bfloat16)
            ver = E.Verifier(Bk, W)
            draft = torch.randint(0, V, (Bk, W), dtype=torch.int32, device=dev)
            vo = ver.verify(logits, draft, None, move_kv=False)
            out[f"B{Bk}_W{W}"] = {"stop_match_us": _time(fn),
                                  "verify_compact_V32000_bf16_us": _time(lambda: ver.verify(logits, draft, None, move_kv=False,
                                                                                           out=vo))}
            out[f"B{Bk}_W{W}"]["ratio"] = out[f"B{Bk}_W{W}"]["stop_match_us"] / out[f"B{Bk}_W{W}"]["verify_compact_V32000_bf16_us"]
            del logits
    return out


def _time(fn, reps=20):
    """Device time of one launch: a CUDA graph of `reps` launches, CUDA events around each replay, median of 30 replays
    after 3 warm-up ones, divided by reps (the host-side argument checks are not in the timed window)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    for _ in range(3):
        g.replay()
    times = []
    for _ in range(30):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        g.replay()
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e) * 1e3 / reps)
    return statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r08_stop_sequences.json")
    args = ap.parse_args()
    name, power = gpu_info()
    kern = kernel_times()
    serve = serve_arms()
    line = json.dumps({
        "gpu": name, "power_limit": power,
        "serve_workload": f"r04: B={B} slots, max_cache_len {MAX_LEN}, N={N} requests, copy_mix prompts of 64-1024 tokens "
                          "(V=96), max_new_tokens log-uniform in [16, 512]; tiny Llama (2 layers, d=128, V=96) fp16, greedy; "
                          f"samd: sequence mode, n_predicts 8; sam_only: max_predicts {T_SO}, alpha 4, K 8, the r03 static "
                          "corpus",
        "serve_method": f"one untimed warm-up pass per arm (outputs compared), then {ROUNDS} rounds of one timed pass per "
                        "arm, arms alternating; host clock ending in a device synchronise; median reported; planted: one "
                        "4-id sequence per request ending at a uniform random position of its unstopped output (seed 8)",
        "serve": serve,
        "kernel_method": "16 sequences x 16 ids per request, full candidate rows, 40 history tokens, every (position, "
                         "sequence) pair compared in full and none matching; a CUDA graph of 20 back-to-back launches, CUDA "
                         "events per replay, median of 30 replays / 20; verify_compact = the greedy verify without KV moves at the same B and T, "
                         "V=32000 bf16",
        "kernel": kern})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
