"""Logit controls (logit bias, bad words, min_tokens), measured two ways.

1. samd_apply_logit_controls alone, worst case, at B in {64, 256}, T in {16, 40, 61 (the Token-Recycle tree), 128} and
   V in {32000, 128256} bf16: every request with 256 bias entries, 16 bad words of 16 ids and 16 stop sequences of 16
   ids under min_tokens (every row predicts a position below it), 40 history tokens, and every (row, sequence) pair
   compared in full (each head equals the context tail, the last id differs per sequence).  A CUDA graph of 20
   launches, CUDA events per replay, median of 30 replays / 20.  samd_verify_compact (greedy, no KV move) at the same
   B, T and V, timed the same way, stands beside it.
2. serve() on the r04 workload (tools/continuous_batching_bench.py: B = 64 slots, N = 512 requests with copy_mix prompts
   of 64-1024 tokens and max_new_tokens log-uniform in [16, 512], the tiny fp16 Llama, the r03 static corpus for
   sam_only), for both decoders, greedy, with three arms: controls=None; neutral LogitControls(); and active controls
   (a -inf ban and two biases, four bad words taken from the None arm's most frequent bigrams, min_tokens 8, per
   request).  Every arm runs one untimed warm-up pass (graph capture, outputs compared), then ROUNDS timed passes with
   the arms alternating inside each round (host clock ending in a device synchronise); the median pass is reported
   beside all of them with the steps and output tokens.  The neutral arm's outputs are compared with None's; the active
   arm's are checked to contain no banned token and no bad word.
    python tools/logit_controls_bench.py [--out profiles/r09_logit_controls.json]
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
from samd_b200 import engine as E, synth
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder, LogitControls
from batched_sam_only_bench import gpu_info
from continuous_batching_bench import B, MAX_LEN, N, T_SO, r03_corpus, workload
from stop_bench import _time

ROUNDS = 3
V_TINY = 96


def kernel_times():
    out = {}
    dev = "cuda"
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
    for V in (32000, 128256):
        for Bk in (64, 256):
            for T in (16, 40, 61, 128):
                g = torch.Generator(device=dev).manual_seed(Bk * T)
                logits = (torch.randn(Bk, T, V, generator=g, device=dev) * 2.0).to(torch.bfloat16)
                tokens = torch.full((Bk, T), 7, dtype=torch.int32, device=dev)          # every context: 7 7 7 ...
                hist, hist_len = torch.full((Bk, 64), 7, dtype=torch.int32, device=dev), torch.full((Bk,), 40, dtype=torch.int32, device=dev)
                bias_ids = torch.stack([torch.randperm(V, device=dev)[:256] for _ in range(Bk)]).to(torch.int32)
                bias, bias_n = torch.full((Bk, 256), 0.5, device=dev), torch.full((Bk,), 256, dtype=torch.int32, device=dev)
                seqs = torch.full((Bk, 16, 16), 7, dtype=torch.int32, device=dev)
                seqs[:, :, 15] = 100 + torch.arange(16, device=dev, dtype=torch.int32)  # heads match, last ids differ
                lens = torch.full((Bk, 16), 16, dtype=torch.int32, device=dev)
                min_tokens = torch.full((Bk,), 1 << 20, dtype=torch.int32, device=dev)
                kw = {}
                if T == 61:                                                           # the tree: its path table
                    ri = torch.as_tensor(synth.tree_retrieve_indices(synth.token_recycle_tree()), dtype=torch.int32)
                    kw = dict(retrieve=ri[None].expand(Bk, -1, -1).contiguous().to(dev))
                fn = lambda: E.apply_logit_controls(logits, bias_ids, bias, bias_n, seqs, lens, min_tokens, tokens=tokens,
                                                    hist=hist, hist_len=hist_len, stop_tokens=seqs, stop_len=lens, eos=3,
                                                    **kw)
                ver = E.Verifier(Bk, T)
                draft = torch.randint(0, V, (Bk, T), dtype=torch.int32, device=dev)
                vo = ver.verify(logits, draft, None, move_kv=False)
                key = f"V{V}_B{Bk}_T{T}"
                out[key] = {"logit_controls_us": _time(fn),
                            "verify_compact_bf16_us": _time(lambda: ver.verify(logits, draft, None, move_kv=False, out=vo))}
                out[key]["ratio"] = out[key]["logit_controls_us"] / out[key]["verify_compact_bf16_us"]
                del logits, ver
                torch.cuda.empty_cache()
    return out


def run_serve(dec, prompts, limits, controls):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = {i: (tokens, info) for i, tokens, info in dec.serve(prompts, limits, controls=controls)}
    torch.cuda.synchronize()
    return time.perf_counter() - t0, got, dict(dec.serve_stats)


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
        counts = np.bincount(np.concatenate([none[1][i][0] for i in range(N)]), minlength=V_TINY)
        counts[0] = 0
        top = [int(t) for t in np.argsort(-counts)[:4]]
        pairs = {}
        for i in range(N):
            u = none[1][i][0]
            for k in range(len(u) - 1):
                pairs[(u[k], u[k + 1])] = pairs.get((u[k], u[k + 1]), 0) + 1
        bad = [list(p) for p, _ in sorted(pairs.items(), key=lambda kv: -kv[1])[:4]]
        active = [LogitControls(logit_bias={top[0]: -float("inf"), top[1]: -2.0, top[2]: 1.5}, bad_words=bad,
                                min_tokens=min(8, limits[i])) for i in range(N)]
        arms = {"none": None, "neutral": LogitControls(), "active": active}
        warm = {"none": none}
        warm.update({arm: run_serve(dec, prompts, limits, lc) for arm, lc in arms.items() if arm != "none"})
        outs = {arm: w[1] for arm, w in warm.items()}
        neutral_same = all(outs["neutral"][i][0] == outs["none"][i][0] and
                           outs["neutral"][i][1]["accept_lengths"] == outs["none"][i][1]["accept_lengths"]
                           for i in range(N))
        clean = all(top[0] not in outs["active"][i][0] and
                    not any(outs["active"][i][0][k:k + 2] == w for w in bad for k in range(len(outs["active"][i][0])))
                    for i in range(N))
        secs = {arm: [] for arm in arms}
        for _ in range(ROUNDS):
            for arm, lc in arms.items():
                secs[arm].append(run_serve(dec, prompts, limits, lc)[0])
        r = {"neutral_equals_none": neutral_same, "active_has_no_banned_token_or_bad_word": clean,
             "active_requests_changed": sum(outs["active"][i][0] != outs["none"][i][0] for i in range(N))}
        for arm in arms:
            st = warm[arm][2]
            r[arm] = {"seconds_median": statistics.median(secs[arm]), "seconds_all": secs[arm], "steps": st["steps_run"],
                      "output_tokens": sum(len(outs[arm][i][0]) for i in range(N)),
                      "vs_none": statistics.median(secs[arm]) / statistics.median(secs["none"])}
        res[flavour] = r
        del dec
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r09_logit_controls.json")
    args = ap.parse_args()
    name, power = gpu_info()
    kern = kernel_times()
    serve = serve_arms()
    line = json.dumps({
        "gpu": name, "power_limit": power,
        "kernel_method": "worst case per request: 256 bias entries, 16 bad words x 16 ids and 16 stop sequences x 16 ids "
                         "under min_tokens, every head matching the context tail (every pair compared in full), 40 "
                         "history tokens; T=61 with the Token-Recycle path table, the others identity chains; bf16 "
                         "logits; a CUDA graph of 20 back-to-back launches, CUDA events per replay, median of 30 replays "
                         "/ 20; verify_compact = the greedy verify without KV moves at the same B, T and V",
        "kernel": kern,
        "serve_workload": f"r04: B={B} slots, max_cache_len {MAX_LEN}, N={N} requests, copy_mix prompts of 64-1024 tokens "
                          "(V=96), max_new_tokens log-uniform in [16, 512]; tiny Llama (2 layers, d=128, V=96) fp16, greedy; "
                          f"samd: sequence mode, n_predicts 8; sam_only: max_predicts {T_SO}, alpha 4, K 8, the r03 static "
                          "corpus",
        "serve_method": f"one untimed warm-up pass per arm (outputs compared), then {ROUNDS} rounds of one timed pass per "
                        "arm, arms alternating; host clock ending in a device synchronise; median reported; active: "
                        "-inf on the most frequent token, -2 / +1.5 on the next two, the four most frequent bigrams of "
                        "the None arm as bad words, min_tokens min(8, max_new_tokens)",
        "serve": serve})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
