"""Repetition / presence / frequency penalties, measured two ways.

1. serve() on the r04 workload (tools/continuous_batching_bench.py: B = 64 slots, N = 512 requests with copy_mix prompts
   of 64-1024 tokens and max_new_tokens log-uniform in [16, 512], the tiny fp16 Llama, the r03 static corpus for sam_only),
   for both decoders, greedy, with penalties=None, neutral Penalties(), repetition_penalty=1.1 and presence_penalty =
   frequency_penalty = 0.5.  Every arm runs one untimed warm-up pass (graph capture), then ROUNDS timed passes with the
   arms alternating inside each round (host clock ending in a device synchronise); the median pass is reported beside all
   of them, with the steps and the tokens per live request-step (penalties push against what the automaton drafts).  The
   outputs of None and neutral are compared.
2. samd_apply_penalties at B = 64, T in {16, 40}, V in {32000, 128256}, bf16 logits normal(0, 2), identity chains of
   random node tokens, with 256 / 2048 / 8192 distinct history tokens per request (counts 1-3, a quarter also in the
   prompt), r = 1.1, p = f = 0.5.  Bytes moved = the count table (B * V * 4) + the distinct 32-byte logits sectors the
   rewrites touch, read and written.  Each timed launch follows a write of 512 MB to a scratch buffer, so that the count
   table and the logits come from DRAM, not L2; CUDA events around each launch, median of 30 after 3 warm-up launches.
   samd_verify_compact (greedy, no KV move) at the same shape, timed the same way, stands beside it.
    python tools/penalties_bench.py [--out profiles/r07_penalties.json]
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
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder, Penalties
from batched_sam_only_bench import gpu_info
from continuous_batching_bench import B, MAX_LEN, N, T_SO, r03_corpus, workload

PEAK_BPS = 7.7e12                      # HGX B200 data sheet, one GPU (HBM3e)
ARMS = {"none": None, "neutral": Penalties(), "repetition_1.1": Penalties(repetition_penalty=1.1),
        "presence_frequency_0.5": Penalties(presence_penalty=0.5, frequency_penalty=0.5)}
ROUNDS = 3


def run_serve(dec, prompts, limits, penalties):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = {i: (tokens, info) for i, tokens, info in dec.serve(prompts, limits, penalties=penalties)}
    torch.cuda.synchronize()
    return time.perf_counter() - t0, got, dict(dec.serve_stats)


def serve_arms():
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=4, max_position_embeddings=4096)
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
        warm = {arm: run_serve(dec, prompts, limits, pn) for arm, pn in ARMS.items()}
        outs = {arm: w[1] for arm, w in warm.items()}
        same = all(outs["neutral"][i][0] == outs["none"][i][0] and
                   outs["neutral"][i][1]["accept_lengths"] == outs["none"][i][1]["accept_lengths"] for i in range(N))
        secs = {arm: [] for arm in ARMS}
        for _ in range(ROUNDS):
            for arm, pn in ARMS.items():
                secs[arm].append(run_serve(dec, prompts, limits, pn)[0])
        r = {"none_equals_neutral": same}
        for arm in ARMS:
            st = warm[arm][2]
            tokens = sum(len(outs[arm][i][0]) for i in range(N))
            r[arm] = {"seconds_median": statistics.median(secs[arm]), "seconds_all": secs[arm], "steps": st["steps_run"],
                      "output_tokens": tokens, "live_slot_steps": st["live_slot_steps"],
                      "tokens_per_live_request_step": tokens / st["live_slot_steps"],
                      "vs_none": statistics.median(secs[arm]) / statistics.median(secs["none"])}
        res[flavour] = r
        del dec
    return res


def sectors_touched(hist, tokens, T):
    """Distinct 32-byte bf16 logits sectors the launch rewrites: per request, the history tokens and the node tokens of
    every row (an upper bound for a chain: row j holds only the first j + 1 node tokens)."""
    n = 0
    for b in range(hist.shape[0]):
        n += T * len(np.unique(np.concatenate([hist[b], tokens[b]]) // 16))
    return n


def kernel_times():
    rng = np.random.default_rng(7)
    scratch = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    out = {}
    Bk = 64
    one = lambda v: torch.full((Bk,), v, dtype=torch.float32, device="cuda")
    r, p, f = one(1.1), one(0.5), one(0.5)
    for T in (16, 40):
        for V in (32000, 128256):
            g = torch.Generator(device="cuda").manual_seed(T * V)
            logits = (torch.randn(Bk, T, V, generator=g, device="cuda") * 2.0).to(torch.bfloat16)
            tokens_np = rng.integers(0, V, size=(Bk, T)).astype(np.int32)
            tokens = torch.as_tensor(tokens_np).cuda()
            ver = E.Verifier(Bk, T)
            vo = ver.verify(logits, tokens, None, move_kv=False)
            res = {}
            for n_hist in (256, 2048, 8192):
                hist = np.stack([rng.choice(V, size=n_hist, replace=False) for _ in range(Bk)])
                counts = np.zeros((Bk, V), np.uint32)
                rows = np.arange(Bk)[:, None]
                counts[rows, hist] = rng.integers(1, 4, size=(Bk, n_hist)).astype(np.uint32)
                counts[rows, hist[:, :n_hist // 4]] |= np.uint32(1 << 31)
                cnt = torch.as_tensor(counts.view(np.int32)).cuda()
                fn = lambda: E.apply_penalties(logits, cnt, r, p, f, tokens=tokens)
                sectors = sectors_touched(hist, tokens_np, T)
                nbytes = Bk * V * 4 + 2 * 32 * sectors
                res[f"hist{n_hist}"] = {"us": _time(fn, scratch), "count_table_bytes": Bk * V * 4,
                                        "logits_sectors": sectors, "bytes_moved": nbytes}
            res["verify_compact"] = {"us": _time(lambda: ver.verify(logits, tokens, None, move_kv=False, out=vo), scratch),
                                     "logits_bytes": Bk * T * V * 2}
            for n_hist in (256, 2048, 8192):
                x = res[f"hist{n_hist}"]
                x["bytes_per_s"] = x["bytes_moved"] / (x["us"] * 1e-6)
                x["share_of_7.7TBps"] = x["bytes_per_s"] / PEAK_BPS
                x["vs_verify_compact"] = x["us"] / res["verify_compact"]["us"]
            out[f"T{T}_V{V}"] = res
            del logits
    return out


def _time(fn, scratch):
    for _ in range(3):
        fn()
    times = []
    for _ in range(30):
        scratch.fill_(1)                                        # evict the count table and the logits from L2
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e) * 1e3)
    return statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07_penalties.json")
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
        "serve_method": f"one untimed warm-up pass per arm (None and neutral outputs compared), then {ROUNDS} rounds of one "
                        "timed pass per arm, arms alternating; host clock ending in a device synchronise; median reported",
        "serve": serve,
        "kernel_method": "B=64, identity chains of random node tokens, bf16 logits normal(0, 2); per request n distinct "
                         "history tokens with counts 1-3, a quarter of them also prompt tokens; r=1.1, p=f=0.5; 512 MB "
                         "scratch write before each timed launch (count table and logits from DRAM); CUDA events per "
                         "launch, median of 30 after 3 warm-up launches; bytes_moved = count table + touched 32-byte logits "
                         "sectors read and written; verify_compact = the greedy verify without KV moves, same shape",
        "kernel": kern})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
