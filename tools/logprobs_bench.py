"""Per-token log-probabilities, measured two ways.

1. serve() on the r04 workload (tools/continuous_batching_bench.py: B = 64 slots, N = 512 requests with copy_mix prompts
   of 64-1024 tokens and max_new_tokens log-uniform in [16, 512], the tiny fp16 Llama, the r03 static corpus for sam_only),
   for both decoders, greedy, with logprobs=None, 0 and 8.  Every arm runs one untimed warm-up pass (graph capture), then
   ROUNDS timed passes with the arms alternating inside each round (host clock ending in a device synchronise); the
   median pass is reported beside all of them, with the host time spent turning the finished rows into the returned
   Python lists (batched._logprob_lists, timed inside the same passes).  The outputs of the three arms are compared
   first.
2. samd_token_logprobs at B = 64, T in {16, 40}, V in {32000, 128256}, bf16 logits normal(0, 2), n_top 0 and 8, on the
   identity path with accept lengths drawn (seeded) from the accept-length histogram of the sam_only logprobs=None
   serve() pass above (max_predicts 40; capped at T).  Scored bytes = sum(count) * V * 2.  Each timed launch follows a
   write of 512 MB to a scratch buffer, so that the scored rows (scored_bytes, per shape) come from DRAM, not L2;
   CUDA events around each launch, median of 30 after 3 warm-up launches.  samd_verify_compact (greedy, no KV move) at
   the same shape, timed the same way, stands beside it.
    python tools/logprobs_bench.py [--out profiles/r06_logprobs.json]
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
from samd_b200 import batched, engine as E
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
from batched_sam_only_bench import gpu_info
from continuous_batching_bench import B, MAX_LEN, N, T_SO, r03_corpus, workload

PEAK_BPS = 7.7e12                      # HGX B200 data sheet, one GPU (HBM3e)
ARMS = {"none": None, "logprobs0": 0, "logprobs8": 8}
ROUNDS = 5


HOST_LISTS = [0.0]                     # seconds spent building the returned Python lists (batched._logprob_lists)


def _timed_lists(rows, n, _inner=batched._logprob_lists):
    t0 = time.perf_counter()
    out = _inner(rows, n)
    HOST_LISTS[0] += time.perf_counter() - t0
    return out


batched._logprob_lists = _timed_lists


def run_serve(dec, prompts, limits, logprobs):
    torch.cuda.synchronize()
    HOST_LISTS[0] = 0.0
    t0 = time.perf_counter()
    got = {i: (tokens, info) for i, tokens, info in dec.serve(prompts, limits, logprobs=logprobs)}
    torch.cuda.synchronize()
    return time.perf_counter() - t0, HOST_LISTS[0], got


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
    res, hist = {}, None
    for flavour, make in makers.items():
        dec = make()
        outs = {arm: run_serve(dec, prompts, limits, lp)[2] for arm, lp in ARMS.items()}      # warm-up
        same = all(outs[arm][i][0] == outs["none"][i][0] and
                   outs[arm][i][1]["accept_lengths"] == outs["none"][i][1]["accept_lengths"]
                   for arm in ARMS for i in range(N))
        if flavour == "sam_only":
            hist = np.bincount(np.concatenate([outs["none"][i][1]["accept_lengths"] for i in range(N)]))
        secs, host = {arm: [] for arm in ARMS}, {arm: [] for arm in ARMS}
        for _ in range(ROUNDS):
            for arm, lp in ARMS.items():
                t, h, _ = run_serve(dec, prompts, limits, lp)
                secs[arm].append(t)
                host[arm].append(h)
        st = dec.serve_stats
        r = {"outputs_equal": same, "steps": st["steps_run"], "host_syncs": st["host_syncs"],
             "output_tokens": sum(len(outs["none"][i][0]) for i in range(N))}
        for arm in ARMS:
            r[arm] = {"seconds_median": statistics.median(secs[arm]), "seconds_all": secs[arm],
                      "host_lists_seconds_median": statistics.median(host[arm])}
        for arm in ("logprobs0", "logprobs8"):
            r[arm]["vs_none"] = r[arm]["seconds_median"] / r["none"]["seconds_median"]
            r[arm]["extra_us_per_step"] = (r[arm]["seconds_median"] - r["none"]["seconds_median"]) * 1e6 / st["steps_run"]
        res[flavour] = r
        del dec
    return res, hist


def kernel_times(hist):
    p = hist[1:].astype(np.float64)
    p /= p.sum()
    rng = np.random.default_rng(6)
    scratch = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    out = {}
    Bk = 64
    for T in (16, 40):
        count = np.minimum(rng.choice(np.arange(1, len(p) + 1), size=Bk, p=p), T).astype(np.int32)
        for V in (32000, 128256):
            g = torch.Generator(device="cuda").manual_seed(T * V)
            logits = (torch.randn(Bk, T, V, generator=g, device="cuda") * 2.0).to(torch.bfloat16)
            tokens = torch.randint(0, V, (Bk, T), generator=g, device="cuda", dtype=torch.int32)
            idx = torch.arange(T, dtype=torch.int32, device="cuda").repeat(Bk, 1).contiguous()
            cnt = torch.as_tensor(count).cuda()
            nxt = tokens[:, 0].contiguous()
            ver = E.Verifier(Bk, T)
            scored = int(count.sum()) * V * 2
            res = {"scored_rows": int(count.sum()), "scored_bytes": scored}
            arms = [(f"logprobs_top{n}", (lambda n: lambda o: ver.token_logprobs(logits, idx, cnt, tokens, nxt, n_top=n,
                                                                                out=o))(n)) for n in (0, 8)]
            arms.append(("verify_compact", lambda o: ver.verify(logits, tokens, None, move_kv=False, out=o)))
            for name, fn in arms:
                o = fn(None)
                for _ in range(3):
                    fn(o)
                times = []
                for _ in range(30):
                    scratch.fill_(1)                                    # evict the scored rows from L2
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    fn(o)
                    e.record()
                    torch.cuda.synchronize()
                    times.append(s.elapsed_time(e) * 1e3)
                res[name] = {"us": statistics.median(times)}
            for n in (0, 8):
                r = res[f"logprobs_top{n}"]
                r["bytes_per_s"] = scored / (r["us"] * 1e-6)
                r["share_of_7.7TBps"] = r["bytes_per_s"] / PEAK_BPS
                r["vs_verify_compact"] = r["us"] / res["verify_compact"]["us"]
            out[f"T{T}_V{V}"] = res
            del logits
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r06_logprobs.json")
    args = ap.parse_args()
    name, power = gpu_info()
    serve, hist = serve_arms()
    kern = kernel_times(hist)
    line = json.dumps({
        "gpu": name, "power_limit": power,
        "serve_workload": f"r04: B={B} slots, max_cache_len {MAX_LEN}, N={N} requests, copy_mix prompts of 64-1024 tokens "
                          "(V=96), max_new_tokens log-uniform in [16, 512]; tiny Llama (2 layers, d=128, V=96) fp16, greedy; "
                          f"samd: sequence mode, n_predicts 8; sam_only: max_predicts {T_SO}, alpha 4, K 8, the r03 static "
                          "corpus",
        "serve_method": f"one untimed warm-up pass per arm (outputs compared), then {ROUNDS} rounds of one timed pass per arm, "
                        "arms alternating; host clock ending in a device synchronise; median reported",
        "serve": serve,
        "accept_len_hist": hist.tolist(),
        "kernel_method": "B=64, identity path, bf16 logits normal(0, 2), accept lengths drawn from accept_len_hist (sam_only "
                         "serve, logprobs=None) capped at T; 512 MB scratch write before each timed launch (scored rows "
                         "from DRAM); CUDA events per launch, median of 30 after 3 warm-up launches; bytes_per_s = scored "
                         "bytes / time; verify_compact = the greedy verify without KV moves, same shape, same method",
        "kernel": kern})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
