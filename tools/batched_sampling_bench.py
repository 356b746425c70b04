"""Sampled decoding in the batched decoders, measured two ways.

1. serve() on the r04 workload (tools/continuous_batching_bench.py: B = 64 slots, N = 512 requests with copy_mix prompts
   of 64-1024 tokens and max_new_tokens log-uniform in [16, 512], the tiny fp16 Llama, the r03 static corpus for sam_only),
   for both decoders, greedy against sampled at (temperature 1.0) and at (temperature 0.7, top-p 0.9), one shared
   SamplingParams per arm (request i: seed 7 + i).  Per arm: wall seconds of one pass (host clock ending in a device
   synchronise, after an untimed warm-up pass of the same arm that captures every graph), decode steps, live slot-steps
   and output tokens per live request-step.
2. samd_verify_sample_requests against samd_verify_compact (greedy, no KV move) on the same logits: B = 64 sequence drafts
   of T in {16, 40} nodes, V in {32000, 128256}, bf16, the processor off (temperature 1) and on (temperature 0.7, top-p
   0.9, top-k 50).  Logits are seeded normal(0, 2) with every draft token raised by 14 in its parent's row, so that the
   sampled walk goes several levels deep (mean accept length reported).  CUDA events around 20 back-to-back launches
   after 3 warm-up launches; the 16 x 32000 block (65 MB) fits in L2, the others do not.
    python tools/batched_sampling_bench.py [--out profiles/r05_batched_sampling.json]
(GPU box, from the repo root; prints one JSON line and writes it to --out)"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, "sam-decoding_b200")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch
from transformers import LlamaConfig, LlamaForCausalLM
from samd_b200 import engine as E
from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder, SamplingParams
from batched_sam_only_bench import gpu_info
from continuous_batching_bench import B, MAX_LEN, N, T_SO, r03_corpus, workload

ARMS = {"greedy": None, "t1.0": SamplingParams(temperature=1.0, seed=7),
        "t0.7_p0.9": SamplingParams(temperature=0.7, top_p=0.9, seed=7)}


def run_serve(dec, prompts, limits, sampling):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_out = sum(len(tokens) for _, tokens, _ in dec.serve(prompts, limits, sampling=sampling))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    st = dec.serve_stats
    return {"seconds": dt, "steps": st["steps_run"], "live_slot_steps": st["live_slot_steps"], "output_tokens": n_out,
            "tokens_per_live_request_step": n_out / st["live_slot_steps"]}


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
        r = {}
        for arm, sp in ARMS.items():
            run_serve(dec, prompts, limits, sp)                   # warm-up: graph capture for every bucket the arm reaches
            r[arm] = run_serve(dec, prompts, limits, sp)
        for arm in ARMS:
            r[arm]["seconds_vs_greedy"] = r[arm]["seconds"] / r["greedy"]["seconds"]
        res[flavour] = r
        del dec
    return res


def kernel_times():
    out = {}
    Bk = 64
    for T in (16, 40):
        for V in (32000, 128256):
            g = torch.Generator(device="cuda").manual_seed(T * V)
            logits = torch.randn(Bk, T, V, generator=g, device="cuda") * 2.0
            tokens = torch.randint(0, V, (Bk, T), generator=g, device="cuda", dtype=torch.int32)
            logits.scatter_add_(2, tokens[:, 1:, None].long(), torch.full((Bk, T - 1, 1), 14.0, device="cuda"))
            logits = logits.to(torch.bfloat16)
            ver = E.Verifier(Bk, T)
            seeds = torch.arange(1, Bk + 1, dtype=torch.int64, device="cuda")
            offs = torch.zeros(Bk, dtype=torch.int64, device="cuda")
            cu = lambda v, dt=torch.float32: torch.full((Bk,), v, dtype=dt, device="cuda")
            off = (cu(1.0), cu(0.0), cu(0, torch.int32))
            on = (cu(0.7), cu(0.9), cu(50, torch.int32))
            res = {}
            for name, fn in (
                ("verify_compact", lambda o: ver.verify(logits, tokens, None, move_kv=False, out=o)),
                ("sample_off", lambda o: ver.verify_sample(logits, tokens, None, *off, seeds, offs, out=o)),
                ("sample_on", lambda o: ver.verify_sample(logits, tokens, None, *on, seeds, offs, out=o)),
            ):
                o = fn(None)
                for _ in range(2):
                    fn(o)
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(20):
                    fn(o)
                e.record()
                torch.cuda.synchronize()
                res[name] = {"us": s.elapsed_time(e) * 1e3 / 20,
                             "mean_accept_len": float(o["accept_len"].float().mean())}
            for name in ("sample_off", "sample_on"):
                res[name]["x_verify_compact"] = res[name]["us"] / res["verify_compact"]["us"]
            out[f"T{T}_V{V}"] = res
            del logits
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r05_batched_sampling.json")
    args = ap.parse_args()
    name, power = gpu_info()
    kern = kernel_times()
    serve = serve_arms()
    line = json.dumps({
        "gpu": name, "power_limit": power,
        "serve_workload": f"r04: B={B} slots, max_cache_len {MAX_LEN}, N={N} requests, copy_mix prompts of 64-1024 tokens "
                          "(V=96), max_new_tokens log-uniform in [16, 512]; tiny Llama (2 layers, d=128, V=96) fp16; samd: "
                          f"sequence mode, n_predicts 8; sam_only: max_predicts {T_SO}, alpha 4, K 8, the r03 static corpus",
        "serve_method": "one untimed warm-up pass per arm, then one timed pass (host clock ending in a device synchronise); "
                        "sampled arms: one shared SamplingParams, request i seeded 7 + i",
        "serve": serve,
        "kernel_method": "B=64 sequence drafts, bf16 logits normal(0, 2) with each draft token +14 in its parent's row; "
                         "CUDA events over 20 launches after 3 warm-up launches, us per launch; sample_off = temperature "
                         "1, no top-p / top-k; sample_on = temperature 0.7, top-p 0.9, top-k 50; verify_compact = the "
                         "greedy verify without KV moves",
        "kernel": kern})
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
