"""Batched sam_only decoding (BatchedSamOnlyDecoder) at B = 64 on a tiny random-init fp16 Llama with a static corpus built
with counts: steps per second graphed and eager, mean accepted tokens per step, the share of request-steps that drafted a
static tree, and the device time of samd_draft_assemble at kv_len 1024 / 2048 next to the torch-op construction of the
same buffers (both captured as CUDA graphs of 50 launches, timed with CUDA events; the outputs are compared first).
    python tools/batched_sam_only_bench.py        (GPU box, from the repo root; prints one JSON line)"""
import json
import subprocess
import sys
import time

sys.path.insert(0, "sam-decoding_b200")
import numpy as np
import torch
from transformers import LlamaConfig, LlamaForCausalLM
from samd_b200 import _cabi as K, engine as E, synth
from samd_b200.batched import BatchedSamOnlyDecoder


def gpu_info():
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # reported, not guessed
        limit = f"unknown ({type(e).__name__})"
    return torch.cuda.get_device_name(0), limit


def torch_buffers(eng, cache_len, kv_len, dtype):
    """The same buffers as samd_draft_assemble, with torch ops (ancestor sets by T - 1 rounds of parent jumps)."""
    B, T = eng.draft.shape
    dev = eng.draft.device
    ar = torch.arange(T, device=dev)
    is_tree = eng.out_type == K.DRAFT_STATIC_TREE
    n = torch.where(is_tree, eng.tree_n, eng.draft_len).clamp(1, T)
    live = ar[None, :] < n[:, None]
    par = torch.where(is_tree[:, None] & live, eng.tree_parents.long(), ar[None, :] - 1)
    anc = torch.eye(T, dtype=torch.bool, device=dev).expand(B, T, T).clone()
    cur = par.clone()
    for _ in range(T - 1):
        ok = cur >= 0
        c = cur.clamp(min=0)
        anc.scatter_(2, c[:, :, None], anc.gather(2, c[:, :, None]) | ok[:, :, None])
        cur = torch.where(ok, par.gather(1, c), cur)
    anc = torch.where(live[:, :, None], anc, torch.eye(T, dtype=torch.bool, device=dev)[None])
    tokens = torch.where(live, torch.where(is_tree[:, None], eng.tree_tokens, eng.draft), 0)
    pos = cache_len.long()[:, None] + torch.where(live & is_tree[:, None], eng.tree_depth.long(), ar[None, :])
    leaves = eng.tree_shape[:, 0]
    tree_ret = torch.where(ar[None, :, None] < leaves[:, None, None], eng.tree_retrieve, -1)
    seq_ret = torch.full((B, T, T), -1, dtype=torch.int32, device=dev)
    seq_ret[:, 0] = torch.where(live, ar[None, :].int(), -1)
    retrieve = torch.where(is_tree[:, None, None], tree_ret, seq_ret)
    n_paths = torch.where(is_tree, leaves, 1)
    j = torch.arange(kv_len, device=dev)[None, None, :]
    rel = j - cache_len.long()[:, None, None]
    ok = (rel < 0) | ((rel < T) & torch.gather(anc, 2, rel.clamp(0, T - 1).expand(B, T, kv_len)))
    mask = torch.zeros(B, T, kv_len, dtype=dtype, device=dev).masked_fill_(~ok, torch.finfo(dtype).min)
    return tokens, pos, n, n_paths, retrieve, mask


def graph_time_us(fn, reps=50, rounds=20):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    t = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        b.synchronize()
        t.append(a.elapsed_time(b) * 1e3 / reps)
    return float(np.median(t))


def main():
    name, power = gpu_info()
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=4, max_position_embeddings=4096)
    dtype = torch.float16
    lm = LlamaForCausalLM(cfg).cuda().to(dtype).eval()
    B, n_new, T = 64, 128, 40
    prompts = [synth.copy_mix(192 + (i % 5) * 16, 96, 900 + i, p_copy=0.7).tolist() for i in range(B)]
    # the static corpus: pieces of the LM's own greedy continuations (from the lossless decoder without a corpus) - the
    # stand-in for a corpus in the domain the model writes - and unrelated copy_mix documents
    plain = BatchedSamOnlyDecoder(lm, B, 2048, max_predicts=T, alpha=4.0, dtype=dtype)
    cont, _ = plain.generate(prompts, n_new)
    docs = [c[i % 16:i % 16 + 64] for i, c in enumerate(cont)] + [synth.copy_mix(2000, 96, 5000 + k, p_copy=0.7).tolist()
                                                                  for k in range(8)]
    corpus = np.concatenate([np.asarray(d) for d in docs])
    static = E.StaticSamDevice.build(docs, synth.EOS, with_counts=True)
    dec = BatchedSamOnlyDecoder(lm, B, 2048, max_predicts=T, alpha=4.0, K=8, len_bias=5, static=static, dtype=dtype)
    res = {}
    for mode, kw in (("graph", dict(graph=True)), ("eager", dict(graph=False))):
        dec.generate(prompts, n_new, **kw)                   # warm-up (graph capture, allocator)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out, st = dec.generate(prompts, n_new, **kw)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        live_steps = sum(sum(1 for a in h if a) for h in st["accept_lengths"])
        res[mode] = {"steps": st["steps_run"], "host_syncs": st["host_syncs"], "graphed": st["graphed"], "seconds": dt,
                     "steps_per_s": st["steps_run"] / dt, "tokens_per_s": sum(len(o) for o in out) / dt,
                     "mean_accept": sum(map(sum, st["accept_lengths"])) / max(1, live_steps),
                     "tree_share": st["tree_steps"] / max(1, live_steps)}
        res[mode + "_tokens"] = out
    assert res.pop("graph_tokens") == res.pop("eager_tokens")
    # samd_draft_assemble vs torch ops on the drafts of a step early in a run (a mix of trees and sequences)
    dec.generate(prompts, 24)
    eng = dec.eng
    n_tree = int((eng.out_type == K.DRAFT_STATIC_TREE).sum())
    rng = np.random.default_rng(0)
    asm = {}
    for kv_len in (1024, 2048):
        cache_len = torch.as_tensor(rng.integers(0, kv_len - T + 1, size=B).astype(np.int32)).cuda()
        buf = dict(tokens=torch.zeros(B, T, dtype=torch.int32, device="cuda"),
                   pos=torch.zeros(B, T, dtype=torch.long, device="cuda"),
                   n_nodes=torch.zeros(B, dtype=torch.int32, device="cuda"), n_paths=torch.zeros(B, dtype=torch.int32, device="cuda"),
                   retrieve=torch.zeros(B, T, T, dtype=torch.int32, device="cuda"),
                   mask=torch.zeros(B, T, kv_len, dtype=dtype, device="cuda"))
        kernel = lambda: eng.assemble(cache_len, buf["tokens"], buf["pos"], buf["n_nodes"], buf["n_paths"], buf["retrieve"],
                                      buf["mask"])
        kernel()
        ref = torch_buffers(eng, cache_len, kv_len, dtype)
        torch.cuda.synchronize()
        for got, want in zip((buf["tokens"], buf["pos"], buf["n_nodes"], buf["n_paths"], buf["retrieve"]), ref[:5]):
            assert torch.equal(got.long(), want.long())
        assert torch.equal(buf["mask"].view(torch.int16), ref[5].view(torch.int16))
        us_k = graph_time_us(kernel)
        us_t = graph_time_us(lambda: torch_buffers(eng, cache_len, kv_len, dtype))
        mb = B * T * kv_len * 2 / 1e6
        asm[str(kv_len)] = {"assemble_us": us_k, "torch_ops_us": us_t, "mask_MB": mb, "mask_GB_per_s": mb * 1e-3 / (us_k * 1e-6)}
    print(json.dumps({
        "gpu": name, "power_limit": power,
        "workload": f"BatchedSamOnlyDecoder, B={B}, tiny Llama (2 layers, d=128, V=96) fp16, {n_new} new tokens, max_predicts {T}, "
                    f"alpha 4, K 8, len_bias 5, static corpus of {len(corpus)} tokens with counts (64-token pieces of the "
                    f"greedy continuations + copy_mix documents); `seconds` = one generate() "
                    "call incl. prefill (graphs captured by the warm-up call); mean_accept = tokens per live request-step; "
                    "tree_share = live request-steps that drafted a static tree",
        **res,
        "assemble": {"note": f"B={B}, T={T}, fp16 mask, the drafts of the last step of a 24-token run ({n_tree} trees), random cache lengths; device time "
                             "per call, median of 20 replays of a graph of 50 calls (CUDA events); the 10 MB mask stays in "
                             "the 126 MB L2 between calls; outputs checked equal first", **asm}}))


if __name__ == "__main__":
    main()
