"""GPU tests of per-token log-probabilities: samd_token_logprobs against torch.log_softmax (-1 path entries, counts of 0,
finished requests, -inf and NaN rows, 16-bit ties at V = 128256), its determinism, and the decoders' logprobs= against a
teacher-forced forward over prompt + output, with the tokens, accept lengths and launches of logprobs=None unchanged."""
import numpy as np
import pytest
import torch

import samd_oracle as O

pytestmark = pytest.mark.gpu

N_REQ = 13
NAN = float("nan")


def _tiny_llama():
    """The fp32 tiny Llama of the sampling tests, with token 0 pushed out of its greedy choices.  A -1 pad of a path
    table selects token 0 and is "accepted" when the compared row's argmax is 0 (the reference's A9 corner, see
    BatchedSamOnlyDecoder): that token is then decided by another node's row and its KV row is not its own, so the outputs
    after it are not what a clean forward over prompt + tokens computes.  This untrained LM predicts 0 after 0 almost
    everywhere, which made the corner common; with token 0 never the argmax it cannot occur."""
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, max_position_embeddings=2048, attn_implementation="eager")
    lm = LlamaForCausalLM(cfg).to("cuda", torch.float32).eval()
    head = torch.nn.Linear(cfg.hidden_size, cfg.vocab_size, bias=True).to("cuda")
    with torch.no_grad():
        head.weight.copy_(lm.lm_head.weight)
        head.bias.zero_()
        head.bias[0] = -30.0
    lm.lm_head = head
    return lm


@pytest.fixture(scope="module")
def lm():
    return _tiny_llama()


@pytest.fixture(scope="module")
def work():
    from samd_b200 import synth
    from samd_b200.batched import SamplingParams
    lens = (150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70)
    prompts = [synth.copy_mix(n, 96, 300 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    limits = [8, 96] + [8 + (37 * i) % 89 for i in range(2, N_REQ)]
    procs = [dict(temperature=1.0), dict(temperature=0.7, top_p=0.9), dict(temperature=1.3, top_k=5), dict(greedy=True)]
    params = [SamplingParams(seed=1000 + 7 * i, **procs[i % len(procs)]) for i in range(N_REQ)]
    return prompts, limits, params


def _decoders(lm):
    from samd_b200 import engine as E, synth
    from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
    docs = [synth.copy_mix(300, 96, 5 + k).tolist() for k in range(3)] + [[i] for i in range(3, 96)]
    static = E.StaticSamDevice.build(docs, 2, with_counts=True)
    samd = lambda B, **kw: BatchedSamdDecoder(lm, B, 512, n_predicts=8, len_bias=5, len_threshold=3, dtype=torch.float32,
                                              **kw)
    sam_only = lambda B, **kw: BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0,
                                                     static=static, dtype=torch.float32, **kw)
    return dict(samd=samd, sam_only=sam_only)


def _close(got, want, tol):
    """Elementwise: both NaN, equal (infinities included), or within tol."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    ok = (np.isnan(got) & np.isnan(want)) | (got == want) | (np.abs(got - want) <= tol)
    return bool(ok.all())


# ---- 1. the kernel against torch --------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [997, 32000, 128256])
@pytest.mark.parametrize("dt", ["fp32", "bf16", "fp16"])
def test_kernel_matches_torch(dt, V):
    from samd_b200 import engine as E
    B, T, W = 12, 10, 8
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[dt]
    rng = np.random.default_rng(V)
    g = torch.Generator(device="cuda").manual_seed(V + 1)
    lg = (torch.randn(B, T, V, generator=g, device="cuda") * 3.0).to(tdt)
    n_nodes = rng.integers(W // 2, T + 1, size=B).astype(np.int32)
    idx = np.full((B, W), -1, np.int32)
    for b in range(B):
        rows = rng.permutation(n_nodes[b])[:W]
        idx[b, :len(rows)] = rows
        idx[b, rng.random(W) < 0.2] = -1                                          # -1: the request's last live row
    count = rng.integers(1, W + 1, size=B).astype(np.int32)
    count[[2, 7]] = 0
    done = np.zeros(B, np.uint8)
    done[[4, 9]] = 1
    tokens = rng.integers(0, V, size=(B, W)).astype(np.int32)
    nxt = rng.integers(0, V, size=B).astype(np.int32)
    row_of = lambda b, j: n_nodes[b] - 1 if idx[b, j] < 0 else idx[b, j]
    # a -inf row (half of it, the targets included) and a row with one NaN
    r_inf, r_nan = row_of(0, 0), row_of(1, 1)
    count[0], count[1] = max(count[0], 2), max(count[1], 2)
    lg[0, r_inf, ::2] = float("-inf")
    tokens[0, 1] = 4
    lg[1, r_nan, 17] = NAN
    cu = lambda a: torch.as_tensor(a).cuda()
    ver = E.Verifier(B, T)
    for n_top in (0, 3, 8):
        out = dict(logprob=torch.full((B, W), NAN, device="cuda"), next_logprob=torch.full((B,), NAN, device="cuda"))
        if n_top:
            out.update(top_ids=torch.full((B, W, n_top), -7, dtype=torch.int32, device="cuda"),
                       top_logprob=torch.full((B, W, n_top), NAN, device="cuda"),
                       next_top_ids=torch.full((B, n_top), -7, dtype=torch.int32, device="cuda"),
                       next_top_logprob=torch.full((B, n_top), NAN, device="cuda"))
        got = ver.token_logprobs(lg, cu(idx), cu(count), cu(tokens), cu(nxt), n_top=n_top, n_nodes=cu(n_nodes),
                                 done=cu(done), out=out)
        assert got is out
        res = {k: v.cpu().numpy() for k, v in out.items()}
        rows32 = lg.float()
        ref = torch.log_softmax(rows32, -1).cpu().numpy()
        rows_np = rows32.cpu().numpy()
        for b in range(B):
            a = 0 if done[b] else count[b]
            for j in range(W):
                last = j == a - 1
                lp = res["next_logprob"][b] if last else res["logprob"][b, j]
                if j >= a:
                    assert np.isnan(res["logprob"][b, j]), (b, j)
                    if n_top:
                        assert (res["top_ids"][b, j] == -7).all() and np.isnan(res["top_logprob"][b, j]).all(), (b, j)
                    continue
                r = row_of(b, j)
                target = nxt[b] if last else tokens[b, j + 1]
                assert _close(lp, ref[b, r, target], 2e-5), (n_top, b, j, lp, ref[b, r, target])
                if last and j + 1 < W:
                    assert np.isnan(res["logprob"][b, j]), (b, j)
                if n_top:
                    ids = res["next_top_ids"][b] if last else res["top_ids"][b, j]
                    tlp = res["next_top_logprob"][b] if last else res["top_logprob"][b, j]
                    assert ids.tolist() == O.row_topk(rows_np[b, r], n_top).tolist(), (n_top, b, j)
                    assert _close(tlp, ref[b, r, ids], 2e-5), (n_top, b, j)
            if a == 0:
                assert np.isnan(res["next_logprob"][b]), b
                if n_top:
                    assert (res["next_top_ids"][b] == -7).all(), b
        assert res["logprob"][0, 0] == -np.inf                                    # target 4 sits on a -inf logit
        assert np.isnan(res["next_logprob"][1] if count[1] == 2 else res["logprob"][1, 1])   # the row with a NaN


# ---- 2. determinism ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt,V", [("fp32", 997), ("bf16", 997), ("bf16", 32000), ("bf16", 128256)])
def test_same_row_gives_bit_identical_results(dt, V):
    """One row at different (b, j), at B = 3 and 17, at different alignments (V = 997: 16-byte loads or element loads),
    and in a captured-and-replayed launch."""
    from samd_b200 import engine as E
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16}[dt]
    g = torch.Generator(device="cuda").manual_seed(3)
    row = (torch.randn(V, generator=g, device="cuda") * 4.0).to(tdt)
    tgt = 123
    outs = []
    for B, T, places in ((3, 5, [(0, 0), (1, 3), (2, 4)]), (17, 9, [(5, 1), (11, 8), (16, 6)])):
        lg = (torch.randn(B, T, V, generator=g, device="cuda") * 4.0).to(tdt)
        W = T
        idx = torch.arange(W, dtype=torch.int32, device="cuda").repeat(B, 1).contiguous()
        count = torch.full((B,), W, dtype=torch.int32, device="cuda")
        toks = torch.full((B, W), tgt, dtype=torch.int32, device="cuda")
        nxt = torch.full((B,), tgt, dtype=torch.int32, device="cuda")
        for b, r in places:
            lg[b, r] = row
        ver = E.Verifier(B, T)
        eager = ver.token_logprobs(lg, idx, count, toks, nxt, n_top=8)
        gout = ver.token_logprobs(lg, idx, count, toks, nxt, n_top=8)
        for v in gout.values():
            v.zero_()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ver.token_logprobs(lg, idx, count, toks, nxt, n_top=8, out=gout)
        graph.replay()
        torch.cuda.synchronize()
        for res in (eager, gout):
            for b, r in places:
                # position r - 1 is scored on row r - 1; the row at r is scored at position r (target tokens[b][r + 1]
                # or next_token: both tgt)
                last = r == W - 1
                lp = res["next_logprob"][b] if last else res["logprob"][b, r]
                ids = res["next_top_ids"][b] if last else res["top_ids"][b, r]
                tl = res["next_top_logprob"][b] if last else res["top_logprob"][b, r]
                outs.append((lp.view(torch.int32).item(), ids.tolist(), tl.view(torch.int32).tolist()))
    assert all(o == outs[0] for o in outs), outs
    ref = torch.log_softmax(row.float(), -1)[tgt].item()
    assert abs(torch.tensor(outs[0][0], dtype=torch.int32).view(torch.float32).item() - ref) <= 2e-5


# ---- 3. the decoders against a teacher-forced forward -----------------------------------------------------------------
def _serve(dec, prompts, limits, **kw):
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info)
    assert sorted(got) == list(range(len(prompts)))
    return got


@torch.inference_mode()
def _teacher_check(lm, prompt, tokens, info, n):
    """info["logprobs"] (and top_logprobs) against log_softmax of one forward over prompt + tokens; returns the number
    of top-n lists compared."""
    assert len(info["logprobs"]) == len(tokens)
    ids = torch.as_tensor([prompt + tokens]).cuda()
    rows = lm(input_ids=ids).logits[0, len(prompt) - 1:len(prompt) - 1 + len(tokens)].float()
    ref = torch.log_softmax(rows, -1).cpu().numpy()
    want = ref[np.arange(len(tokens)), tokens]
    assert np.abs(np.asarray(info["logprobs"]) - want).max() <= 1e-4, np.abs(np.asarray(info["logprobs"]) - want).max()
    if not n:
        assert "top_logprobs" not in info
        return 0
    assert len(info["top_logprobs"]) == len(tokens) and all(len(t) == n for t in info["top_logprobs"])
    rows_np = rows.cpu().numpy()
    srt = -np.sort(-rows_np, -1)
    compared = 0
    for k, top in enumerate(info["top_logprobs"]):
        if (srt[k, :n] - srt[k, 1:n + 1]).min() <= 1e-4:                  # order within 1e-4: not well defined
            continue
        compared += 1
        assert [t for t, _ in top] == O.row_topk(rows_np[k], n).tolist(), k
        assert np.abs(np.asarray([v for _, v in top]) - ref[k, [t for t, _ in top]]).max() <= 1e-4, k
    return compared


@pytest.mark.parametrize("mode", ["samd", "samd_tree", "sam_only", "samd_sampled", "sam_only_sampled"])
def test_logprobs_match_a_teacher_forced_forward(lm, work, mode):
    """serve() at B = 4 over 13 requests with refills, logprobs=8; a prefix pool with a prompt equal to its prefix; EOS
    truncation."""
    from samd_b200 import synth
    prompts, limits, params = work
    flavour = mode.split("_sampled")[0].replace("_tree", "")
    mk = _decoders(lm)[flavour]
    kw = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    sampling = params if mode.endswith("sampled") else None
    dec = mk(4, **kw)
    got = _serve(dec, prompts, limits, sampling=sampling, logprobs=8)
    assert dec.serve_stats["graphed"]
    compared = total = 0
    for i in range(N_REQ):
        compared += _teacher_check(lm, prompts[i], got[i][0], got[i][1], 8)
        total += len(got[i][0])
    assert compared >= total // 3, (compared, total)
    pooled = mk(4, max_prefixes=2, **kw)
    pooled.add_prefix(prompts[1])
    pooled.add_prefix(prompts[6][:40])
    pgot = _serve(pooled, prompts, limits, sampling=sampling, logprobs=2)
    assert pgot[1][1]["prefix_len"] == len(prompts[1]) and pgot[6][1]["prefix_len"] == 40
    for i in range(N_REQ):
        assert pgot[i][0] == got[i][0], i
        _teacher_check(lm, prompts[i], pgot[i][0], pgot[i][1], 2)
    counts = np.bincount(np.concatenate([got[i][0] for i in range(N_REQ)]), minlength=96)
    eos = int(counts.argmax())
    egot = _serve(mk(4, eos_token_id=eos, **kw), prompts, limits, sampling=sampling, logprobs=0)
    cut = 0
    for i in range(N_REQ):
        w = got[i][0]
        want = w[:w.index(eos) + 1] if eos in w else w
        cut += len(want) < len(w)
        assert egot[i][0] == want, i
        _teacher_check(lm, prompts[i], egot[i][0], egot[i][1], 0)
        assert _close(egot[i][1]["logprobs"], got[i][1]["logprobs"][:len(want)], 1e-5), i
    assert cut >= 2


# ---- 4. nothing else changes ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
@pytest.mark.parametrize("sampled", [False, True])
def test_logprobs_change_nothing_else(lm, work, flavour, sampled):
    from samd_b200 import engine as E
    prompts, limits, params = work
    sampling = params if sampled else None
    mk = _decoders(lm)[flavour]
    dec = mk(4)
    base = _serve(dec, prompts, limits, sampling=sampling)
    with0 = _serve(dec, prompts, limits, sampling=sampling, logprobs=0)
    with8 = _serve(dec, prompts, limits, sampling=sampling, logprobs=8)
    for i in range(N_REQ):
        assert "logprobs" not in base[i][1]
        for other in (with0, with8):
            assert other[i][0] == base[i][0] and other[i][1]["accept_lengths"] == base[i][1]["accept_lengths"], i
        assert _close(with0[i][1]["logprobs"], with8[i][1]["logprobs"], 1e-6), i
    # graphed and eager, check_every 1 and 4, generate() and serve(): the same log-probabilities
    eager = _serve(dec, prompts, limits, sampling=sampling, logprobs=8, graph=False)
    every1 = _serve(dec, prompts, limits, sampling=sampling, logprobs=8, check_every=1)
    for i in range(N_REQ):
        for other in (eager, every1):
            assert other[i][0] == with8[i][0], i
            assert _close(other[i][1]["logprobs"], with8[i][1]["logprobs"], 1e-6), i
            assert [[t for t, _ in x] for x in other[i][1]["top_logprobs"]] == \
                   [[t for t, _ in x] for x in with8[i][1]["top_logprobs"]], i
    sub = prompts[4:8]
    sp = params[4:8] if sampled else None
    out, st = dec.generate(sub, 24, sampling=sp, logprobs=8)
    ref = _serve(dec, sub, [24] * 4, sampling=sp, logprobs=8)
    for k in range(4):
        assert out[k] == ref[k][0]
        assert _close(st["logprobs"][k], ref[k][1]["logprobs"], 1e-6), k
        assert [[t for t, _ in x] for x in st["top_logprobs"][k]] == [[t for t, _ in x] for x in ref[k][1]["top_logprobs"]]
    # launches, eager: logprobs=0 adds one per step and one per admission batch; None issues the step's launches only
    # step + verify; sam_only adds the static tree draft and the assembly, and sampled, samd_kv_compact (row moves and the
    # length bump: two launches)
    per_step = {("samd", False): 2, ("samd", True): 2, ("sam_only", False): 4, ("sam_only", True): 6}[flavour, sampled]
    runs = {}
    for lp in (None, 0):
        for n_new in (16, 40):
            c0 = E.launch_count()
            _, st = dec.generate(sub, n_new, sampling=sp, graph=False, logprobs=lp)
            runs[lp, n_new] = (E.launch_count() - c0, st["steps_run"])
    for n_new in (16, 40):
        (c_none, s_none), (c_lp, s_lp) = runs[None, n_new], runs[0, n_new]
        assert s_none == s_lp and c_lp - c_none == s_none + 1, (n_new, runs)
    (c1, s1), (c2, s2) = runs[None, 16], runs[None, 40]
    assert s2 > s1 and c2 - c1 == per_step * (s2 - s1), runs
