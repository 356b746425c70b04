"""GPU tests of stop sequences: samd_stop_match against a Python restatement (widths 1 to 256, sequences straddling the
history / candidate boundary, ending at count - 1 and at count, overlapping themselves, ties and duplicates, finished
requests, empty tables, an aliased out_count, a captured launch), and the decoders' stop= in every mode: tokens are the
unstopped run's cut at the earliest stop, with the finish reason, the stop index, the accept lengths and the
log-probabilities that go with it, the same across execution variants; EOS, the cache guard, stop=None and fewer steps."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N_REQ = 13
V_LM = 96
S, L = 16, 16


# ---- the restatement ----------------------------------------------------------------------------------------------------
def _earliest(hist, cand, seqs):
    """(e, j): the earliest candidate position e where a sequence of `seqs` ends, matched against the output hist + cand
    (never before output position 0), and the lowest such j; None without a match."""
    out = list(hist) + list(cand)
    for i in range(len(cand)):
        end = len(hist) + i
        for j, s in enumerate(seqs):
            if s and end - len(s) + 1 >= 0 and out[end - len(s) + 1:end + 1] == list(s):
                return i, j
    return None


def _restate(tokens, count, hist, hist_len, stop_tok, stop_len, done):
    B, W = tokens.shape
    out_c, out_h = count.copy(), np.full(B, -1, np.int32)
    for b in range(B):
        if (done is not None and done[b]) or count[b] <= 0:
            continue
        seqs = [list(stop_tok[b, j, :stop_len[b, j]]) for j in range(S)]
        m = _earliest(hist[b, :hist_len[b]], tokens[b, :min(count[b], W)], seqs)
        if m is not None:
            out_c[b], out_h[b] = m[0] + 1, m[1]
    return out_c, out_h


def _batch(rng, W, B=48):
    """A random batch with planted sequences; tokens from a small alphabet so that chance matches occur too."""
    H = 48
    tokens = rng.integers(1, 6, size=(B, W)).astype(np.int32)
    hist = rng.integers(1, 6, size=(B, H)).astype(np.int32)
    hist_len = rng.integers(0, 41, size=B).astype(np.int32)
    hist_len[:6] = [0, 1, 3, 14, 15, 16]
    count = rng.integers(0, W + 1, size=B).astype(np.int32)
    count[6:9] = [0, W, min(1, W)]
    stop_tok = np.zeros((B, S, L), np.int32)
    stop_len = np.zeros((B, S), np.int32)
    done = np.zeros(B, np.uint8)
    done[rng.choice(B, size=4, replace=False)] = 1
    for b in range(B):
        if b % 7 == 3:
            continue                                            # no sequences
        hl, c = int(hist_len[b]), int(count[b])
        tokens[b, c:] = 9                                       # tokens at or past count: never read
        seqs = []
        if c >= 6 and b % 3 == 0:                               # overlaps itself in a run
            x = int(rng.integers(0, c - 5))
            tokens[b, x:x + 5] = 7
            seqs.append([7, 7, 7])
        full = [int(t) for t in hist[b, :hl]] + [int(t) for t in tokens[b]]
        if hl and c:                                            # straddles the boundary
            a, k = int(rng.integers(1, min(hl, 8) + 1)), int(rng.integers(1, min(c, 8) + 1))
            seqs.append(full[hl - a:hl + k])
        if c:                                                   # ends exactly at count - 1
            n = int(rng.integers(1, min(hl + c, 16) + 1))
            seqs.append(full[hl + c - n:hl + c])
        if c < W:                                               # ends at count: must not fire
            n = int(rng.integers(1, min(hl + c + 1, 16) + 1))
            seqs.append(full[hl + c + 1 - n:hl + c + 1])
        if seqs and b % 4 == 1:                                 # the same end twice (a suffix), and a duplicate
            seqs.append(seqs[0][-max(1, len(seqs[0]) // 2):])
            seqs.append(list(seqs[0]))
        if b % 5 == 2:                                          # would need output position -1
            seqs.append([8] + full[:min(2, hl + c)])
        seqs += [[int(t) for t in rng.integers(1, 6, size=int(rng.integers(1, 17)))] for _ in range(int(rng.integers(0, 4)))]
        seqs = [s for s in seqs if 1 <= len(s) <= L][:S]
        order = rng.permutation(len(seqs))
        for j, o in enumerate(order):
            s = seqs[o]
            stop_tok[b, j, :len(s)] = s
            stop_len[b, j] = len(s)
        if b % 11 == 5:                                         # an unused entry between used ones
            stop_len[b, 0] = 0
    return tokens, count, hist, hist_len, stop_tok, stop_len, done


@pytest.mark.parametrize("W", [1, 16, 61, 128, 256])
def test_kernel_matches_restatement(W):
    from samd_b200 import engine as E
    cu = lambda a: torch.as_tensor(a).cuda()
    hits = 0
    for seed in range(4):
        rng = np.random.default_rng(1000 * W + seed)
        tokens, count, hist, hist_len, stop_tok, stop_len, done = _batch(rng, W)
        want_c, want_h = _restate(tokens, count, hist, hist_len, stop_tok, stop_len, done)
        hits += int((want_h >= 0).sum())
        args = [cu(x) for x in (tokens, count, hist, hist_len, stop_tok, stop_len)]
        c, h = E.match_stops(*args, done=cu(done))
        assert np.array_equal(c.cpu().numpy(), want_c) and np.array_equal(h.cpu().numpy(), want_h), seed
        # without done, and with out_count aliasing count
        want_c2, want_h2 = _restate(tokens, count, hist, hist_len, stop_tok, stop_len, None)
        cnt = args[1].clone()
        hit = torch.full_like(cnt, 5)
        c2, h2 = E.match_stops(args[0], cnt, *args[2:], out_count=cnt, out_hit=hit)
        assert c2 is cnt and h2 is hit
        assert np.array_equal(cnt.cpu().numpy(), want_c2) and np.array_equal(hit.cpu().numpy(), want_h2), seed
        # a captured launch equals the eager one
        oc, oh = torch.zeros_like(cnt), torch.zeros_like(cnt)
        d = cu(done)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            E.match_stops(*args, done=d, out_count=oc, out_hit=oh)
        oc.zero_()
        oh.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(oc, c) and torch.equal(oh, h)
    assert hits >= 8


# ---- the decoders -------------------------------------------------------------------------------------------------------
MODES = ["samd", "samd_tree", "samd_sampled", "sam_only", "sam_only_sampled"]


def _tiny_llama():
    """An fp32 tiny Llama whose head never prefers token 0 (bias -30): the decoy stop sequences use it."""
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=V_LM, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
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
    lens = (150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70)
    prompts = [synth.copy_mix(n, V_LM, 300 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    limits = [8, 96] + [8 + (37 * i) % 89 for i in range(2, N_REQ)]
    return prompts, limits


def _maker(lm, mode, max_len=512):
    from samd_b200 import engine as E, synth
    from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
    if mode.startswith("sam_only"):
        docs = [synth.copy_mix(300, V_LM, 5 + k).tolist() for k in range(3)] + [[i] for i in range(3, V_LM)]
        static = E.StaticSamDevice.build(docs, 2, with_counts=True)
        return lambda B, **kw: BatchedSamOnlyDecoder(lm, B, max_len, max_predicts=16, alpha=4.0, K=4, len_bias=0,
                                                     static=static, dtype=torch.float32, **kw)
    tree = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    return lambda B, **kw: BatchedSamdDecoder(lm, B, max_len, n_predicts=8, len_bias=5, len_threshold=3,
                                              dtype=torch.float32, **tree, **kw)


def _sampling(mode):
    from samd_b200.batched import SamplingParams
    if not mode.endswith("sampled"):
        return None
    procs = [dict(temperature=1.0), dict(temperature=0.7, top_p=0.9), dict(temperature=1.3, top_k=5), dict(greedy=True)]
    return [SamplingParams(seed=1000 + 7 * i, **procs[i % len(procs)]) for i in range(N_REQ)]


def _serve(dec, prompts, limits, **kw):
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info)
    assert sorted(got) == list(range(len(prompts)))
    return got


DECOYS = [[0], [0, 0, 0], [0] * 15 + [1]]


def _plant(i, prompt, u, acc, limit):
    """Request i's stop sequences, planted from its unstopped output u (accept lengths acc) by kind i % 6, with decoys
    that never occur mixed in."""
    starts = np.concatenate([[0], np.cumsum(acc)]).astype(int)
    kind = i % 6
    seq = None
    if kind == 0:                                               # ends inside a step
        k = next((k for k in range(len(acc)) if acc[k] >= 2 and starts[k] + acc[k] - 2 < len(u)), None)
        if k is not None:
            e = starts[k] + acc[k] - 2
            seq = u[max(0, e - 5):e + 1]
    elif kind == 1:                                             # straddles a step boundary
        k = next((k for k in range(1, len(acc)) if 2 <= starts[k] < len(u)), None)
        if k is not None:
            e = starts[k]
            seq = u[max(0, e - 5):e + 1]
    elif kind == 2:                                             # the first output token
        seq = u[:1]
    elif kind == 3 and len(u) == limit:                         # ends exactly at max_new_tokens
        seq = u[max(0, limit - 4):limit]
    elif kind == 4:                                             # would end one token past it
        seq = u[max(0, limit - 3):limit] + [u[-1]]
    elif kind == 5:                                             # starts in the prompt
        seq = prompt[-2:] + u[:2]
    seqs = [d for d in DECOYS[:i % 3]] + ([seq] if seq else []) + DECOYS[i % 3:i % 3 + 1]
    return seqs


def _expect(u, seqs):
    m = _earliest([], u, seqs)
    return (len(u), None) if m is None else (m[0] + 1, m[1])


def _check(got, base, seqs_of, limits, mode, eos=None):
    """Every request of `got` (stopped) against `base` (unstopped): tokens, finish reason, stop index, accept lengths.
    Returns the (inside a step, straddling) counts of the stops that fired."""
    from samd_b200.batched import StopSequences  # noqa: F401
    inside = straddle = 0
    for i in range(len(base)):
        u, info_u = base[i]
        tokens, info = got[i]
        n, j = _expect(u, seqs_of[i])
        assert tokens == u[:n], (mode, i, tokens, u, seqs_of[i])
        assert info["stop_index"] == j, (mode, i, info["stop_index"], j)
        if j is not None:
            assert info["finish_reason"] == "stop", (mode, i)
        else:
            assert info["finish_reason"] == info_u["finish_reason"], (mode, i)
            want = "stop" if eos is not None and u and u[-1] == eos else "length" if len(u) >= limits[i] else "cache"
            assert info_u["finish_reason"] == want, (mode, i)
        hist = info["accept_lengths"]
        if j is not None:
            assert sum(hist) == n, (mode, i)
        if mode == "samd_tree":                                   # the shared successor table: drafts depend on neighbours
            continue
        acc = info_u["accept_lengths"]
        if j is None:
            assert hist == acc, (mode, i)
            continue
        starts = np.concatenate([[0], np.cumsum(acc)]).astype(int)
        k = int(np.searchsorted(starts, n - 1, side="right")) - 1          # the step that emitted position n - 1
        assert hist == acc[:k] + [n - starts[k]], (mode, i, hist, acc, n)
        inside += n - starts[k] < acc[k]
        straddle += n - len(seqs_of[i][j]) < starts[k]
    return inside, straddle


@pytest.mark.parametrize("mode", MODES)
def test_stops_cut_the_unstopped_output(lm, work, mode):
    from samd_b200.batched import Penalties, StopSequences
    prompts, limits = work
    sp = _sampling(mode)
    mk = _maker(lm, mode)
    dec = mk(4)
    base = _serve(dec, prompts, limits, sampling=sp)
    assert all(base[i][1]["finish_reason"] == "length" for i in range(N_REQ))
    seqs_of = [_plant(i, prompts[i], base[i][0], base[i][1]["accept_lengths"], limits[i]) for i in range(N_REQ)]
    stops = [StopSequences(s) for s in seqs_of]
    got = _serve(dec, prompts, limits, sampling=sp, stop=stops)
    inside, straddle = _check(got, base, seqs_of, limits, mode)
    fired = sum(got[i][1]["stop_index"] is not None for i in range(N_REQ))
    assert fired >= 4 and any(got[i][1]["finish_reason"] == "length" for i in range(N_REQ)), mode
    assert got[2][1]["stop_index"] is not None and len(got[2][0]) == 1          # the first output token
    if mode in ("samd", "sam_only"):                              # (sampled drafts are accepted less often)
        assert inside >= 1 and straddle >= 1, (mode, inside, straddle)
    elif mode != "samd_tree":
        assert inside + straddle >= 1, (mode, inside, straddle)

    # the same results in every execution variant
    def same(other, what):
        for i in range(N_REQ):
            a, b = other[i], got[i]
            assert a[0] == b[0], (mode, what, i)
            for key in ("finish_reason", "stop_index"):
                assert a[1][key] == b[1][key], (mode, what, i, key)
            if mode != "samd_tree":
                assert a[1]["accept_lengths"] == b[1]["accept_lengths"], (mode, what, i)
    same(_serve(dec, prompts, limits, sampling=sp, stop=stops, graph=False, check_every=1), "eager, check_every 1")
    assert dec.serve_stats["graphed"] is False
    same(_serve(dec, prompts, limits, sampling=sp, stop=stops, check_every=1), "graphed, check_every 1")
    same(_serve(mk(1), prompts, limits, sampling=sp, stop=stops), "B = 1")
    pooled = mk(4, max_prefixes=2)
    pooled.add_prefix(prompts[1])
    pooled.add_prefix(prompts[6][:40])
    pgot = _serve(pooled, prompts, limits, sampling=sp, stop=stops)
    assert pgot[1][1]["prefix_len"] == len(prompts[1]) and pgot[6][1]["prefix_len"] == 40
    same(pgot, "prefix pool")
    sub = slice(4, 8)
    gsp = None if sp is None else sp[sub]
    out0, st0 = dec.generate(prompts[sub], 24, sampling=gsp)
    out, st = dec.generate(prompts[sub], 24, sampling=gsp, stop=stops[sub])
    assert st0["finish_reasons"] == ["length"] * 4 and "stop_indices" not in st0
    for k, i in enumerate(range(4, 8)):
        n, j = _expect(out0[k], seqs_of[i])
        assert out[k] == out0[k][:n] and st["stop_indices"][k] == j, (mode, i)
        assert st["finish_reasons"][k] == ("stop" if j is not None else "length"), (mode, i)

    # log-probabilities (and penalties) are a prefix of the unstopped run's
    pens = [Penalties(repetition_penalty=1.2), Penalties(), Penalties(presence_penalty=0.4, frequency_penalty=0.3)]
    pens = [pens[i % 3] for i in range(N_REQ)]
    lbase = _serve(dec, prompts, limits, sampling=sp, penalties=pens, logprobs=2)
    lseqs = [_plant(i, prompts[i], lbase[i][0], lbase[i][1]["accept_lengths"], limits[i]) for i in range(N_REQ)]
    lgot = _serve(dec, prompts, limits, sampling=sp, penalties=pens, logprobs=2, stop=[StopSequences(s) for s in lseqs])
    _check(lgot, lbase, lseqs, limits, mode)
    for i in range(N_REQ):
        n = len(lgot[i][0])
        a, b = lgot[i][1], lbase[i][1]
        assert len(a["logprobs"]) == n
        assert np.allclose(a["logprobs"], b["logprobs"][:n], rtol=0, atol=1e-5), (mode, i)
        assert [[t for t, _ in top] for top in a["top_logprobs"]] == [[t for t, _ in top] for top in b["top_logprobs"][:n]]


def test_eos_and_cache(lm, work):
    from samd_b200.batched import StopSequences
    prompts, limits = work
    mk = _maker(lm, "samd")
    base = _serve(mk(4), prompts, limits)
    counts = np.bincount(np.concatenate([base[i][0] for i in range(N_REQ)]), minlength=V_LM)
    eos = int(counts.argmax())
    edec = mk(4, eos_token_id=eos)
    ebase = _serve(edec, prompts, limits)
    cut = [i for i in range(N_REQ) if eos in base[i][0] and base[i][0].index(eos) >= 1]
    assert len(cut) >= 2
    for i in cut:
        assert ebase[i][0] == base[i][0][:base[i][0].index(eos) + 1] and ebase[i][1]["finish_reason"] == "stop"
    # a stop ending on EOS fires (stop_index set); a stop after the EOS does not (EOS ends it, stop_index None)
    seqs = {}
    for i in range(N_REQ):
        u = base[i][0]
        if i in cut[::2]:
            p = u.index(eos)
            seqs[i] = [[0], u[p - 1:p + 1]]
        elif i in cut:                                           # starts on the EOS, ends after it
            p = u.index(eos)
            seqs[i] = [u[p:p + 2] if p + 2 <= len(u) else [eos, 1]]
        else:
            seqs[i] = []
    got = _serve(edec, prompts, limits, stop=[StopSequences(seqs[i]) for i in range(N_REQ)])
    for i in range(N_REQ):
        assert got[i][0] == ebase[i][0], i
        assert got[i][1]["finish_reason"] == ebase[i][1]["finish_reason"], i
        assert got[i][1]["stop_index"] == (1 if i in cut[::2] else None), i
    # a small cache: the guard ends the long requests first
    small = _maker(lm, "samd", max_len=224)(4)
    cgot = _serve(small, prompts, limits, stop=StopSequences([[0]]))
    reasons = [cgot[i][1]["finish_reason"] for i in range(N_REQ)]
    assert "cache" in reasons and "length" in reasons, reasons
    for i in range(N_REQ):
        tokens, info = cgot[i]
        assert tokens == base[i][0][:len(tokens)] and info["stop_index"] is None, i
        assert info["finish_reason"] == ("length" if len(tokens) == limits[i] else "cache"), i
        if info["finish_reason"] == "cache":
            assert len(prompts[i]) + len(tokens) + 2 * 8 > 224, i


@pytest.mark.parametrize("mode", ["samd", "sam_only"])
def test_none_and_empty_stops(lm, work, mode):
    from samd_b200 import engine as E
    from samd_b200.batched import StopSequences
    prompts, limits = work
    dec = _maker(lm, mode)(4)
    base = _serve(dec, prompts, limits)
    stats = dict(dec.serve_stats)
    none = _serve(dec, prompts, limits, stop=None)
    assert "stop_tok" not in dec._st                              # stop=None allocates nothing
    assert dec.serve_stats["steps_run"] == stats["steps_run"] and dec.serve_stats["graphs"] == stats["graphs"]
    empty = _serve(dec, prompts, limits, stop=StopSequences(()))
    for i in range(N_REQ):
        assert none[i][0] == base[i][0] and empty[i][0] == base[i][0], i
        assert "stop_index" not in none[i][1] and empty[i][1]["stop_index"] is None, i
        assert empty[i][1]["accept_lengths"] == base[i][1]["accept_lengths"], i
    again = _serve(dec, prompts, limits)
    assert dec.serve_stats["steps_run"] == stats["steps_run"]
    assert all(again[i][0] == base[i][0] for i in range(N_REQ))
    # launches, eager: stops add one per step; None issues the step's launches only
    runs = {}
    for ss in (None, StopSequences(())):
        c0 = E.launch_count()
        _, st = dec.generate(prompts[4:8], 24, graph=False, stop=ss)
        runs[ss is None] = (E.launch_count() - c0, st["steps_run"])
    (c_none, s_none), (c_stop, s_stop) = runs[True], runs[False]
    assert s_none == s_stop and c_stop - c_none == s_none, runs


@pytest.mark.parametrize("mode", ["samd", "sam_only_sampled"])
def test_early_stops_run_fewer_steps(lm, work, mode):
    from samd_b200.batched import StopSequences
    prompts, limits = work
    sp = _sampling(mode)
    dec = _maker(lm, mode)(4)
    base = _serve(dec, prompts, limits, sampling=sp)
    steps, live = dec.serve_stats["steps_run"], dec.serve_stats["live_slot_steps"]
    stops = [StopSequences([base[i][0][min(3, len(base[i][0]) - 1):][:2]]) for i in range(N_REQ)]
    got = _serve(dec, prompts, limits, sampling=sp, stop=stops)
    assert dec.serve_stats["steps_run"] < steps and dec.serve_stats["live_slot_steps"] < live
    for i in range(N_REQ):
        n, j = _expect(base[i][0], stops[i].sequences)
        assert got[i][0] == base[i][0][:n] and got[i][1]["stop_index"] == j, i
