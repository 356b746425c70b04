"""GPU tests of logit controls: samd_apply_logit_controls against a torch restatement, bit for bit (identity chains and
random trees, done and neutral requests, rows off every path, the admission form, -inf and NaN, biased and banned ids,
bad words straddling history and path, heads reaching before output position 0, the min_tokens boundary, stop heads,
graph and eager), and the decoders' controls= against plain controlled greedy decoding, min_tokens with an EOS bias,
sampled decoding that never emits a banned token, None and neutral controls, and log-probabilities of controlled rows."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N_REQ = 13
V_LM = 96
NAN = float("nan")
INF = math.inf


def _tiny_llama(head_scale: float = 1.0):
    """The fp32 tiny Llama of the log-probability tests: token 0 is never its argmax (a -30 head bias), so a -1 pad of a
    path table is never "accepted" (the reference's A9 corner, see BatchedSamOnlyDecoder)."""
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=V_LM, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, max_position_embeddings=2048, attn_implementation="eager")
    lm = LlamaForCausalLM(cfg).to("cuda", torch.float32).eval()
    head = torch.nn.Linear(cfg.hidden_size, cfg.vocab_size, bias=True).to("cuda")
    with torch.no_grad():
        head.weight.copy_(lm.lm_head.weight * head_scale)
        head.bias.zero_()
        head.bias[0] = -30.0 * head_scale
    lm.lm_head = head
    return lm


# ---- the torch restatement ----------------------------------------------------------------------------------------------
def _ends_with(ctx, head) -> bool:
    return len(head) <= len(ctx) and list(ctx[len(ctx) - len(head):]) == list(head)


def _control_row(x: torch.Tensor, ctx, pos: int, bias, bad, m: int, eos, stops) -> tuple:
    """One logits row [V] (any dtype) predicting output position `pos` after the output context `ctx`: each finite bias
    one fp32 add and one rounding into the row's dtype, then -inf on every ban.  Returns (row, multi-token matches)."""
    y = x.clone()
    ban, multi = set(), 0
    for t, v in bias:
        if v == -INF:
            ban.add(t)
        else:
            y[t] = (x[t].float() + torch.tensor(np.float32(v), device=x.device)).to(x.dtype)
    heads = [(s, False) for s in bad] + ([(s, True) for s in stops] if pos < m else [])
    for s, _ in heads:
        if _ends_with(ctx, s[:-1]):
            ban.add(s[-1])
            multi += len(s) > 1
    if pos < m and eos is not None:
        ban.add(eos)
    if ban:
        y[torch.tensor(sorted(ban), device=x.device)] = -INF
    return y, multi


def _paths(ret_b, n, n_paths):
    """{row j: path node list 0 .. j} from the first (path, depth) listing j, each path ending at its first -1."""
    out = {}
    for p in range(n_paths):
        for d in range(ret_b.shape[1]):
            j = int(ret_b[p, d])
            if j < 0:
                break
            if j < n and j not in out:
                out[j] = [int(k) for k in ret_b[p, :d + 1]]
    return out


def _restate(lg, ctl, tokens=None, ret=None, n_nodes=None, n_paths=None, done=None, slots=None, hist=None,
             hist_len=None, stops=None, eos=None):
    """ctl: per state row (bias pairs, bad words, min_tokens); stops: per state row lists (or None)."""
    want, matches = lg.clone(), 0
    B, T, V = lg.shape
    for b in range(B):
        s = b if slots is None else int(slots[b])
        bias, bad, m = ctl[s]
        st = stops[s] if stops is not None else []
        if (done is not None and done[b]) or not (bias or bad or (m > 0 and (eos is not None or st))):
            continue
        n = T if n_nodes is None else min(T, int(n_nodes[b]))
        hl = 0 if hist_len is None else int(hist_len[s])
        h = [int(t) for t in hist[s, :hl]] if hl else []
        if tokens is None:
            rows = {j: [] for j in range(n)}
        elif ret is None:
            rows = {j: list(range(j + 1)) for j in range(n)}
        else:
            rows = _paths(ret[b], n, ret.shape[1] if n_paths is None else int(n_paths[b]))
        for j, nodes in rows.items():
            ctx = h + [int(tokens[b, k]) for k in nodes]
            pos = hl + len(nodes) if tokens is not None else hl
            want[b, j], k = _control_row(lg[b, j], ctx, pos, bias, bad, m, eos, st)
            matches += k
    return want, matches


def _same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    """Bit-identical, except that any NaN matches any NaN."""
    ia = a.view(torch.int32 if a.dtype == torch.float32 else torch.int16)
    ib = b.view(ia.dtype)
    return bool(((ia == ib) | (torch.isnan(a) & torch.isnan(b))).all())


def _random_tree(rng, n):
    parent = [-1] + [int(rng.integers(0, j)) for j in range(1, n)]
    kids = {j for j in parent if j >= 0}
    paths = []
    for leaf in (j for j in range(n) if j not in kids):
        path = [leaf]
        while parent[path[-1]] >= 0:
            path.append(parent[path[-1]])
        paths.append(path[::-1])
    return paths


def _tables(ctl, stops, dev="cuda"):
    """Device tables of per-state-row controls (and stops)."""
    S = len(ctl)
    ids, bias, bn = np.zeros((S, 256), np.int32), np.zeros((S, 256), np.float32), np.zeros(S, np.int32)
    bt, bl, mn = np.zeros((S, 16, 16), np.int32), np.zeros((S, 16), np.int32), np.zeros(S, np.int32)
    st, sl = np.zeros((S, 16, 16), np.int32), np.zeros((S, 16), np.int32)
    for s, (bi, bad, m) in enumerate(ctl):
        bn[s], mn[s] = len(bi), m
        for e, (t, v) in enumerate(bi):
            ids[s, e], bias[s, e] = t, v
        for k, w in enumerate(bad):
            bt[s, k, :len(w)], bl[s, k] = w, len(w)
        for k, w in enumerate(stops[s] if stops is not None else []):
            st[s, k, :len(w)], sl[s, k] = w, len(w)
    cu = lambda a: torch.as_tensor(a).to(dev)
    return [cu(x) for x in (ids, bias, bn, bt, bl, mn)], dict(stop_tokens=cu(st), stop_len=cu(sl))


# ---- 1. the kernel against the restatement ------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [997, 32000, 128256])
@pytest.mark.parametrize("dt", ["fp32", "bf16", "fp16"])
def test_kernel_matches_torch(dt, V):
    from samd_b200 import engine as E
    B, T, P, H = 12, 12, 12, 40
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[dt]
    rng = np.random.default_rng(V + len(dt))
    g = torch.Generator(device="cuda").manual_seed(V)
    lg = (torch.randn(B, T, V, generator=g, device="cuda") * 3.0).to(tdt)
    pool = [int(t) for t in rng.choice(V, size=6, replace=False)]       # a small pool: heads match often
    pick = lambda *sh: np.asarray(pool)[rng.integers(0, len(pool), size=sh)].astype(np.int32)
    tokens, hist = pick(B, T), pick(B, H)
    hist_len = rng.integers(0, H + 1, size=B).astype(np.int32)
    eos = pool[0]
    ctl, stops = [], []
    for b in range(B):
        ids = [t for t in rng.choice(V, size=int(rng.integers(1, 40)), replace=False).tolist() if t != pool[1]]
        bias = [(int(t), float(rng.choice([-100.0, -2.5, 0.75, 3.0, 100.0, -INF]))) for t in ids]
        bias.append((pool[1], 1.5))                                     # a biased id that is also a banned one
        bad = [[int(t) for t in pick(int(rng.integers(1, 5)))] for _ in range(int(rng.integers(1, 16)))]
        bad.append([pool[1]])
        st = [[int(t) for t in pick(int(rng.integers(1, 4)))] for _ in range(int(rng.integers(0, 6)))]
        ctl.append((bias, bad, int(hist_len[b]) + int(rng.integers(0, 5))))
        stops.append(st)
    ctl[3], stops[3] = ([], [], 0), []                                  # neutral
    ctl[4] = ([(t, 1.0) for t in rng.choice(V, size=256, replace=False).tolist()], [list(pool[:2]) * 8], ctl[4][2])
    # the min_tokens boundary on request 6 (a chain): node 0 predicts hl + 1 < m, node 1 predicts hl + 2 = m
    hist_len[6] = 20
    ctl[6] = ([], [], 22)
    stops[6] = [[int(tokens[6, 0]), pool[2]], [int(tokens[6, 1]), pool[3]]]
    # a bad word straddling history and path on request 1 (a tree): its head is the last history token and node 0
    hist_len[1] = 9
    # a head reaching before output position 0 on request 8: no history, a 3-id word whose head would need it
    hist_len[8] = 0
    ctl[8] = ([], [[pool[5], int(tokens[8, 0]), pool[3]], [int(tokens[8, 0]), pool[4]]], 0)
    hist[8] = pool[5]                                                   # (stale tokens past hist_len that would match)
    done = np.zeros(B, np.uint8)
    done[7] = 1
    n_nodes = rng.integers(T // 2, T + 1, size=B).astype(np.int32)
    n_nodes[[1, 6, 8, 9]] = T
    ret = np.full((B, P, T), -1, np.int32)
    n_paths = np.zeros(B, np.int32)
    for b in range(B):
        paths = _random_tree(rng, int(n_nodes[b])) if b % 3 == 1 else [list(range(int(n_nodes[b])))]
        n_paths[b] = len(paths)
        for k, path in enumerate(paths):
            ret[b, k, :len(path)] = path
    n_paths[10] = max(1, n_paths[10] - 1)                               # rows on no live path: a tree's last leaves, ...
    ret[9, 0, 8:] = -1                                                  # ... a chain's tail
    ctl[1] = (ctl[1][0], ctl[1][1][:14] + [[int(hist[1, 8]), int(tokens[1, 0]), pool[4]]], ctl[1][2])
    lg[0, :, ctl[0][0][0][0]] = -INF                                    # -inf and NaN inputs on biased ids
    lg[0, 2, ctl[0][0][1][0]] = NAN
    lg[2, 1, pool[1]] = NAN
    cu = lambda a: torch.as_tensor(a).cuda()
    tabs, stop_kw = _tables(ctl, stops)
    kw = dict(tokens=cu(tokens), retrieve=cu(ret), n_nodes=cu(n_nodes), n_paths=cu(n_paths), done=cu(done),
              hist=cu(hist), hist_len=cu(hist_len), eos=eos, **stop_kw)

    got = lg.clone()
    E.apply_logit_controls(got, *tabs, **kw)
    want, matches = _restate(lg, ctl, tokens, ret, n_nodes, n_paths, done, None, hist, hist_len, stops, eos)
    assert _same_bits(got, want)
    assert matches > 0
    for b in (3, 7):                                                    # neutral and finished: untouched
        assert torch.equal(got[b], lg[b]), b
    assert torch.equal(got[9, 8:], lg[9, 8:]) and not torch.equal(got[9, :8], lg[9, :8])    # rows off every path
    assert got[0, 0, ctl[0][0][0][0]].item() == -INF                    # -inf stays -inf
    assert got[2, 1, pool[1]].item() == -INF                            # a biased NaN on a banned id: banned
    assert got[6, 0, eos].item() == -INF and got[6, 1, eos].item() != -INF    # predicts m - 1: suppressed; m: not
    assert got[6, 0, pool[2]].item() == -INF                            # a stop whose head ends row 0's context ...
    assert got[6, 1, pool[2]].item() != -INF and got[6, 1, pool[3]].item() != -INF     # ... none at position m
    assert got[1, 0, pool[4]].item() == -INF                            # a head of history + path
    assert got[8, 0, pool[4]].item() == -INF                            # the 2-id head (node 0) matches, ...
    assert got[8, 0, pool[3]].item() != -INF                            # ... the 3-id one would reach before position 0

    # the identity chain (samd sequences), no stops
    got = lg.clone()
    chain_kw = {k: v for k, v in kw.items() if k not in ("retrieve", "n_paths", "stop_tokens", "stop_len")}
    E.apply_logit_controls(got, *tabs, **chain_kw)
    assert _same_bits(got, _restate(lg, ctl, tokens, None, n_nodes, None, done, None, hist, hist_len, None, eos)[0])

    # the admission form: one row per admitted request, no node tokens, state rows through slots, position 0
    slots = np.array([9, 2, 6, 0, 4], np.int32)
    rows = lg[:5, :1].clone()
    got = rows.clone()
    E.apply_logit_controls(got, *tabs, slots=cu(slots), eos=eos, **stop_kw)
    assert _same_bits(got, _restate(rows, ctl, slots=slots, stops=stops, eos=eos)[0])
    assert got[2, 0, eos].item() == -INF                                # min_tokens 22 > 0

    # graph and eager: the same bits
    eager = lg.clone()
    E.apply_logit_controls(eager, *tabs, **kw)
    graphed = lg.clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        E.apply_logit_controls(graphed, *tabs, **kw)
    graphed.copy_(lg)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(graphed.view(torch.uint8), eager.view(torch.uint8))


# ---- 2. lossless controlled greedy decoding -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lm():
    return _tiny_llama()


def _decoders(lm):
    from samd_b200 import engine as E, synth
    from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
    docs = [synth.copy_mix(300, V_LM, 5 + k).tolist() for k in range(3)] + [[i] for i in range(3, V_LM)]
    static = E.StaticSamDevice.build(docs, 2, with_counts=True)
    samd = lambda B, **kw: BatchedSamdDecoder(lm, B, 512, n_predicts=8, len_bias=5, len_threshold=3, dtype=torch.float32,
                                              **kw)
    sam_only = lambda B, **kw: BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0,
                                                     static=static, dtype=torch.float32, **kw)
    return dict(samd=samd, sam_only=sam_only)


def _penalize_row(x, gen, prompt, pn):
    """Penalties' documented formula (tests/test_gpu_penalties.py's restatement)."""
    c = torch.bincount(torch.as_tensor(gen, dtype=torch.long), minlength=V_LM).to(x.device)
    seen = torch.bincount(torch.as_tensor(prompt, dtype=torch.long), minlength=V_LM).to(x.device).gt(0) | (c > 0)
    rt, pt, ft = (torch.tensor([v], dtype=torch.float32, device=x.device)
                  for v in (pn.repetition_penalty, pn.presence_penalty, pn.frequency_penalty))
    y = x.float()
    y = torch.where(y < 0, y * rt, y / rt)
    y = y - ft * c.float()
    y = y - pt * (c > 0).float()
    return torch.where(seen, y.to(x.dtype), x)


def _controls_row(row, gen, lc, eos, stops):
    bias = [(int(t), float(v)) for t, v in lc.bias_items()] if lc is not None else []
    bad = [list(w) for w in lc.bad_words] if lc is not None else []
    m = lc.min_tokens if lc is not None else 0
    return _control_row(row, gen, len(gen), bias, bad, m, eos, [list(s) for s in stops])[0]


@torch.inference_mode()
def _controlled_greedy(lm, prompt, n_new, lc, eos=None, stops=(), pn=None, rows=False):
    """Plain greedy decoding: full forward, penalties (pn), then the controls on logits[:, -1], then the argmax; ends at
    EOS, a stop sequence (output only) or n_new.  rows=True also returns the controlled rows."""
    ids = torch.as_tensor([prompt]).cuda()
    gen, kept = [], []
    for _ in range(n_new):
        row = lm(input_ids=ids).logits[0, -1]
        if pn is not None:
            row = _penalize_row(row, gen, prompt, pn)
        row = _controls_row(row, gen, lc, eos, stops)
        kept.append(row)
        nxt = int(row.argmax())
        gen.append(nxt)
        if nxt == eos or any(_ends_with(gen, s) for s in stops):
            break
        ids = torch.cat([ids, torch.tensor([[nxt]], device="cuda")], 1)
    return (gen, kept) if rows else gen


def _serve(dec, prompts, limits, **kw):
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info)
    assert sorted(got) == list(range(len(prompts)))
    return got


@pytest.fixture(scope="module")
def work(lm):
    """Prompts, limits and mixed per-request controls whose bans bite: the bad words and biases are taken from the
    uncontrolled greedy outputs.  Token 0 gets no positive bias (the A9 corner)."""
    from samd_b200 import synth
    from samd_b200.batched import LogitControls
    lens = (150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70)
    prompts = [synth.copy_mix(n, V_LM, 300 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    limits = [8, 96] + [8 + (37 * i) % 89 for i in range(2, N_REQ)]
    plain = [_controlled_greedy(lm, prompts[i], limits[i], None) for i in range(N_REQ)]
    counts = np.bincount(np.concatenate(plain), minlength=V_LM)
    counts[0] = 0
    top = [int(t) for t in np.argsort(-counts)[:8]]
    pairs = {}
    for u in plain:
        for k in range(len(u) - 1):
            pairs[(u[k], u[k + 1])] = pairs.get((u[k], u[k + 1]), 0) + 1
    bigrams = [list(p) for p, _ in sorted(pairs.items(), key=lambda kv: -kv[1])[:6]]
    trigram = plain[1][10:13]
    kinds = [LogitControls(logit_bias={top[0]: -INF, top[1]: -4.0, top[5]: 3.0}),
             LogitControls(bad_words=[[top[2]], bigrams[0], bigrams[1], trigram]),
             LogitControls(),
             LogitControls(logit_bias=[(top[3], -INF), (top[4], 2.5)], bad_words=bigrams[2:5], min_tokens=4),
             LogitControls(min_tokens=6)]
    ctls = [kinds[i % len(kinds)] for i in range(N_REQ)]
    return prompts, limits, ctls, plain, top


@pytest.fixture(scope="module")
def reference(lm, work):
    prompts, limits, ctls, _, _ = work
    return [_controlled_greedy(lm, prompts[i], limits[i], ctls[i]) for i in range(N_REQ)]


@pytest.mark.parametrize("mode", ["samd", "samd_tree", "sam_only"])
def test_controlled_greedy_is_lossless(lm, work, reference, mode):
    """serve() at B = 4 over 13 requests with mixed per-request controls (neutral ones included) equals plain controlled
    greedy decoding: graphed and eager, check_every 4 and 1, with a prefix pool, with penalties, with EOS and stops, and
    through generate()."""
    from samd_b200 import synth
    from samd_b200.batched import Penalties, StopSequences
    prompts, limits, ctls, plain, top = work
    assert sum(reference[i] != plain[i] for i in range(N_REQ)) >= 4                    # the controls bite
    flavour = mode.replace("_tree", "")
    kw = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    mk = _decoders(lm)[flavour]
    dec = mk(4, **kw)
    for run in (dict(), dict(graph=False, check_every=1)):
        got = _serve(dec, prompts, limits, controls=ctls, **run)
        assert dec.serve_stats["graphed"] == run.get("graph", True)
        for i in range(N_REQ):
            assert got[i][0] == reference[i], (run, i)
    assert sum(sum(a > 1 for a in got[i][1]["accept_lengths"]) for i in range(N_REQ)) > 0     # drafts accepted
    pooled = mk(4, max_prefixes=2, **kw)
    pooled.add_prefix(prompts[1])
    pooled.add_prefix(prompts[6][:40])
    pgot = _serve(pooled, prompts, limits, controls=ctls)
    assert pgot[1][1]["prefix_len"] == len(prompts[1]) and pgot[6][1]["prefix_len"] == 40
    for i in range(N_REQ):
        assert pgot[i][0] == reference[i], i
    pn = Penalties(repetition_penalty=1.2, frequency_penalty=0.3)
    pen = _serve(dec, prompts, limits, controls=ctls, penalties=pn)
    for i in range(N_REQ):
        assert pen[i][0] == _controlled_greedy(lm, prompts[i], limits[i], ctls[i], pn=pn), i
    eos = top[6]
    stops = [[top[7]], [reference[1][20], reference[1][21]]]
    edec = mk(4, eos_token_id=eos, **kw)
    egot = _serve(edec, prompts, limits, controls=ctls, stop=StopSequences(stops))
    ended = 0
    for i in range(N_REQ):
        want = _controlled_greedy(lm, prompts[i], limits[i], ctls[i], eos=eos, stops=stops)
        assert egot[i][0] == want, i
        ended += egot[i][1]["finish_reason"] == "stop"
        if egot[i][1]["finish_reason"] == "stop":
            assert len(want) > ctls[i].min_tokens, i
    assert ended >= 2
    out, _ = dec.generate(prompts[4:8], 24, controls=ctls[4:8])
    assert out == [reference[i][:24] if limits[i] >= 24 else _controlled_greedy(lm, prompts[i], 24, ctls[i])
                   for i in range(4, 8)]


# ---- 3. min_tokens has teeth --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["samd", "samd_tree", "sam_only"])
def test_min_tokens_holds_back_eos_and_stops(lm, work, mode):
    from samd_b200 import synth
    from samd_b200.batched import LogitControls, StopSequences
    prompts, limits, _, plain, top = work
    flavour = mode.replace("_tree", "")
    kw = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    eos = top[1]
    dec = _decoders(lm)[flavour](4, eos_token_id=eos, **kw)
    mins = [min(limits[i] - 1, 3 + (5 * i) % 17) for i in range(N_REQ)]
    ctls = [LogitControls(logit_bias={eos: 100.0}, min_tokens=m) for m in mins]
    got = _serve(dec, prompts, limits, controls=ctls)
    for i in range(N_REQ):
        tokens, info = got[i]
        assert len(tokens) == mins[i] + 1 and tokens[-1] == eos and eos not in tokens[:-1], (i, tokens)
        assert info["finish_reason"] == "stop"
    # stops: a common token and a common bigram; nothing ends "stop" before min_tokens
    stops = StopSequences([[top[0]], plain[1][4:6]])
    mins = [min(limits[i], 2 + (7 * i) % 23) for i in range(N_REQ)]
    ctls = [LogitControls(min_tokens=m) for m in mins]
    got = _serve(dec, prompts, limits, controls=ctls, stop=stops)
    free = _serve(dec, prompts, limits, stop=stops)
    early = 0
    for i in range(N_REQ):
        tokens, info = got[i]
        if info["finish_reason"] == "stop":
            assert len(tokens) > mins[i], (i, tokens)
        early += free[i][1]["finish_reason"] == "stop" and len(free[i][0]) <= mins[i]
        assert tokens == _controlled_greedy(lm, prompts[i], limits[i], ctls[i], eos=eos, stops=stops.sequences), i
    assert early >= 1                                                  # without min_tokens some end before it


# ---- 4. sampled decoding never emits a banned token ---------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_sampled_never_emits_a_banned_token(flavour):
    from samd_b200 import synth
    from samd_b200.batched import LogitControls, SamplingParams
    lm = _tiny_llama(head_scale=4.0)
    mk = _decoders(lm)[flavour]
    prompts = [synth.copy_mix(40 + 7 * (i % 9), V_LM, 900 + i % 9, p_copy=0.7).tolist() for i in range(96)]
    plain = _serve(mk(8), prompts, 32, sampling=SamplingParams(seed=5))
    counts = np.bincount(np.concatenate([plain[i][0] for i in range(96)]), minlength=V_LM)
    counts[0] = 0
    top = [int(t) for t in np.argsort(-counts)[:6]]
    bad = [[top[2], top[3]], [top[3], top[2]], [top[4], top[4]], [top[1], top[5], top[1]]]
    lc = LogitControls(logit_bias={top[0]: -INF, top[1]: 1.0, 0: -INF}, bad_words=bad, min_tokens=5)
    procs = [dict(temperature=1.0), dict(temperature=1.5, top_p=0.95), dict(temperature=0.8, top_k=20)]
    params = [SamplingParams(seed=31 * i + 7, **procs[i % 3]) for i in range(96)]
    dec = mk(8, eos_token_id=top[5])
    got = _serve(dec, prompts, 32, sampling=params, controls=lc)
    alone = mk(1, eos_token_id=top[5])
    for i in range(96):
        u = got[i][0]
        assert top[0] not in u and 0 not in u, (i, u)
        for w in bad:
            assert not any(u[k:k + len(w)] == w for k in range(len(u))), (i, w, u)
        assert top[5] not in u[:5], (i, u)
        if i % 12 == 0:                                                # slot, B and graph do not matter
            one = _serve(alone, [prompts[i]], [32], sampling=[params[i]], controls=[lc], graph=False)[0]
            assert one[0] == u and one[1]["accept_lengths"] == got[i][1]["accept_lengths"], i


# ---- 5. None and neutral controls ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_neutral_is_none(lm, work, flavour):
    from samd_b200 import engine as E
    from samd_b200.batched import LogitControls
    prompts, limits, _, _, _ = work
    dec = _decoders(lm)[flavour](4)
    base = _serve(dec, prompts, limits)
    assert not any(k.startswith("ctl_") for k in dec._st)              # controls=None allocates nothing
    n_graphs = len(dec._graphs)
    for lc in (LogitControls(), LogitControls(min_tokens=3)):          # (no EOS, no stop: nothing to suppress)
        neutral = _serve(dec, prompts, limits, controls=lc)
        for i in range(N_REQ):
            assert neutral[i][0] == base[i][0] and neutral[i][1]["accept_lengths"] == base[i][1]["accept_lengths"], i
    n_graphs2 = len(dec._graphs)
    assert n_graphs2 > n_graphs
    again = _serve(dec, prompts, limits)                               # None replays the graphs it captured before
    assert len(dec._graphs) == n_graphs2
    for i in range(N_REQ):
        assert again[i][0] == base[i][0], i
    # launches, eager: controls add one per step and one per admission batch; None issues the step's launches only
    per_step = {"samd": 2, "sam_only": 4}[flavour]
    sub, runs = prompts[4:8], {}
    for lc in (None, LogitControls()):
        for n_new in (16, 40):
            c0 = E.launch_count()
            _, st = dec.generate(sub, n_new, graph=False, controls=lc)
            runs[lc is None, n_new] = (E.launch_count() - c0, st["steps_run"])
    for n_new in (16, 40):
        (c_none, s_none), (c_ctl, s_ctl) = runs[True, n_new], runs[False, n_new]
        assert s_none == s_ctl and c_ctl - c_none == s_none + 1, (n_new, runs)
    (c1, s1), (c2, s2) = runs[True, 16], runs[True, 40]
    assert s2 > s1 and c2 - c1 == per_step * (s2 - s1), runs


# ---- 6. log-probabilities of the controlled rows ------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["samd", "samd_tree", "sam_only"])
@torch.inference_mode()
def test_logprobs_are_those_of_the_controlled_rows(lm, work, reference, mode):
    from samd_b200 import synth
    prompts, limits, ctls, _, _ = work
    flavour = mode.replace("_tree", "")
    kw = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    dec = _decoders(lm)[flavour](4, **kw)
    got = _serve(dec, prompts, limits, controls=ctls, logprobs=2)
    for i in range(N_REQ):
        tokens, info = got[i]
        assert tokens == reference[i], i
        ids = torch.as_tensor([prompts[i] + tokens]).cuda()
        rows = lm(input_ids=ids).logits[0, len(prompts[i]) - 1:len(prompts[i]) - 1 + len(tokens)]
        ctl = torch.stack([_controls_row(rows[k], tokens[:k], ctls[i], None, []) for k in range(len(tokens))])
        ref = torch.log_softmax(ctl.float(), -1).cpu().numpy()
        want = ref[np.arange(len(tokens)), tokens]
        lp = np.asarray(info["logprobs"])
        assert np.isfinite(lp).all(), i
        assert np.abs(lp - want).max() <= 1e-4, (i, np.abs(lp - want).max())
        assert [top[0][0] for top in info["top_logprobs"]] == tokens, i
