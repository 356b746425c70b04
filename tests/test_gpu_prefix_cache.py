"""GPU tests of prefix reuse in the batched decoders (max_prefixes, add_prefix, drop_prefix): a request whose prompt starts
with a registered prefix starts from copies of the prefix's KV rows (samd_kv_copy_rows), automaton (samd_dyn_clone) and
static cursor, and must come out exactly as without the pool - tokens, and accept lengths, which a stale automaton or
cursor would change."""
import numpy as np
import pytest
import torch

import samd_oracle as O

pytestmark = pytest.mark.gpu


def _tiny_llama():
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, max_position_embeddings=2048, attn_implementation="eager")
    return LlamaForCausalLM(cfg).to("cuda", torch.float32).eval()


@torch.inference_mode()
def _plain_greedy(lm, prompt, n_new):
    out = torch.as_tensor([prompt]).cuda()
    for _ in range(n_new):
        nxt = lm(input_ids=out).logits[:, -1].argmax(-1, keepdim=True)
        out = torch.cat([out, nxt], dim=1)
    return out[0, len(prompt):].tolist()


@pytest.fixture(scope="module")
def lm():
    return _tiny_llama()


def _mix(n, seed):
    from samd_b200 import synth
    return synth.copy_mix(n, 96, seed, p_copy=0.7).tolist()


@pytest.fixture(scope="module")
def work(lm):
    """Three registered heads - A, A2 (A extended: the longest must win) and C - and 14 prompts: heads plus suffixes, a
    prompt equal to C, one equal to A2, prompts with no registered head, one that shares only part of A2 (it uses A) and
    one that shares only part of C (no match).  Limits 8 to 64; every prompt's plain greedy continuation."""
    A = _mix(60, 11)
    A2 = A + _mix(45, 12)
    C = _mix(80, 13)
    heads = [A, A2, C]
    prompts = [A + _mix(30, 20), A2 + _mix(25, 21), C + _mix(50, 22), list(C), _mix(120, 23), A2 + _mix(70, 24),
               A + _mix(12, 25), A2[:80] + _mix(20, 26), C[:50] + _mix(40, 27), _mix(90, 28), C + _mix(9, 29), list(A2),
               A2 + _mix(3, 30), _mix(64, 31)]
    plens = [60, 105, 80, 80, 0, 105, 60, 60, 0, 0, 80, 105, 105, 0]
    limits = [8 + (29 * i) % 57 for i in range(len(prompts))]
    greedy = [_plain_greedy(lm, p, 64) for p in prompts]
    return heads, prompts, plens, limits, greedy


def _serve(dec, prompts, limits, **kw):
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info)
    assert sorted(got) == list(range(len(prompts)))
    return got


def _samd(lm, B, **kw):
    from samd_b200.batched import BatchedSamdDecoder
    return BatchedSamdDecoder(lm, B, 512, **{**dict(n_predicts=8, len_bias=5, len_threshold=3, dtype=torch.float32), **kw})


def _snapshot(dyn, rows):
    torch.cuda.synchronize()
    meta = dyn.meta()
    return {r: (dyn.export(r), dyn.export_edges(r), meta[r].copy()) for r in rows}


def _same(a, b):
    (ea, ga, ma), (eb, gb, mb) = a, b
    assert ea.keys() == eb.keys()
    for k in ea:
        assert np.array_equal(ea[k], eb[k]), k
    assert np.array_equal(ga, gb) and np.array_equal(ma, mb)


def test_dyn_clone_engine_level():
    """Vocabulary 1000 (the root's overflow slots are in use), three pairs in one launch onto destinations that held
    larger automata: each destination equals its source (states, edges, meta words), the other destinations are
    untouched, and both extended by the same tokens equal the oracle's automaton over prefix + suffix - stale records
    past the source's states would break that, since creating a state writes only three words."""
    from samd_b200 import _cabi as K, engine as E, synth
    V, cap = 1000, 6000
    src, dst = E.DynSamBatch(4, cap), E.DynSamBatch(6, cap)
    se = E.DraftEngine(src, None, K.FLAVOUR_SAMD, n_predicts=8)
    de = E.DraftEngine(dst, None, K.FLAVOUR_SAMD, n_predicts=8)

    def feed(eng, R, seqs):
        n = max(len(x) for x in seqs.values())
        tok, cnt = torch.zeros(R, max(n, 1), dtype=torch.int32), torch.zeros(R, dtype=torch.int32)
        for r, x in seqs.items():
            tok[r, :len(x)] = torch.as_tensor(x)
            cnt[r] = len(x)
        eng.step(tok.cuda(), cnt.cuda(), None)

    pre = {r: synth.copy_mix(800 + 150 * r, V, 60 + r, p_copy=0.6).tolist() for r in range(4)}
    old = {r: synth.copy_mix(2500 - 100 * r, V, 70 + r, p_copy=0.4).tolist() for r in range(6)}
    feed(se, 4, pre)
    feed(de, 6, old)
    pairs = [(0, 1), (2, 4), (3, 0)]                                             # (src, dst)
    before = _snapshot(dst, range(6))
    assert all(before[d][2][0] > _snapshot(src, [s])[s][2][0] for s, d in pairs)
    dst.clone_from(src, torch.tensor([s for s, _ in pairs], dtype=torch.int32, device="cuda"),
                   torch.tensor([d for _, d in pairs], dtype=torch.int32, device="cuda"))
    after, srcs = _snapshot(dst, range(6)), _snapshot(src, range(4))
    for s, d in pairs:
        _same(after[d], srcs[s])
    for d in (2, 3, 5):
        _same(after[d], before[d])
    suf = {s: synth.copy_mix(700, V, 90 + s, p_copy=0.6).tolist() for s, _ in pairs}
    feed(se, 4, suf)
    feed(de, 6, {d: suf[s] for s, d in pairs})
    after, srcs = _snapshot(dst, range(6)), _snapshot(src, range(4))
    for s, d in pairs:
        ex, edges, _ = after[d]
        ora = O.Automaton()
        ora.extend(pre[s] + suf[s])
        assert ex["overflow"] == 0 and ex["n_states"] == len(ora.link)
        assert np.array_equal(ex["link"], ora.link) and np.array_equal(ex["length"], ora.length)
        assert np.array_equal(ex["min_endpos"], ora.first_end) and np.array_equal(ex["text"][1:], pre[s] + suf[s])
        assert sorted(map(tuple, edges.tolist())) == sorted((a, t, b) for a, tr in enumerate(ora.trans) for t, b in tr.items())
        assert np.array_equal(edges, srcs[s][1])
    assert max(len(tr) for tr in ora.trans) > 16
    other = E.DynSamBatch(1, cap + 1)
    one = torch.zeros(1, dtype=torch.int32, device="cuda")
    with pytest.raises(K.SamdError, match="max_tokens differ"):
        other.clone_from(src, one, one)


@pytest.mark.parametrize("dtype, dh", [(torch.bfloat16, 64), (torch.float16, 36), (torch.float32, 36), (torch.float32, 13)])
def test_kv_copy_rows(dtype, dh):
    """Ragged row counts (0 and the source's full length among them), a pool and a cache of different batch sizes and
    lengths, rows of 72 / 52 bytes (not multiples of 16, so most rows are not 16-byte aligned): every listed row equals
    torch slicing bit for bit and nothing else of either side changes."""
    from samd_b200 import engine as E
    g = torch.Generator(device="cuda").manual_seed(3)
    n_kv, H, Ls, Ld = 4, 2, 40, 48
    src = [torch.randn(3, H, Ls, dh, device="cuda", generator=g).to(dtype) for _ in range(n_kv)]
    dst = [torch.randn(5, H, Ld, dh, device="cuda", generator=g).to(dtype) for _ in range(n_kv)]
    src0, want = [t.clone() for t in src], [t.clone() for t in dst]
    pairs = [(4, 1, Ls), (0, 2, 0), (2, 0, 17), (1, 2, 5)]                         # (dst row, src row, n_rows)
    for d, s, n in pairs:
        for k in range(n_kv):
            want[k][d, :, :n] = src[k][s, :, :n]
    col = lambda j: torch.tensor([p[j] for p in pairs], dtype=torch.int32, device="cuda")
    E.kv_copy_rows(E.kv_table(dst, "cuda"), E.kv_table(src, "cuda"), col(0), col(1), col(2))
    torch.cuda.synchronize()
    bits = {torch.bfloat16: torch.int16, torch.float16: torch.int16, torch.float32: torch.int32}[dtype]
    for k in range(n_kv):
        assert torch.equal(dst[k].view(bits), want[k].view(bits)), k
        assert torch.equal(src[k].view(bits), src0[k].view(bits)), k


def _check_prefix_serve(dec, work, ref_acc=None, **kw):
    heads, prompts, plens, limits, greedy = work
    got = _serve(dec, prompts, limits, **kw)
    for i, (tokens, info) in got.items():
        assert tokens == greedy[i][:limits[i]], i
        assert info["prefix_len"] == plens[i], i
        if ref_acc is not None:
            assert info["accept_lengths"] == ref_acc[i], i
    st = dec.serve_stats
    assert st["prefix_hits"] == sum(p > 0 for p in plens) and st["prefix_tokens"] == sum(plens)
    return got


def test_serve_is_lossless_with_prefixes(lm, work):
    """B = 4, 14 requests over 3 registered heads: tokens are plain greedy decoding, graphed and eager; the accept lengths
    equal those of the same requests served without a pool; prefix_hits / prefix_tokens are exact."""
    heads, prompts, plens, limits, greedy = work
    nopool = _samd(lm, 4)
    plain = _serve(nopool, prompts, limits)
    assert "prefix_hits" not in nopool.serve_stats and nopool.pool is None
    ref = {i: info["accept_lengths"] for i, (_, info) in plain.items()}
    assert all("prefix_len" not in info for _, info in plain.values())
    dec = _samd(lm, 4, max_prefixes=4)
    ids = [dec.add_prefix(h) for h in heads]
    assert ids == [0, 1, 2] and dec.add_prefix(list(heads[1])) == 1
    _check_prefix_serve(dec, work, ref)
    assert dec.serve_stats["graphed"]
    _check_prefix_serve(dec, work, ref, graph=False)
    assert not dec.serve_stats["graphed"]


def test_samd_prefix_state_matches_requests_run_alone(lm, work):
    """With a static corpus, a request started from a prefix accepts what its full prompt accepts on a B = 1 decoder."""
    from samd_b200 import engine as E, synth
    heads, prompts, plens, limits, greedy = work
    static = E.StaticSamDevice.build([g[10:60] for g in greedy[::3]] + [synth.copy_mix(300, 96, 5).tolist()], 2)
    dec = _samd(lm, 4, static=static, max_prefixes=3)
    for h in heads:
        dec.add_prefix(h)
    got = _serve(dec, prompts, limits)
    one = _samd(lm, 1, static=static)
    for i, p in enumerate(prompts):
        out, st = one.generate([p], limits[i])
        assert got[i][0] == out[0] == greedy[i][:limits[i]], i
        assert got[i][1]["accept_lengths"] == [a for a in st["accept_lengths"][0] if a], i
        assert got[i][1]["prefix_len"] == plens[i]


def test_sam_only_prefix_state_matches_requests_run_alone(lm):
    """The same for BatchedSamOnlyDecoder with a with-counts static corpus: static trees are drafted from cloned state."""
    from samd_b200 import engine as E, synth
    from samd_b200.batched import BatchedSamOnlyDecoder
    heads = [_mix(70, 41), _mix(90, 42)]
    prompts, wants = [], []
    # prompts whose greedy continuation never holds token 0 (the -1 pad corner, see BatchedSamOnlyDecoder)
    for i in range(40):
        p = heads[i % 2] + _mix(20 + (31 * i) % 90, 800 + i) if i % 5 else _mix(80 + i, 800 + i)
        w = _plain_greedy(lm, p, 64)
        if 0 not in w:
            prompts.append(p)
            wants.append(w)
        if len(prompts) == 8:
            break
    assert len(prompts) >= 6
    limits = [16 + (23 * i) % 49 for i in range(len(prompts))]
    docs = [w[5:59] for w in wants] + [synth.copy_mix(300, 96, 5).tolist()] + [[i] for i in range(3, 96)]
    static = E.StaticSamDevice.build(docs, 2, with_counts=True)
    mk = lambda B, **kw: BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0, static=static,
                                               dtype=torch.float32, **kw)
    dec = mk(3, max_prefixes=2)
    for h in heads:
        dec.add_prefix(h)
    got = _serve(dec, prompts, limits)
    assert dec.serve_stats["tree_steps"] > 0 and dec.serve_stats["prefix_hits"] >= 4
    one = mk(1)
    for i, p in enumerate(prompts):
        out, st = one.generate([p], limits[i])
        assert got[i][0] == out[0] == wants[i][:limits[i]], i
        assert got[i][1]["accept_lengths"] == [a for a in st["accept_lengths"][0] if a], i


def test_token_recycle_tree_with_prefixes_is_lossless(lm, work):
    from samd_b200 import synth
    heads, prompts, plens, limits, greedy = work
    dec = _samd(lm, 4, len_threshold=6, tree=synth.token_recycle_tree(), max_prefixes=3)
    for h in heads:
        dec.add_prefix(h)
    assert all(e["topk"].shape == (len(h), 8) for e, h in zip(dec._prefixes, heads))
    _check_prefix_serve(dec, work)


def test_recycle_apply_is_sequential_last_writer_wins():
    """RecycleTable.apply on rows whose tokens repeat across and within requests gives the table that assigning the rows
    one after the other gives."""
    from samd_b200 import engine as E, synth
    V = 50
    rng = np.random.default_rng(7)
    tokens = rng.integers(0, 12, size=300)
    rows = rng.integers(-1, V, size=(300, 8)).astype(np.int32)
    tab = E.RecycleTable(synth.token_recycle_tree(), V, "cuda")
    tab.table[20] = 5
    want = tab.table.cpu().numpy().copy()
    for t, r in zip(tokens, rows):
        want[t] = r
    tab.apply(torch.as_tensor(tokens).cuda(), torch.as_tensor(rows).cuda())
    assert np.array_equal(tab.table.cpu().numpy(), want)


def test_multi_turn(lm):
    """Serve a request, register prompt + answer as a prefix, serve prompt + answer + the next turn."""
    p1 = _mix(90, 51)
    dec = _samd(lm, 2, max_prefixes=2)
    (_, a1, info), = list(dec.serve([p1], 40))
    assert a1 == _plain_greedy(lm, p1, 40) and info["prefix_len"] == 0
    turn = p1 + a1
    dec.add_prefix(turn)
    p2 = turn + _mix(17, 52)
    (_, a2, info), = list(dec.serve([p2], 32))
    assert a2 == _plain_greedy(lm, p2, 32) and info["prefix_len"] == len(turn)


def test_prefix_edges(lm, work):
    from samd_b200 import _cabi as K
    heads, prompts, plens, limits, greedy = work
    with pytest.raises(K.SamdError, match="no prefix pool"):
        _samd(lm, 2).add_prefix(heads[0])
    dec = _samd(lm, 4, max_prefixes=2, max_tokens=300)
    for toks, msg in (([], "empty prefix"), (list(range(3, 96)) * 6, "does not fit max_cache_len"),
                      (_mix(295, 60), "automaton capacity")):
        with pytest.raises(K.SamdError, match=msg):
            dec.add_prefix(toks)
    a, c = dec.add_prefix(heads[0]), dec.add_prefix(heads[2])
    with pytest.raises(K.SamdError, match="pool is full"):
        dec.add_prefix(heads[1])
    # generate() matches too and stays exact
    sel = [0, 2, 4, 6]
    out, _ = dec.generate([prompts[i] for i in sel], 24)
    assert out == [greedy[i][:24] for i in sel]
    # drop_prefix stops matches
    dec.drop_prefix(a)
    with pytest.raises(K.SamdError, match="no registered prefix"):
        dec.drop_prefix(a)
    got = _serve(dec, prompts[:4], 16)
    assert [got[i][1]["prefix_len"] for i in range(4)] == [0, 0, 80, 80]
    assert all(got[i][0] == greedy[i][:16] for i in range(4))
    # add_prefix while a serve() generator is suspended: that generator's outputs stay exact, later admissions match
    it = dec.serve(prompts, limits)
    seen = dict([next(it)[:2]])
    assert dec.add_prefix(heads[1]) == a
    for i, tokens, info in it:
        seen[i] = tokens
    assert sorted(seen) == list(range(len(prompts)))
    assert all(seen[i] == greedy[i][:limits[i]] for i in seen)
    assert dec.serve_stats["prefix_hits"] >= 4
