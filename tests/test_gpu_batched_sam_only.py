"""GPU tests of the batched sam_only path: samd_draft_assemble (per-request sequence / static-tree drafts as uniform
batch buffers) against the reference's buffer construction, the finished-request rule of the verify launch, and
BatchedSamOnlyDecoder end to end on a tiny Llama against plain greedy decoding and the batch-1 drop-in."""
import numpy as np
import pytest
import torch

import samd_oracle as O

pytestmark = pytest.mark.gpu

DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}


def _torch_mask(allow, cache_len, kv_len, dtype):
    """[B, T, kv_len] additive mask from per-request [T, T] allow tables, with torch ops."""
    B, T, _ = allow.shape
    j = torch.arange(kv_len, device=allow.device)[None, None, :]
    rel = j - cache_len.long()[:, None, None]
    inside = (rel >= 0) & (rel < T)
    ok = torch.gather(allow, 2, rel.clamp(0, T - 1).expand(B, T, kv_len))
    ok = (rel < 0) | (inside & ok)
    m = torch.zeros(B, T, kv_len, dtype=dtype, device=allow.device)
    m.masked_fill_(~ok, torch.finfo(dtype).min)
    return m


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _buffers(B, T, P, D, kv_len, dtype, dev="cuda"):
    mk = lambda *s: torch.full(s, 7, dtype=torch.int32, device=dev)          # garbage: every element must be written
    return dict(tokens=mk(B, T), position_ids=torch.full((B, T), 7, dtype=torch.long, device=dev), n_nodes=mk(B),
                n_paths=mk(B), retrieve=mk(B, P, D), mask=torch.full((B, T, kv_len), 3.0, dtype=dtype, device=dev))


def _assemble(eng, cache_len, buf, done=None):
    eng.assemble(cache_len, buf["tokens"], buf["position_ids"], buf["n_nodes"], buf["n_paths"], buf["retrieve"], buf["mask"],
                 done=done)
    torch.cuda.synchronize()


def test_assembled_buffers_equal_the_reference_buffers():
    """B = 16 copy_mix streams through DynSamBatch + DraftEngine(sam_only) + a with-counts static SAM, several steps:
    tree requests get gen_buffers of the reference's best-first tree, sequence requests the chain of the step kernel's
    draft; the whole mask equals a torch construction bit for bit in bf16 / fp16 / fp32 at kv_len = T, a bucketed kv_len
    and an unaligned one, pad rows included; finished requests get the one-node draft."""
    from samd_b200 import _cabi as K, engine as E, synth
    from samd_sam_only.sam.static_sam import tree_buffers_from_parents
    B, V, T, alpha, Kt, len_bias = 16, 400, 24, 4.0, 4, 2
    docs = [synth.copy_mix(300, V, 1000 + k, p_copy=0.6).tolist() for k in range(6)]
    corpus = np.concatenate([np.asarray(d) for d in docs])
    streams = [synth.copy_mix(600, V, 40 + b, p_copy=0.6, source=corpus, p_source=0.6) for b in range(B)]
    static = E.StaticSamDevice.build(docs, synth.EOS, with_counts=True)
    dyn = E.DynSamBatch(B, 2048)
    eng = E.DraftEngine(dyn, static, K.FLAVOUR_SAM_ONLY, n_predicts=T, len_bias=len_bias, alpha=alpha)
    ora_static = O.build_static(docs, synth.EOS, count_occurrences=True)
    topk = O.build_topk(ora_static, 8)
    ora_dyn = [O.Automaton() for _ in range(B)]
    curs = [(0, 0)] * B
    pos = [150 + 7 * b for b in range(B)]
    chunks = [streams[b][:pos[b]] for b in range(B)]
    kinds_seen = set()
    for step in range(6):
        kmax = max(len(c) for c in chunks)
        tok = torch.zeros(B, kmax, dtype=torch.int32)
        for b, c in enumerate(chunks):
            tok[b, :len(c)] = torch.as_tensor(c, dtype=torch.int32)
        counts = torch.tensor([len(c) for c in chunks], dtype=torch.int32, device="cuda")
        start = torch.tensor([int(streams[b][pos[b]]) for b in range(B)], dtype=torch.int32, device="cuda")
        eng.step(tok.cuda(), counts, start)
        eng.tree_draft(start, K_top=Kt)
        cache_len = torch.tensor([3 * b + 5 * step for b in range(B)], dtype=torch.int32, device="cuda")
        cl = cache_len.tolist()
        # the reference's buffers, request by request
        allow = torch.zeros(B, T, T, dtype=torch.bool)
        want = []
        for b in range(B):
            ora_dyn[b].extend(chunks[b])
            ora_static.cur, ora_static.cur_len = curs[b]
            ora_static.advance(chunks[b])
            curs[b] = (ora_static.cur, ora_static.cur_len)
            kind, toks, par, _ = O.select_sam_only(ora_dyn[b], ora_static, topk, int(start[b]), T, alpha, Kt, len_bias)
            kinds_seen.add(kind)
            n = len(toks)
            if kind == "tree":
                m, depth, ret = O.tree_buffers(par)
            else:
                m = np.tril(np.ones((n, n), dtype=bool))
                depth, ret = np.arange(n), np.arange(n)[None, :]
            allow[b, :n, :n] = torch.as_tensor(m)
            for i in range(n, T):
                allow[b, i, i] = True
            want.append((kind, toks, depth, ret, par))
        allow = allow.cuda()
        bucket = (max(cl) + T + 63) // 64 * 64
        for dt in DTYPES.values():
            for kv_len in (T, bucket, T + 7):
                buf = _buffers(B, T, T, T, kv_len, dt)
                _assemble(eng, cache_len, buf)
                assert torch.equal(_bits(buf["mask"]), _bits(_torch_mask(allow, cache_len, kv_len, dt))), (dt, kv_len)
        # small outputs, and the tree blocks of the mask next to the batch-1 drop-in's gen_buffers
        buf = _buffers(B, T, T, T, bucket, torch.float32)
        _assemble(eng, cache_len, buf)
        for b, (kind, toks, depth, ret, par) in enumerate(want):
            n = len(toks)
            assert int(eng.out_type[b]) == (K.DRAFT_STATIC_TREE if kind == "tree" else K.DRAFT_DYN_SEQ)
            assert buf["tokens"][b].tolist() == list(toks) + [0] * (T - n)
            assert buf["position_ids"][b].tolist() == [cl[b] + int(d) for d in depth] + [cl[b] + i for i in range(n, T)]
            assert int(buf["n_nodes"][b]) == n and int(buf["n_paths"][b]) == ret.shape[0]
            full = -np.ones((T, T), dtype=np.int64)
            full[:ret.shape[0], :ret.shape[1]] = ret
            assert np.array_equal(buf["retrieve"][b].cpu().numpy(), full)
            if kind == "tree":                                       # ... and the batch-1 drop-in's gen_buffers
                leaves, width = eng.tree_shape[b].tolist()
                ref = tree_buffers_from_parents(eng.tree_parents[b, :n], eng.tree_depth[b, :n], eng.tree_retrieve[b, :leaves, :width])
                blk = buf["mask"][b, :n, cl[b]:cl[b] + n] == 0
                assert torch.equal(blk, ref["tree_attn_mask"][0, 0])
                assert torch.equal(buf["position_ids"][b, :n] - cl[b], ref["tree_position_ids"][0])
                assert torch.equal(buf["retrieve"][b, :leaves, :width].long(), ref["tree_retrieve_indices"])
            else:
                assert int(eng.draft_len[b]) == n
        # finished requests: a one-node draft with no path, whatever their type
        done = torch.tensor([b % 3 == 0 for b in range(B)], device="cuda")
        buf = _buffers(B, T, T, T, bucket, torch.float16)
        _assemble(eng, cache_len, buf, done=done)
        dallow = allow.clone()
        for b in range(0, B, 3):
            dallow[b] = torch.eye(T, dtype=torch.bool, device="cuda")
            assert int(buf["n_nodes"][b]) == 1 and int(buf["n_paths"][b]) == 0
            assert buf["retrieve"][b, 0].tolist() == [0] + [-1] * (T - 1) and bool((buf["retrieve"][b, 1:] == -1).all())
            assert buf["tokens"][b].tolist() == [int(start[b])] + [0] * (T - 1)
            assert buf["position_ids"][b].tolist() == [cl[b] + i for i in range(T)]
        assert torch.equal(_bits(buf["mask"]), _bits(_torch_mask(dallow, cache_len, bucket, torch.float16)))
        # next step: feed a few true tokens of every stream
        for b in range(B):
            k = 1 + (b + step) % 5
            chunks[b] = streams[b][pos[b]:pos[b] + k]
            pos[b] += k
    assert kinds_seen == {"tree", "sequence"}


def test_assemble_rejects_bad_shapes():
    from samd_b200 import _cabi as K, engine as E
    B, T = 2, 8
    dyn = E.DynSamBatch(B, 64)
    eng = E.DraftEngine(dyn, None, K.FLAVOUR_SAM_ONLY, n_predicts=T)
    cl = torch.zeros(B, dtype=torch.int32, device="cuda")
    buf = _buffers(B, T, T, T, T - 1, torch.float16)                 # kv_len < T
    with pytest.raises(K.SamdError, match="kv_len"):
        _assemble(eng, cl, buf)
    buf = _buffers(B, 300, T, T, 300, torch.float16)                 # T > 256
    with pytest.raises(K.SamdError, match="n_nodes"):
        _assemble(eng, cl, buf)


def _plant(eng, B, T, kinds, parents, tokens):
    """Engine outputs set by hand: request b drafts tokens[b] as a sequence or as a tree with parents[b]."""
    from samd_b200 import _cabi as K
    dev = "cuda"
    mk = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
    eng.tree_tokens, eng.tree_parents, eng.tree_depth = mk(B, T), mk(B, T), mk(B, T)
    eng.tree_n, eng.tree_shape, eng.tree_retrieve = mk(B), mk(B, 2), torch.full((B, T, T), 5, dtype=torch.int32, device=dev)
    eng.draft.zero_()
    for b in range(B):
        n = len(tokens[b])
        if kinds[b] == "tree":
            eng.out_type[b] = K.DRAFT_STATIC_TREE
            _, depth, ret = O.tree_buffers(parents[b])
            eng.tree_tokens[b, :n] = torch.as_tensor(tokens[b])
            eng.tree_parents[b, :n] = torch.as_tensor(parents[b])
            eng.tree_depth[b, :n] = torch.as_tensor(depth)
            eng.tree_n[b] = n
            eng.tree_shape[b] = torch.tensor(ret.shape)
            r = -np.ones((T, T), dtype=np.int64)
            r[:ret.shape[0], :ret.shape[1]] = ret
            r[ret.shape[0]:] = 3                                      # stale rows past the leaves: must not be read
            eng.tree_retrieve[b] = torch.as_tensor(r)
            eng.draft_len[b] = 0
        else:
            eng.out_type[b] = K.DRAFT_DYN_SEQ
            eng.draft[b, :n] = torch.as_tensor(tokens[b])
            eng.draft_len[b] = n


@pytest.mark.parametrize("T", [8, 16])
def test_finished_requests_move_no_kv_rows(T):
    """KV rows hold their own position; some requests are finished (one at the very end of its cache).  After assemble +
    samd_verify_compact(move_kv=True) on logits planted to accept each request's deepest path, every KV byte of a finished
    request is unchanged and the live requests match O.kv_compact."""
    from samd_b200 import _cabi as K, engine as E
    B, V, H, ML, DH = 8, 64, 2, 96, 8
    dev = "cuda"
    dyn = E.DynSamBatch(B, 64)
    eng = E.DraftEngine(dyn, None, K.FLAVOUR_SAM_ONLY, n_predicts=T)
    rng = np.random.default_rng(T)
    kinds, parents, tokens = [], [], []
    for b in range(B):
        n = int(rng.integers(3, T + 1))
        par = [-1] + [int(rng.integers(max(0, i - 3), i)) for i in range(1, n)]
        kinds.append("tree" if b % 2 else "sequence")
        parents.append(par)
        tokens.append(rng.integers(3, V, size=n).tolist())
    _plant(eng, B, T, kinds, parents, tokens)
    done = torch.tensor([b in (1, 2, 5) for b in range(B)], device=dev)
    cache_len = torch.tensor([10 + 4 * b for b in range(B)], dtype=torch.int32, device=dev)
    cache_len[5] = ML                                                 # full: rows from cache_len would leave the request
    kv = [torch.arange(B * H * ML * DH, dtype=torch.float32, device=dev).view(B, H, ML, DH) + 1e5 * l for l in range(4)]
    ref = [t.clone() for t in kv]
    buf = _buffers(B, T, T, T, ML + T, torch.float32)
    _assemble(eng, cache_len, buf, done=done)
    # plant logits: along the deepest path (tree) / the whole chain (sequence) every row predicts the next node's token
    logits = torch.randn(B, T, V, device=dev)
    logits[:, :, 0] = -100.0                                          # argmax never 0 (the -1 pad corner stays out)
    for b in range(B):
        n, P = int(buf["n_nodes"][b]), max(int(buf["n_paths"][b]), 1)
        ret = buf["retrieve"][b, :P].tolist()
        path = max(ret, key=lambda r: sum(x >= 0 for x in r))
        path = [x for x in path if x >= 0]
        for a, c in zip(path[:-1], path[1:]):
            logits[b, a, int(buf["tokens"][b, c])] = 50.0
    ver = E.Verifier(B, T)
    ver.bind_kv(kv)
    before = cache_len.clone()
    out = ver.verify(logits, buf["tokens"], buf["retrieve"], cache_len=cache_len, move_kv=True, n_nodes=buf["n_nodes"],
                     n_paths=buf["n_paths"])
    torch.cuda.synchronize()
    am = O.row_argmax(logits)
    deep = 0
    for b in range(B):
        if bool(done[b]):
            assert int(out["accept_len"][b]) == 1
            for t, r in zip(kv, ref):
                assert torch.equal(t[b], r[b]), f"finished request {b}: KV rows moved"
            continue
        n, P = int(buf["n_nodes"][b]), int(buf["n_paths"][b])
        r = O.verify_greedy(am[b][:n], buf["tokens"][b, :n].cpu().numpy(), buf["retrieve"][b, :P].cpu().numpy().astype(np.int64))
        al = r["accept_len"]
        assert int(out["accept_len"][b]) == al and int(out["next_token"][b]) == r["next_token"]
        deep = max(deep, al)
        want = [t[b].cpu().numpy().copy() for t in ref]
        O.kv_compact(want, int(before[b]), r["indices"], al)
        for t, w in zip(kv, want):
            assert np.array_equal(t[b].cpu().numpy(), w)
    assert deep >= 3


# ---------------------------------------------------------------------------------------------------------------------
# BatchedSamOnlyDecoder end to end
# ---------------------------------------------------------------------------------------------------------------------
def _setup(n_new):
    from test_gpu_dropin import _tiny_llama, _plain_greedy
    from samd_b200 import synth
    lm = _tiny_llama(torch.float32)
    prompts, want = [], []
    # ragged prompts whose greedy continuation never holds token 0 (the -1 pad corner, see BatchedSamOnlyDecoder)
    for i, n in enumerate((150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70, 190, 100, 84)):
        p = synth.copy_mix(n, 96, 300 + i, p_copy=0.7).tolist()
        w = _plain_greedy(lm, torch.as_tensor([p]).cuda(), n_new)[len(p):]
        if 0 not in w:
            prompts.append(p)
            want.append(w)
        if len(prompts) == 5:
            break
    assert len(prompts) >= 4
    docs = [w[5:n_new - 5] for w in want] + [synth.copy_mix(300, 96, 5).tolist()] + [[i] for i in range(3, 96)]
    return lm, prompts, want, docs


def test_batched_sam_only_decoder_is_lossless():
    from samd_b200 import _cabi as K, engine as E
    from samd_b200.batched import BatchedSamOnlyDecoder
    n_new = 64
    lm, prompts, want, docs = _setup(n_new)
    B = len(prompts)
    static = E.StaticSamDevice.build(docs, 2, with_counts=True)
    dec = BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0, static=static, dtype=torch.float32)
    got, stats = dec.generate(prompts, n_new)
    assert got == want
    assert stats["steps"] < n_new and stats["tree_steps"] > 0
    assert stats["graphed"] and stats["graphs"] >= 1
    assert stats["host_syncs"] <= stats["steps_run"] // 4 + 1 and stats["steps_run"] - stats["steps"] < 4
    got_e, stats_e = dec.generate(prompts, n_new, graph=False)
    assert got_e == want and stats_e["accept_lengths"] == stats["accept_lengths"] and not stats_e["graphed"]
    assert stats_e["tree_steps"] == stats["tree_steps"]
    # EOS truncation
    eos = want[1][10]
    dec2 = BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0, static=static, eos_token_id=eos,
                                 dtype=torch.float32)
    got2, _ = dec2.generate(prompts, n_new)
    for g, w in zip(got2, want):
        cut = w.index(eos) + 1 if eos in w else len(w)
        assert g == w[:cut]
    # no static automaton: dynamic sequences only
    dec3 = BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, dtype=torch.float32)
    got3, stats3 = dec3.generate(prompts, n_new)
    assert got3 == want and stats3["tree_steps"] == 0
    got3_e, stats3_e = dec3.generate(prompts, n_new, graph=False)
    assert got3_e == want and stats3_e["accept_lengths"] == stats3["accept_lengths"]
    # a static automaton without counts cannot draft trees
    with pytest.raises(K.SamdError, match="with_counts"):
        BatchedSamOnlyDecoder(lm, B, 512, static=E.StaticSamDevice.build(docs, 2), dtype=torch.float32)


def test_batched_sam_only_matches_the_batch1_dropin():
    """Every request's accept lengths equal those of samd_sam_only.SamdModel.generate on that prompt alone."""
    import samd_sam_only as so
    from samd_b200 import engine as E
    from samd_b200.batched import BatchedSamOnlyDecoder
    n_new = 64
    lm, prompts, want, docs = _setup(n_new)
    B = len(prompts)
    dec = BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0,
                                static=E.StaticSamDevice.build(docs, 2, with_counts=True), dtype=torch.float32)
    got, stats = dec.generate(prompts, n_new)
    assert got == want
    cfg = so.SamdConfig(max_predicts=16, alpha=4.0, K=4, len_bias=0)
    for b, p in enumerate(prompts):
        draft = so.DraftModel(cfg, sam_static=so.build_sam(docs, 2), lm=lm, dtype=torch.float32, device="cuda")
        model = so.SamdModel(cfg, lm, draft, eos_token_id=-1, dtype=torch.float32, device="cuda")
        out = model.generate(torch.as_tensor([p]).cuda(), generation_config=so.SamdGenerationConfig(max_new_tokens=n_new,
                                                                                                   max_cache_len=512))
        assert out.output_ids[0][len(p):] == want[b]
        assert out.accepet_length_per_step == [a for a in stats["accept_lengths"][b] if a]
