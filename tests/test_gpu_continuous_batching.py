"""GPU tests of continuous batching in the batched decoders (BatchedSamdDecoder.serve / BatchedSamOnlyDecoder.serve):
more requests than slots, refilled into finished slots between graphed decode steps, must each come out exactly as plain
greedy decoding of that prompt alone - tokens, and accept lengths where the drafter is per request - and an admission
must leave every other request's drafter state untouched."""
import numpy as np
import pytest
import torch

import samd_oracle as O

pytestmark = pytest.mark.gpu

N_REQ = 13


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


@pytest.fixture(scope="module")
def work(lm):
    """13 ragged copy_mix prompts, per-request limits from 8 to 96 and every prompt's plain greedy continuation."""
    from samd_b200 import synth
    lens = (150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70)
    prompts = [synth.copy_mix(n, 96, 300 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    limits = [8, 96] + [8 + (37 * i) % 89 for i in range(2, N_REQ)]
    greedy = [_plain_greedy(lm, p, 96) for p in prompts]
    return prompts, limits, greedy


def _serve(dec, prompts, limits, **kw):
    """{index: (tokens, info)}; every request exactly once."""
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info)
    assert sorted(got) == list(range(len(prompts)))
    return got


def _samd(lm, B, **kw):
    from samd_b200.batched import BatchedSamdDecoder
    return BatchedSamdDecoder(lm, B, 512, **{**dict(n_predicts=8, len_bias=5, len_threshold=3, dtype=torch.float32), **kw})


def test_serve_is_lossless_with_refills(lm, work):
    """B = 4 slots, 13 requests: every request's tokens equal plain greedy decoding up to its own limit; one admission
    per request; graphs are captured per key-length bucket only; the eager body gives the same tokens and accept lengths."""
    prompts, limits, greedy = work
    dec = _samd(lm, 4)
    reached = set()
    advance = dec._advance
    dec._advance = lambda kv_len, graph: (reached.add(kv_len), advance(kv_len, graph))[1]
    got = _serve(dec, prompts, limits)
    for i, (tokens, info) in got.items():
        assert tokens == greedy[i][:limits[i]], i
        assert len(info["accept_lengths"]) > 0 and all(a > 0 for a in info["accept_lengths"])
    st = dec.serve_stats
    assert st["admissions"] == N_REQ and st["graphed"] and 1 <= st["graphs"] <= len(reached)
    assert st["live_slot_steps"] == sum(len(info["accept_lengths"]) for _, info in got.values())
    assert st["host_syncs"] <= st["steps_run"] // 4 + 1
    eager = _serve(dec, prompts, limits, graph=False)
    assert not dec.serve_stats["graphed"]
    for i in range(N_REQ):
        assert eager[i][0] == got[i][0] and eager[i][1]["accept_lengths"] == got[i][1]["accept_lengths"], i


def test_samd_refills_match_requests_run_alone(lm, work):
    """A stale automaton or static cursor would still give greedy tokens, so compare accept lengths: every request served
    through refilled slots accepts what it accepts run by itself on a B = 1 decoder with the same settings."""
    from samd_b200 import engine as E, synth
    prompts, limits, greedy = work
    static = E.StaticSamDevice.build([g[10:80] for g in greedy[::3]] + [synth.copy_mix(300, 96, 5).tolist()], 2)
    got = _serve(_samd(lm, 4, static=static), prompts, limits)
    one = _samd(lm, 1, static=static)
    for i, p in enumerate(prompts):
        out, st = one.generate([p], limits[i])
        assert got[i][0] == out[0] == greedy[i][:limits[i]], i
        assert got[i][1]["accept_lengths"] == [a for a in st["accept_lengths"][0] if a], i


def test_sam_only_refills_match_requests_run_alone(lm):
    """The same for BatchedSamOnlyDecoder with a with-counts static corpus: static trees are drafted after refills."""
    from samd_b200 import engine as E, synth
    from samd_b200.batched import BatchedSamOnlyDecoder
    prompts, wants = [], []
    # prompts whose greedy continuation never holds token 0 (the -1 pad corner, see BatchedSamOnlyDecoder)
    for i in range(40):
        p = synth.copy_mix(64 + (29 * i) % 140, 96, 700 + i, p_copy=0.7).tolist()
        w = _plain_greedy(lm, p, 64)
        if 0 not in w:
            prompts.append(p)
            wants.append(w)
        if len(prompts) == 7:
            break
    assert len(prompts) >= 6
    limits = [16 + (23 * i) % 49 for i in range(len(prompts))]
    docs = [w[5:59] for w in wants] + [synth.copy_mix(300, 96, 5).tolist()] + [[i] for i in range(3, 96)]
    static = E.StaticSamDevice.build(docs, 2, with_counts=True)
    mk = lambda B: BatchedSamOnlyDecoder(lm, B, 512, max_predicts=16, alpha=4.0, K=4, len_bias=0, static=static,
                                         dtype=torch.float32)
    dec = mk(3)
    got = _serve(dec, prompts, limits)
    assert dec.serve_stats["tree_steps"] > 0 and dec.serve_stats["admissions"] == len(prompts)
    one = mk(1)
    for i, p in enumerate(prompts):
        out, st = one.generate([p], limits[i])
        assert got[i][0] == out[0] == wants[i][:limits[i]], i
        assert got[i][1]["accept_lengths"] == [a for a in st["accept_lengths"][0] if a], i


def test_token_recycle_tree_serve_is_lossless(lm, work):
    """Token-Recycle tree mode shares one successor table across requests, so the drafts depend on the admission order;
    the tokens must still be plain greedy decoding."""
    from samd_b200 import synth
    prompts, limits, greedy = work
    dec = _samd(lm, 4, len_threshold=6, tree=synth.token_recycle_tree())      # most steps draft the tree
    got = _serve(dec, prompts, limits)
    for i, (tokens, _) in got.items():
        assert tokens == greedy[i][:limits[i]], i


def test_eos_and_fewer_steps_than_lockstep(lm, work):
    prompts, limits, greedy = work
    counts = np.bincount(np.concatenate([g[:limits[i]] for i, g in enumerate(greedy)]), minlength=96)
    eos = int(counts.argmax())
    got = _serve(_samd(lm, 4, eos_token_id=eos), prompts, limits)
    cut = 0
    for i, (tokens, _) in got.items():
        w = greedy[i][:limits[i]]
        want = w[:w.index(eos) + 1] if eos in w else w
        cut += len(want) < len(w)
        assert tokens == want, i
    assert cut >= 2
    # one long request per group of 4: lockstep decoding waits for it in every group, serve() overlaps the long ones
    skew = [96 if i % 4 == 0 else 8 for i in range(12)]
    dec = _samd(lm, 4)
    got = _serve(dec, prompts[:12], skew)
    for i, (tokens, _) in got.items():
        assert tokens == greedy[i][:skew[i]], i
    lockstep = sum(dec.generate(prompts[g:g + 4], max(skew[g:g + 4]))[1]["steps_run"] for g in range(0, 12, 4))
    assert dec.serve_stats["steps_run"] < lockstep


def test_admission_leaves_other_requests_untouched():
    """Engine level: B = 8 automata with a static cursor each; admitting slot 3 (masked reset + ingestion with count 0
    for every other request) changes nothing of the others - states, edges, meta words, cursors - and slot 3 equals
    the oracle's automaton over the new prompt alone.  Vocabulary 1000: the root alone has hundreds of out-edges, far
    more than a record holds inline, so overflow slots are in use."""
    from samd_b200 import _cabi as K, engine as E, synth
    B, V, n = 8, 1000, 3000
    docs = [synth.copy_mix(2000, V, 50 + k, p_copy=0.6).tolist() for k in range(4)]
    corpus = np.concatenate([np.asarray(d) for d in docs])
    static = E.StaticSamDevice.build(docs, synth.EOS)
    streams = [synth.copy_mix(n, V, 80 + b, p_copy=0.6, source=corpus, p_source=0.5) for b in range(B)]
    mk = lambda R: E.DraftEngine(E.DynSamBatch(R, 4 * n), static, K.FLAVOUR_SAMD, n_predicts=16, len_bias=2,
                                 len_threshold=4)
    eng = mk(B)
    lens = [n - 97 * b for b in range(B)]
    tok = torch.zeros(B, n, dtype=torch.int32)
    for b in range(B):
        tok[b, :lens[b]] = torch.as_tensor(streams[b][:lens[b]])
    eng.step(tok.cuda(), torch.tensor(lens, dtype=torch.int32, device="cuda"),
             torch.tensor([int(s[-1]) for s in streams], dtype=torch.int32, device="cuda"))

    def snapshot():
        torch.cuda.synchronize()
        meta = eng.dyn.meta()
        return [(eng.dyn.export(b), eng.dyn.export_edges(b), meta[b].copy(), eng.static_cursor[b].tolist()) for b in range(B)]

    before = snapshot()
    new = synth.copy_mix(2500, V, 999, p_copy=0.6, source=corpus, p_source=0.5)
    mask = torch.zeros(B, dtype=torch.uint8, device="cuda")
    mask[3] = 1
    eng.reset(mask)
    tok = torch.zeros(B, len(new), dtype=torch.int32)
    tok[3] = torch.as_tensor(new)
    counts = torch.zeros(B, dtype=torch.int32)
    counts[3] = len(new)
    eng.step(tok.cuda(), counts.cuda(), None)
    after = snapshot()
    for b in range(B):
        if b == 3:
            continue
        (ea, ga, ma, ca), (eb, gb, mb, cb) = before[b], after[b]
        assert ea.keys() == eb.keys()
        for k in ea:
            assert np.array_equal(ea[k], eb[k]), (b, k)
        assert np.array_equal(ga, gb) and np.array_equal(ma, mb) and ca == cb, b
    ex, edges, _, cursor = after[3]
    ora = O.Automaton()
    ora.extend(new)
    assert ex["overflow"] == 0 and ex["n_states"] == len(ora.link)
    assert np.array_equal(ex["link"], ora.link) and np.array_equal(ex["length"], ora.length)
    assert np.array_equal(ex["min_endpos"], ora.first_end) and np.array_equal(ex["text"][1:], new)
    want = sorted((s, t, d) for s, tr in enumerate(ora.trans) for t, d in tr.items())
    assert sorted(map(tuple, edges.tolist())) == want
    assert max(len(tr) for tr in ora.trans) > 16
    # the static cursor is that of a fresh request fed the same prompt
    fresh = mk(1)
    fresh.step(torch.as_tensor(new[None], dtype=torch.int32).cuda(), None, None)
    torch.cuda.synchronize()
    assert cursor == fresh.static_cursor[0].tolist()


def test_serve_edge_cases(lm, work):
    from samd_b200 import _cabi as K
    prompts, limits, greedy = work
    dec = _samd(lm, 4)
    # fewer requests than slots: the idle slots never emit
    got = _serve(dec, prompts[:2], 24)
    assert {info["slot"] for _, info in got.values()} == {0, 1}
    assert [got[i][0] for i in range(2)] == [greedy[i][:24] for i in range(2)]
    assert dec._st["out_len"][2:].tolist() == [0, 0] and dec.serve_stats["admissions"] == 2
    # generate -> serve -> generate on one decoder
    out, _ = dec.generate(prompts[:4], 32)
    assert out == [g[:32] for g in greedy[:4]]
    got = _serve(dec, prompts[4:11], 32)
    assert [got[i][0] for i in range(7)] == [g[:32] for g in greedy[4:11]]
    out, _ = dec.generate(prompts[8:12], 40)
    assert out == [g[:40] for g in greedy[8:12]]
    # an abandoned generator, then generate(); a generator suspended across another call refuses to go on
    it = dec.serve(prompts, limits)
    next(it)
    del it
    out, _ = dec.generate(prompts[1:5], 48)
    assert out == [g[:48] for g in greedy[1:5]]
    it = dec.serve(prompts, limits)
    next(it)
    out, _ = dec.generate(prompts[:4], 16)
    assert out == [g[:16] for g in greedy[:4]]
    with pytest.raises(K.SamdError, match="suspended"):
        next(it)
    # an invalid request ends the call with its index; the requests finished before it are exact, the decoder usable
    bad = prompts[:6] + [[]] + prompts[6:]
    seen = {}
    with pytest.raises(K.SamdError, match="request 6: empty prompt"):
        for i, tokens, _ in dec.serve(bad, 8):
            seen[i] = tokens
    assert all(seen[i] == greedy[i][:8] for i in seen)
    for args, msg in (((prompts[:3], [8, 8]), "request 2: max_new_tokens has 2 values"),
                      ((prompts[:3], [8, 0, 8]), "request 1: max_new_tokens must be >= 1"),
                      ((prompts[:2] + [list(range(3, 96)) * 6], 8), "request 2: prompt of 558 tokens"),
                      ((prompts[:2], 20000), "request 0: prompt \\+ max_new_tokens")):
        with pytest.raises(K.SamdError, match=msg):
            list(dec.serve(*args))
    out, _ = dec.generate(prompts[:4], 24)
    assert out == [g[:24] for g in greedy[:4]]
