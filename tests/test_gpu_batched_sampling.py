"""GPU tests of sampled decoding in the batched decoders: samd_verify_sample_requests against the oracle per request (own
processor, own width, greedy and finished requests mixed in one launch), the decoders' reproducibility per request, greedy
requests inside a sampled call, exactness in distribution at temperature 1, EOS, and the refusal in tree mode."""
import numpy as np
import pytest
import torch

import samd_oracle as O

pytestmark = pytest.mark.gpu

N_REQ = 13


def _tiny_llama(head_scale: float = 1.0):
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=96, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, max_position_embeddings=2048, attn_implementation="eager")
    lm = LlamaForCausalLM(cfg).to("cuda", torch.float32).eval()
    with torch.no_grad():
        lm.lm_head.weight.mul_(head_scale)
    return lm


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
    from samd_b200 import synth
    from samd_b200.batched import SamplingParams
    lens = (150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70)
    prompts = [synth.copy_mix(n, 96, 300 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    limits = [8, 96] + [8 + (37 * i) % 89 for i in range(2, N_REQ)]
    procs = [dict(temperature=1.0), dict(temperature=0.7, top_p=0.9), dict(temperature=1.3, top_k=5),
             dict(temperature=0.8, top_p=0.85, top_k=8), dict(greedy=True)]
    params = [SamplingParams(seed=1000 + 7 * i, **procs[i % len(procs)]) for i in range(N_REQ)]
    return prompts, limits, params


# ---- 1. the kernel, per request, against the oracle -------------------------------------------------------------------
def _rand_tree(rng, n):
    """Root-to-leaf paths of a random n-node tree (parents precede children), leaves in index order."""
    par = [-1] + [int(rng.integers(0, i)) for i in range(1, n)]
    leaves = [i for i in range(n) if i not in par]
    paths = []
    for leaf in leaves:
        p, j = [], leaf
        while j >= 0:
            p.append(j)
            j = par[j]
        paths.append(p[::-1])
    return par, paths


@pytest.mark.parametrize("dt,B,V", [("fp32", 48, 997), ("bf16", 48, 997), ("fp16", 48, 997), ("bf16", 64, 128256)])
def test_kernel_per_request_matches_oracle(dt, B, V):
    """One launch: sampled trees and sequences of their own width inside a D-wide table (-1 pads beyond), each with its
    own temperature / top-p / top-k and stream; greedy requests; finished requests (done flag, and n_paths 0)."""
    from samd_b200 import engine as E
    T = P = D = 16
    rng = np.random.default_rng(7 + V)
    tokens = rng.integers(1, V, size=(B, T)).astype(np.int32)
    ret = np.full((B, P, D), -1, dtype=np.int32)
    n_nodes, n_paths, depth = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
    kinds, parents = [], []
    for b in range(B):
        kind = ("tree", "seq", "greedy", "done", "nopath", "full")[b % 6]
        kinds.append(kind)
        if kind in ("tree", "greedy", "nopath"):
            n = int(rng.integers(6, T + 1))
            par, paths = _rand_tree(rng, n)
            for p, path in enumerate(paths):
                ret[b, p, :len(path)] = path
            n_nodes[b], n_paths[b] = n, len(paths)
            depth[b] = D if kind == "greedy" else max(len(x) for x in paths)     # greedy: the full table, as verify_compact
            if len(paths) > 1 and rng.random() < 0.5:                           # sibling duplicates of one candidate token
                tokens[b, paths[1][1]] = tokens[b, paths[0][1]]
        else:
            n = T if kind == "full" else int(rng.integers(2, T))
            par = [-1] + list(range(n - 1))
            ret[b, 0, :n] = np.arange(n)
            n_nodes[b], n_paths[b], depth[b] = n, 1, n
        if kind == "nopath":
            n_paths[b] = 0
        parents.append(par)
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[dt]
    g = torch.Generator(device="cuda").manual_seed(V)
    lg = torch.randn(B, T, V, generator=g, device="cuda") * 2.0
    for b in range(B):                                                          # proposals that are often accepted
        for c in range(1, n_nodes[b]):
            if rng.random() < 0.8:
                lg[b, parents[b][c], int(tokens[b, c])] += 4.0
    lg = lg.to(tdt)
    lg_np = lg.float().cpu().numpy()
    temps = np.array([(1.0, 0.7, 1.3, 0.9)[(b // 6) % 4] for b in range(B)], np.float32)
    top_ps = np.array([(0.0, 0.9, 0.8, 0.0)[(b // 6) % 4] for b in range(B)], np.float32)
    top_ks = np.array([(0, 0, 5, 8)[(b // 6) % 4] for b in range(B)], np.int32)
    greedy = np.array([k == "greedy" for k in kinds], np.uint8)
    done = np.array([k == "done" for k in kinds], np.uint8)
    cu = lambda a: torch.as_tensor(a).cuda()
    seeds = cu(rng.integers(1, 2 ** 62, size=B))
    off0 = rng.integers(0, 2 ** 40, size=B)
    offs = cu(off0.copy())
    ver = E.Verifier(B, T)
    sentinel = lambda *s: torch.full(s, -7, dtype=torch.int32, device="cuda")
    out = dict(best=sentinel(B), accept_len=sentinel(B), next_token=sentinel(B), tokens=sentinel(B, D),
               indices=sentinel(B, D))
    got = ver.verify_sample(lg, cu(tokens), cu(ret), cu(temps), cu(top_ps), cu(top_ks), seeds, offs, n_paths=cu(n_paths),
                            greedy=cu(greedy), done=cu(done), n_nodes=cu(n_nodes), depth=cu(depth), out=out)
    assert got is out
    # the accepted rows move into place with samd_kv_compact; finished requests move nothing
    kv = [torch.randn(B, 2, 64, 16, device="cuda").to(torch.float16) for _ in range(4)]
    kv_ref = [t.cpu().view(torch.int16).numpy().copy() for t in kv]
    ver.bind_kv(kv)
    cache_len = torch.full((B,), 20, dtype=torch.int32, device="cuda")
    ver.kv_compact(out["indices"], out["accept_len"], cache_len)
    want_g = ver.verify(lg, cu(tokens), cu(ret), move_kv=False, n_nodes=cu(n_nodes), n_paths=cu(n_paths))
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res_g = {k: v.cpu().numpy() for k, v in want_g.items()}
    kv_now = [t.cpu().view(torch.int16).numpy() for t in kv]
    offs_now, cl = offs.cpu().numpy(), cache_len.cpu().numpy()
    compared = sampled = 0
    for b in range(B):
        kind = kinds[b]
        if kind in ("done", "nopath"):
            assert res["accept_len"][b] == 0 and offs_now[b] == off0[b] and cl[b] == 20, b
            assert res["best"][b] == res["next_token"][b] == -7 and (res["tokens"][b] == -7).all(), b
            assert all(np.array_equal(now[b], ref[b]) for now, ref in zip(kv_now, kv_ref)), b
            continue
        if kind == "greedy":
            for k in ("best", "accept_len", "next_token"):
                assert res[k][b] == res_g[k][b], (b, k)
            n = res["accept_len"][b]
            assert np.array_equal(res["tokens"][b, :n], res_g["tokens"][b, :n]) and (res["tokens"][b, n:] == -1).all(), b
            assert offs_now[b] == off0[b], b
            continue
        sampled += 1
        k = [0]

        def draw():
            u = O.philox_uniform(int(seeds[b]), int(off0[b]) + k[0])
            k[0] += 1
            return u

        nb, db = n_nodes[b], depth[b]
        want = O.verify_typical(lg_np[b, :nb], tokens[b, :nb], ret[b, :n_paths[b], :db].astype(np.int64),
                                float(temps[b]), float(top_ps[b]), int(top_ks[b]), draw)
        if min(want["margins"][:-1], default=1.0) < 1e-4:                   # a razor-edge accept / reject decision
            continue
        compared += 1
        n = want["accept_len"]
        assert (res["best"][b], res["accept_len"][b]) == (want["best"], n), b
        # the next token: the oracle's, or - where u lies within float32 rounding of a step of the CDF (at V = 128256 the
        # steps are ~1e-5 apart) - a token whose CDF interval reaches u
        got_t = int(res["next_token"][b])
        if got_t != want["next_token"]:
            cdf = np.cumsum(want["sample_p"]) / want["sample_p"].sum()
            u = O.philox_uniform(int(seeds[b]), int(off0[b]) + k[0] - 1)
            lo = cdf[got_t - 1] if got_t else 0.0
            assert want["margins"][-1] < 1e-5 and want["sample_p"][got_t] > 0 and lo - 1e-5 <= u <= cdf[got_t] + 1e-5, b
        assert res["tokens"][b, :n].tolist() == want["tokens"] and res["indices"][b, :n].tolist() == want["indices"], b
        assert (res["tokens"][b, n:] == -1).all() and (res["indices"][b, n:] == -1).all(), b
        assert offs_now[b] - off0[b] == k[0], b
        assert cl[b] == 20 + n, b
        for now, ref in zip(kv_now, kv_ref):
            r = [ref[b].copy()]
            O.kv_compact(r, 20, np.asarray(want["indices"]), n)
            assert np.array_equal(now[b], r[0]), b
    assert compared >= sampled * 3 // 4 and sampled >= B // 3


# ---- 2. reproducibility of every request ------------------------------------------------------------------------------
def _serve(dec, prompts, limits, **kw):
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info["accept_lengths"])
    assert sorted(got) == list(range(len(prompts)))
    return got


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


@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_sampled_requests_are_reproducible(lm, work, flavour):
    """A request's tokens and accept lengths depend only on its prompt, parameters and seed: serve() at B = 4 with 13
    requests, each decoded alone at B = 1, eager, check_every 1, generate(), and a prefix pool (one prompt equal to a
    registered prefix)."""
    prompts, limits, params = work
    mk = _decoders(lm)[flavour]
    dec = mk(4)
    ref = _serve(dec, prompts, limits, sampling=params)
    assert dec.serve_stats["graphed"]
    for i in range(N_REQ):
        assert len(ref[i][0]) == limits[i] and all(a > 0 for a in ref[i][1]), i
    one = mk(1)
    for i, p in enumerate(prompts):
        out, st = one.generate([p], limits[i], sampling=[params[i]])
        assert (out[0], [a for a in st["accept_lengths"][0] if a]) == ref[i], i
    assert _serve(dec, prompts, limits, sampling=params, graph=False) == ref
    assert _serve(dec, prompts, limits, sampling=params, check_every=1) == ref
    out, st = dec.generate(prompts[4:8], 24, sampling=params[4:8])
    for k in range(4):
        n = min(24, limits[4 + k])
        assert out[k][:n] == ref[4 + k][0][:n], 4 + k
    pooled = mk(4, max_prefixes=2)
    pooled.add_prefix(prompts[1])
    pooled.add_prefix(prompts[6][:40])
    got = {}
    for i, tokens, info in pooled.serve(prompts, limits, sampling=params):
        got[i] = (tokens, info["accept_lengths"])
        assert info["prefix_len"] == {1: len(prompts[1]), 6: 40}.get(i, 0), i
    assert got == ref
    # a shared SamplingParams gives request i the seed + i: the same as the per-request list with those seeds
    from samd_b200.batched import SamplingParams
    shared = SamplingParams(temperature=0.7, top_p=0.9, seed=50)
    a = _serve(dec, prompts[:6], limits[:6], sampling=shared)
    b = _serve(dec, prompts[:6], limits[:6], sampling=[SamplingParams(temperature=0.7, top_p=0.9, seed=50 + i)
                                                       for i in range(6)])
    assert a == b
    # sampled decoding really samples: the sampled requests differ from greedy decoding somewhere
    greedy = _serve(dec, prompts, limits)
    assert sum(ref[i][0] != greedy[i][0] for i in range(N_REQ) if not params[i].greedy) >= 5


# ---- 3. greedy requests in a sampled call -----------------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_greedy_requests_in_a_sampled_call_are_plain_greedy(lm, work, flavour):
    from samd_b200.batched import BatchedSamOnlyDecoder, SamplingParams
    prompts, limits, _ = work
    if flavour == "samd":
        dec = _decoders(lm)["samd"](4)
    else:                                       # sequences only: every draft is as wide as its own width, no pad column
        dec = BatchedSamOnlyDecoder(lm, 4, 512, max_predicts=16, alpha=4.0, dtype=torch.float32)
    params = [SamplingParams(greedy=True) if i % 2 == 0 else SamplingParams(temperature=1.3, top_k=20, seed=i)
              for i in range(N_REQ)]
    got = _serve(dec, prompts, limits, sampling=params)
    plain = _serve(dec, prompts, limits) if flavour == "samd" else None
    for i in range(0, N_REQ, 2):
        assert got[i][0] == _plain_greedy(lm, prompts[i], limits[i]), i
        if flavour == "samd":
            assert got[i] == plain[i], i                    # the same accept lengths too: sequences have no pad column


# ---- 4. exactness in distribution -------------------------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_temperature_one_is_exact_in_distribution(flavour):
    """tau = 1, no top-p / top-k: typical acceptance is exact, so the first token of 4096 requests with distinct seeds
    follows the LM's softmax after the prompt, and the second one, given each of the three most frequent first tokens,
    the softmax after prompt + that token - within 5 sigma of binomial error, while drafts are really accepted."""
    from samd_b200 import synth
    from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder, SamplingParams
    # a sharp LM (top probabilities ~0.5 along its greedy continuation): its own continuations, drafted from the prompt,
    # often pass
    lm = _tiny_llama(head_scale=25.0)
    s = synth.copy_mix(24, 96, 77).tolist()
    prompt = s + _plain_greedy(lm, s, 40) + s
    N, B = 4096, 128
    if flavour == "samd":
        dec = BatchedSamdDecoder(lm, B, 256, n_predicts=8, len_bias=5, len_threshold=1, dtype=torch.float32)
    else:
        dec = BatchedSamOnlyDecoder(lm, B, 256, max_predicts=8, alpha=4.0, dtype=torch.float32)
    first, second, steps, drafted = [], [], 0, 0
    for i, tokens, info in dec.serve([prompt] * N, 3, sampling=SamplingParams(seed=12345)):
        first.append(tokens[0])
        second.append(tokens[1])
        steps += len(info["accept_lengths"])
        drafted += sum(a > 1 for a in info["accept_lengths"])
    assert drafted >= 0.2 * steps, (drafted, steps)
    first, second = np.asarray(first), np.asarray(second)

    @torch.inference_mode()
    def softmax_after(ids):
        return torch.softmax(lm(input_ids=torch.as_tensor([ids]).cuda()).logits[0, -1].double(), -1).cpu().numpy()

    def close(counts, p, what):
        n = counts.sum()
        tol = 5.0 * np.sqrt(n * p * (1 - p)) + 1.0
        bad = np.abs(counts - n * p) > tol
        assert not bad.any(), (what, np.nonzero(bad)[0][:5].tolist(), counts[bad][:5].tolist(), (n * p)[bad][:5].tolist())

    h1 = np.bincount(first, minlength=96)
    close(h1, softmax_after(prompt), "first token")
    for t in np.argsort(-h1)[:3]:
        sel = first == t
        close(np.bincount(second[sel], minlength=96), softmax_after(prompt + [int(t)]), f"second token after {t}")


# ---- 5. EOS and limits; 6. tree mode ----------------------------------------------------------------------------------
def test_eos_truncation_and_limits(lm, work):
    prompts, limits, params = work
    mk = _decoders(lm)["samd"]
    free = _serve(mk(4), prompts, limits, sampling=params)
    counts = np.bincount(np.concatenate([free[i][0] for i in range(N_REQ)]), minlength=96)
    eos = int(counts.argmax())
    got = _serve(mk(4, eos_token_id=eos), prompts, limits, sampling=params)
    cut = 0
    for i in range(N_REQ):
        w = free[i][0]
        want = w[:w.index(eos) + 1] if eos in w else w
        cut += len(want) < len(w)
        assert got[i][0] == want and len(got[i][0]) <= limits[i], i
    assert cut >= 2


def test_tree_mode_refuses_sampling(lm, work):
    from samd_b200 import _cabi as K, synth
    from samd_b200.batched import SamplingParams
    prompts, _, _ = work
    dec = _decoders(lm)["samd"](4, tree=synth.token_recycle_tree())
    with pytest.raises(K.SamdError, match="tree mode"):
        dec.generate(prompts[:4], 8, sampling=SamplingParams())
    with pytest.raises(K.SamdError, match="tree mode"):
        list(dec.serve(prompts, 8, sampling=SamplingParams()))
    out, _ = dec.generate(prompts[:4], 8)
    assert out == [_plain_greedy(lm, p, 8) for p in prompts[:4]]
