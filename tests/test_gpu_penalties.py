"""GPU tests of repetition / presence / frequency penalties: samd_apply_penalties against a torch restatement, bit for bit
(identity chains and random trees, repeated, history and path-only tokens, untouched rows and requests, -inf and NaN, the
admission form, graph and eager), and the decoders' penalties= against plain penalized greedy decoding, HF generate(),
neutral Penalties() against None, sampled reproducibility and distribution, and log-probabilities of penalized rows."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N_REQ = 13
V_LM = 96
NAN = float("nan")


def _tiny_llama(head_scale: float = 1.0):
    """The fp32 tiny Llama of the log-probability tests: token 0 is never its argmax, so a -1 pad of a path table is never
    "accepted" (the reference's A9 corner, see BatchedSamOnlyDecoder)."""
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
def _penalize_row(x: torch.Tensor, hist: torch.Tensor, prompt: torch.Tensor, r: float, p: float, f: float) -> torch.Tensor:
    """One logits row [V] (any dtype) with output counts `hist` [V] int (emitted + path tokens) and `prompt` [V] bool: the
    documented formula, each operation a separate fp32 torch op (per-element tensors, so x / r is a true division), one
    rounding into the row's dtype; unseen entries are the input's."""
    dev = x.device
    rt, pt, ft = (torch.tensor([v], dtype=torch.float32, device=dev) for v in (r, p, f))
    c = hist.to(dev)
    seen = prompt.to(dev) | (c > 0)
    y = x.float()
    y = torch.where(y < 0, y * rt, y / rt)
    y = y - ft * c.float()
    y = y - pt * (c > 0).float()
    return torch.where(seen, y.to(x.dtype), x)


def _row_counts(tokens, V):
    return torch.bincount(torch.as_tensor(list(tokens), dtype=torch.long), minlength=V)


def _paths(tokens_b, ret_b, n, n_paths):
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


def _restate(lg, counts, r, p, f, tokens=None, ret=None, n_nodes=None, n_paths=None, done=None, slots=None):
    want = lg.clone()
    B, T, V = lg.shape
    cnt = counts.cpu()
    for b in range(B):
        s = b if slots is None else int(slots[b])
        if (done is not None and done[b]) or (r[s] == 1.0 and p[s] == 0.0 and f[s] == 0.0):
            continue
        n = T if n_nodes is None else min(T, int(n_nodes[b]))
        if tokens is None:
            rows = {j: [] for j in range(n)}
        elif ret is None:
            rows = {j: list(range(j + 1)) for j in range(n)}
        else:
            rows = _paths(tokens[b], ret[b], n, ret.shape[1] if n_paths is None else int(n_paths[b]))
        hist, prompt = (cnt[s] & 0x7FFFFFFF).long(), cnt[s] < 0
        for j, nodes in rows.items():
            c = hist + _row_counts([int(tokens[b, k]) for k in nodes], V)
            want[b, j] = _penalize_row(lg[b, j], c, prompt, float(r[s]), float(p[s]), float(f[s]))
    return want


def _same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    """Bit-identical, except that any NaN matches any NaN."""
    ia = a.view(torch.int32 if a.dtype == torch.float32 else torch.int16)
    ib = b.view(ia.dtype)
    return bool(((ia == ib) | (torch.isnan(a) & torch.isnan(b))).all())


def _random_tree(rng, n):
    """parents of a random tree over n nodes (node 0 the root) and its leaf paths."""
    parent = [-1] + [int(rng.integers(0, j)) for j in range(1, n)]
    kids = {j for j in parent if j >= 0}
    paths = []
    for leaf in (j for j in range(n) if j not in kids):
        path = [leaf]
        while parent[path[-1]] >= 0:
            path.append(parent[path[-1]])
        paths.append(path[::-1])
    return paths


# ---- 1. the kernel against the restatement ------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [997, 32000, 128256])
@pytest.mark.parametrize("dt", ["fp32", "bf16", "fp16"])
def test_kernel_matches_torch(dt, V):
    from samd_b200 import engine as E
    B, T, P = 12, 12, 12
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[dt]
    rng = np.random.default_rng(V + len(dt))
    g = torch.Generator(device="cuda").manual_seed(V)
    lg = (torch.randn(B, T, V, generator=g, device="cuda") * 3.0).to(tdt)
    pool = rng.choice(V, size=24, replace=False)                 # a small pool: repeats on paths, history on paths
    tokens = pool[rng.integers(0, len(pool), size=(B, T))].astype(np.int32)
    counts = np.zeros((B, V), np.int64)
    for b in range(B):
        hist = rng.choice(V, size=40, replace=False)
        counts[b, hist[:30]] = rng.integers(1, 6, size=30)        # emitted
        counts[b, hist[20:]] |= 1 << 31                           # prompt (10 of them also emitted)
        counts[b, pool[:6]] += rng.integers(0, 3, size=6)         # pool tokens in the history too (or not)
    r = rng.choice([1.3, 0.7, 1.0, 1.1], size=B).astype(np.float32)
    p = rng.choice([0.0, 0.5, -0.3], size=B).astype(np.float32)
    f = rng.choice([0.0, 0.25, 1.5], size=B).astype(np.float32)
    r[3], p[3], f[3] = 1.0, 0.0, 0.0                              # neutral
    r[5], p[5], f[5] = 1.2, 0.4, 0.6
    counts[5] &= 1 << 31                                          # prompt bits alone (history emptied), ...
    tokens[5] = pool[0]                                           # ... and every node the same path-only token
    counts[5, pool[0]] = 0
    done = np.zeros(B, np.uint8)
    done[7] = 1
    n_nodes = rng.integers(T // 2, T + 1, size=B).astype(np.int32)
    n_nodes[[1, 5]] = T
    ret = np.full((B, P, T), -1, np.int32)
    n_paths = np.zeros(B, np.int32)
    for b in range(B):
        paths = _random_tree(rng, int(n_nodes[b])) if b % 3 else [list(range(int(n_nodes[b])))]   # trees and chains
        n_paths[b] = len(paths)
        for k, path in enumerate(paths):
            ret[b, k, :len(path)] = path
    # -inf and NaN on history and path tokens
    lg[0, :, int(np.nonzero(counts[0])[0][0])] = float("-inf")
    lg[0, 2, int(tokens[0, 0])] = NAN
    lg[1, 1, int(np.nonzero(counts[1])[0][1])] = NAN
    cu = lambda a, t=None: torch.as_tensor(a, dtype=t).cuda()
    cnt = cu(counts.astype(np.uint32).view(np.int32))
    rr, pp, ff = cu(r), cu(p), cu(f)
    tok, nn, done_t = cu(tokens), cu(n_nodes), cu(done)

    # a path table with per-request node and path counts
    got = lg.clone()
    E.apply_penalties(got, cnt, rr, pp, ff, tokens=tok, retrieve=cu(ret), n_nodes=nn, n_paths=cu(n_paths), done=done_t)
    want = _restate(lg, cnt, r, p, f, tokens, ret, n_nodes, n_paths, done)
    assert _same_bits(got, want)
    for b in (3, 7):                                              # neutral and finished: untouched
        assert torch.equal(got[b].view(torch.int16 if tdt != torch.float32 else torch.int32),
                           lg[b].view(torch.int16 if tdt != torch.float32 else torch.int32)), b
    assert not torch.equal(got[5], lg[5])                         # the prompt bits and a path-only token do act
    assert got[0, 0, int(np.nonzero(counts[0])[0][0])].item() == float("-inf")
    assert torch.isnan(got[0, 2, int(tokens[0, 0])]).item()

    # the identity chain (samd sequences)
    got = lg.clone()
    E.apply_penalties(got, cnt, rr, pp, ff, tokens=tok, n_nodes=nn, done=done_t)
    assert _same_bits(got, _restate(lg, cnt, r, p, f, tokens, None, n_nodes, None, done))

    # the admission form: one row per admitted request, no draft context, state rows through slots
    slots = np.array([9, 2, 5, 0], np.int32)
    rows = lg[:4, :1].clone()
    got = rows.clone()
    E.apply_penalties(got, cnt, rr, pp, ff, slots=cu(slots))
    assert _same_bits(got, _restate(rows, cnt, r, p, f, slots=slots))

    # graph and eager: the same bits
    eager = lg.clone()
    E.apply_penalties(eager, cnt, rr, pp, ff, tokens=tok, retrieve=cu(ret), n_nodes=nn, n_paths=cu(n_paths), done=done_t)
    graphed = lg.clone()
    args = (cnt, rr, pp, ff)
    kw = dict(tokens=tok, retrieve=cu(ret), n_nodes=nn, n_paths=cu(n_paths), done=done_t)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        E.apply_penalties(graphed, *args, **kw)
    graphed.copy_(lg)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(graphed.view(torch.uint8), eager.view(torch.uint8))


# ---- 2. lossless penalized greedy decoding ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lm():
    return _tiny_llama()


@pytest.fixture(scope="module")
def work():
    from samd_b200 import synth
    from samd_b200.batched import Penalties
    lens = (150, 97, 200, 64, 120, 180, 88, 140, 110, 76, 160, 130, 70)
    prompts = [synth.copy_mix(n, V_LM, 300 + i, p_copy=0.7).tolist() for i, n in enumerate(lens)]
    limits = [8, 96] + [8 + (37 * i) % 89 for i in range(2, N_REQ)]
    kinds = [Penalties(repetition_penalty=1.3), Penalties(presence_penalty=0.5, frequency_penalty=0.5), Penalties(),
             Penalties(1.1, 0.3, 0.2), Penalties(repetition_penalty=0.8, frequency_penalty=-0.4)]
    pens = [kinds[i % len(kinds)] for i in range(N_REQ)]
    return prompts, limits, pens


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


@torch.inference_mode()
def _penalized_greedy(lm, prompt, n_new, pn, eos=None):
    """Plain greedy decoding with the restatement applied to logits[:, -1] before the argmax."""
    ids = torch.as_tensor([prompt]).cuda()
    prompt_seen = _row_counts(prompt, V_LM) > 0
    gen = []
    for _ in range(n_new):
        row = lm(input_ids=ids).logits[0, -1]
        row = _penalize_row(row, _row_counts(gen, V_LM), prompt_seen, pn.repetition_penalty, pn.presence_penalty,
                            pn.frequency_penalty)
        nxt = int(row.argmax())
        gen.append(nxt)
        if nxt == eos:
            break
        ids = torch.cat([ids, torch.tensor([[nxt]], device="cuda")], 1)
    return gen


def _serve(dec, prompts, limits, **kw):
    got = {}
    for i, tokens, info in dec.serve(prompts, limits, **kw):
        assert i not in got
        got[i] = (tokens, info)
    assert sorted(got) == list(range(len(prompts)))
    return got


@pytest.fixture(scope="module")
def reference(lm, work):
    prompts, limits, pens = work
    return [_penalized_greedy(lm, prompts[i], limits[i], pens[i]) for i in range(N_REQ)]


@pytest.mark.parametrize("mode", ["samd", "samd_tree", "sam_only"])
def test_penalized_greedy_is_lossless(lm, work, reference, mode):
    """serve() at B = 4 over 13 requests with mixed per-request penalties (neutral ones included) equals plain penalized
    greedy decoding: graphed and eager, check_every 4 and 1, with a prefix pool, with EOS, and through generate()."""
    from samd_b200 import synth
    prompts, limits, pens = work
    flavour = mode.replace("_tree", "")
    kw = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    mk = _decoders(lm)[flavour]
    dec = mk(4, **kw)
    for run in (dict(), dict(graph=False, check_every=1)):
        got = _serve(dec, prompts, limits, penalties=pens, **run)
        assert dec.serve_stats["graphed"] == run.get("graph", True)
        for i in range(N_REQ):
            assert got[i][0] == reference[i], (run, i)
    assert sum(sum(a > 1 for a in got[i][1]["accept_lengths"]) for i in range(N_REQ)) > 0     # drafts accepted
    pooled = mk(4, max_prefixes=2, **kw)
    pooled.add_prefix(prompts[1])
    pooled.add_prefix(prompts[6][:40])
    pgot = _serve(pooled, prompts, limits, penalties=pens)
    assert pgot[1][1]["prefix_len"] == len(prompts[1]) and pgot[6][1]["prefix_len"] == 40
    for i in range(N_REQ):
        assert pgot[i][0] == reference[i], i
    counts = np.bincount(np.concatenate(reference), minlength=V_LM)
    eos = int(counts.argmax())
    egot = _serve(mk(4, eos_token_id=eos, **kw), prompts, limits, penalties=pens)
    cut = 0
    for i in range(N_REQ):
        w = reference[i]
        want = w[:w.index(eos) + 1] if eos in w else w
        cut += len(want) < len(w)
        assert egot[i][0] == want, i
    assert cut >= 1
    out, _ = dec.generate(prompts[4:8], 24, penalties=pens[4:8])
    assert out == [reference[i][:24] if limits[i] >= 24 else _penalized_greedy(lm, prompts[i], 24, pens[i])
                   for i in range(4, 8)]


@torch.inference_mode()
def test_repetition_only_equals_hf_generate(lm, work):
    from samd_b200.batched import Penalties
    prompts, _, _ = work
    dec = _decoders(lm)["samd"](4)
    rs = (1.3, 1.1, 0.8, 2.0)
    out, _ = dec.generate(prompts[:4], 24, penalties=[Penalties(repetition_penalty=r) for r in rs])
    for k, r in enumerate(rs):
        ids = torch.as_tensor([prompts[k]]).cuda()
        hf = lm.generate(ids, attention_mask=torch.ones_like(ids), do_sample=False, repetition_penalty=r,
                         max_new_tokens=24, use_cache=False, pad_token_id=0)[0, ids.shape[1]:].tolist()
        assert hf and out[k][:len(hf)] == hf, (r, out[k], hf)          # (generate() stops at the config's EOS)
        assert out[k] == _penalized_greedy(lm, prompts[k], 24, Penalties(repetition_penalty=r))


# ---- 3. neutral penalties and None --------------------------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_neutral_is_none(lm, work, flavour):
    from samd_b200 import engine as E
    from samd_b200.batched import Penalties
    prompts, limits, _ = work
    dec = _decoders(lm)[flavour](4)
    base = _serve(dec, prompts, limits)
    assert "pen_counts" not in dec._st                            # penalties=None allocates nothing
    neutral = _serve(dec, prompts, limits, penalties=Penalties())
    for i in range(N_REQ):
        assert neutral[i][0] == base[i][0] and neutral[i][1]["accept_lengths"] == base[i][1]["accept_lengths"], i
    n_graphs = len(dec._graphs)
    again = _serve(dec, prompts, limits)                          # None replays the graphs it captured before
    assert len(dec._graphs) == n_graphs
    for i in range(N_REQ):
        assert again[i][0] == base[i][0], i
    # launches, eager: penalties add one per step and one per admission batch; None issues the step's launches only
    # (step + verify; sam_only adds the static tree draft and the assembly)
    per_step = {"samd": 2, "sam_only": 4}[flavour]
    sub, runs = prompts[4:8], {}
    for pn in (None, Penalties()):
        for n_new in (16, 40):
            c0 = E.launch_count()
            _, st = dec.generate(sub, n_new, graph=False, penalties=pn)
            runs[pn is None, n_new] = (E.launch_count() - c0, st["steps_run"])
    for n_new in (16, 40):
        (c_none, s_none), (c_pen, s_pen) = runs[True, n_new], runs[False, n_new]
        assert s_none == s_pen and c_pen - c_none == s_none + 1, (n_new, runs)
    (c1, s1), (c2, s2) = runs[True, 16], runs[True, 40]
    assert s2 > s1 and c2 - c1 == per_step * (s2 - s1), runs


# ---- 4. sampled decoding with penalties ---------------------------------------------------------------------------------
@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_sampled_tokens_depend_only_on_the_request(lm, work, flavour):
    from samd_b200.batched import SamplingParams
    prompts, limits, pens = work
    procs = [dict(temperature=1.0), dict(temperature=0.7, top_p=0.9), dict(temperature=1.3, top_k=5), dict(greedy=True)]
    params = [SamplingParams(seed=1000 + 7 * i, **procs[i % len(procs)]) for i in range(N_REQ)]
    mk = _decoders(lm)[flavour]
    dec = mk(4)
    base = _serve(dec, prompts, limits, sampling=params, penalties=pens)
    eager = _serve(dec, prompts, limits, sampling=params, penalties=pens, graph=False, check_every=1)
    alone = mk(1)
    pooled = mk(4, max_prefixes=1)
    pooled.add_prefix(prompts[6][:40])
    pgot = _serve(pooled, prompts, limits, sampling=params, penalties=pens)
    for i in range(N_REQ):
        one = _serve(alone, [prompts[i]], [limits[i]], sampling=[params[i]], penalties=[pens[i]])[0]
        for other in (eager[i], pgot[i], one):
            assert other[0] == base[i][0] and other[1]["accept_lengths"] == base[i][1]["accept_lengths"], i
    greedy = [i for i in range(N_REQ) if params[i].greedy]
    ref = [_penalized_greedy(lm, prompts[i], limits[i], pens[i]) for i in greedy]
    assert [base[i][0] for i in greedy] == ref


@pytest.mark.parametrize("flavour", ["samd", "sam_only"])
def test_temperature_one_follows_the_penalized_softmax(flavour):
    """The first and second tokens of 4096 seeded requests at temperature 1 with repetition_penalty 1.3 follow the softmax
    of the penalized rows (the prompt's last row; the row after prompt + first token, whose path is node 0) within 5
    sigma of binomial error."""
    from samd_b200 import synth
    from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder, Penalties, SamplingParams
    lm = _tiny_llama(head_scale=25.0)
    s = synth.copy_mix(24, V_LM, 77).tolist()
    pn = Penalties(repetition_penalty=1.3)
    prompt = s + _penalized_greedy(lm, s, 40, Penalties()) + s
    N, B = 4096, 128
    if flavour == "samd":
        dec = BatchedSamdDecoder(lm, B, 256, n_predicts=8, len_bias=5, len_threshold=1, dtype=torch.float32)
    else:
        dec = BatchedSamOnlyDecoder(lm, B, 256, max_predicts=8, alpha=4.0, dtype=torch.float32)
    first, second = [], []
    for i, tokens, info in dec.serve([prompt] * N, 3, sampling=SamplingParams(seed=4321), penalties=pn):
        first.append(tokens[0])
        second.append(tokens[1])
    first, second = np.asarray(first), np.asarray(second)
    prompt_seen = _row_counts(prompt, V_LM) > 0

    @torch.inference_mode()
    def softmax_after(ids, gen):
        row = lm(input_ids=torch.as_tensor([ids]).cuda()).logits[0, -1]
        row = _penalize_row(row, _row_counts(gen, V_LM), prompt_seen, 1.3, 0.0, 0.0)
        return torch.softmax(row.double(), -1).cpu().numpy()

    def close(counts, p, what):
        n = counts.sum()
        tol = 5.0 * np.sqrt(n * p * (1 - p)) + 1.0
        bad = np.abs(counts - n * p) > tol
        assert not bad.any(), (what, np.nonzero(bad)[0][:5].tolist(), counts[bad][:5].tolist(), (n * p)[bad][:5].tolist())

    h1 = np.bincount(first, minlength=V_LM)
    close(h1, softmax_after(prompt, []), "first token")
    for t in np.argsort(-h1)[:3]:
        sel = first == t
        close(np.bincount(second[sel], minlength=V_LM), softmax_after(prompt + [int(t)], [int(t)]),
              f"second token after {t}")


# ---- 5. log-probabilities of the penalized rows -------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["samd", "samd_tree", "sam_only"])
@torch.inference_mode()
def test_logprobs_are_those_of_the_penalized_rows(lm, work, mode):
    from samd_b200 import synth
    prompts, limits, pens = work
    flavour = mode.replace("_tree", "")
    kw = dict(tree=synth.token_recycle_tree()) if mode == "samd_tree" else {}
    dec = _decoders(lm)[flavour](4, **kw)
    got = _serve(dec, prompts, limits, penalties=pens, logprobs=2)
    for i in range(N_REQ):
        tokens, info = got[i]
        prompt, pn = prompts[i], pens[i]
        ids = torch.as_tensor([prompt + tokens]).cuda()
        rows = lm(input_ids=ids).logits[0, len(prompt) - 1:len(prompt) - 1 + len(tokens)]
        seen = _row_counts(prompt, V_LM) > 0
        pen = torch.stack([_penalize_row(rows[k], _row_counts(tokens[:k], V_LM), seen, pn.repetition_penalty,
                                         pn.presence_penalty, pn.frequency_penalty) for k in range(len(tokens))])
        ref = torch.log_softmax(pen.float(), -1).cpu().numpy()
        want = ref[np.arange(len(tokens)), tokens]
        assert np.abs(np.asarray(info["logprobs"]) - want).max() <= 1e-4, (i, np.abs(np.asarray(info["logprobs"]) - want).max())
        assert [top[0][0] for top in info["top_logprobs"]] == tokens, i       # greedy: the best entry is the token
