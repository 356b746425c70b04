"""samd_verify_sample_requests' processed distribution and its wide-level walk, deterministically, against float64.

Every sampled token comes out of row_dist (csrc/verify_sample.cu): temperature, then top-p, then top-k, then a
normaliser.  The kernel shows that distribution in `sample_p` when every candidate of a level is rejected: it is the
residual, the processed distribution with the rejected tokens zeroed and the rest renormalised.  So each request here is
a draft whose candidate c has zero or tiny processed probability, with a Philox offset chosen on the host so that the
first draw rejects c by a clear margin; then sample_p must equal the float64 processed distribution without c.

Comparison rule (_check_dist), with S(q) the float64 kept set at top-p q and delta = 1e-6:
  - the kernel's kept set S (sample_p > 0) satisfies S(top_p - delta) <= S <= S(top_p + delta) - both answers are
    allowed only where the float64 boundary is itself that thin; a kept token the kernel shows as 0 must be one whose
    float64 probability is below float32's range;
  - every probability matches the float64 softmax over S within rtol 2e-5, atol 1e-12, and the entries sum to 1 within
    1e-5.  The tolerance follows from the arithmetic: float32 expf of arguments up to 87 (the exponent's own rounding
    costs |x| * 2^-24 relative, and probabilities above 1e-12 have |x| < 28), a double normaliser rounded to float, and
    float32 partial sums over 256 threads' chunks (~4e-6 relative for a flat row of 151936 tokens);
  - at least 80 % of the requests of a launch have S(top_p - delta) = S(top_p + delta), so that the rule cannot
    hollow out the comparison."""
import numpy as np
import pytest
import torch

import samd_oracle as O

pytestmark = pytest.mark.gpu

TDT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
TEMPS = (1e-5, 0.05, 0.7, 1.0, 1.5, 20.0)
TOP_PS = (0.0, 5e-9, 1.0, 1e-8, 0.1, 0.5, 0.9, 0.999)
DELTA = 1e-6
RTOL, ATOL = 2e-5, 1e-12
FAR = 1.0e4                     # what the padding and the unread rows hold: a kernel that reads them fails every check


@pytest.fixture(scope="module")
def E():
    from samd_b200 import engine
    return engine


def _cuda(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


class Ref:
    """One row as the kernel reads it, in float64, at one processor: the kept sets at top_p -/+ DELTA and the weights.
    The processor rules are the kernel's: temperature always divides, top-p is on for 1e-8 <= top_p < 1 (the float32
    value is the cut), top-k for top_k > 0."""

    def __init__(self, row, order, temperature, top_p, top_k):
        t = float(np.float32(temperature))
        s = row.astype(np.float64) / t
        self.w = np.exp(s - s.max())
        keep = []
        q = float(np.float32(top_p))
        for qq in (q - DELTA, q + DELTA):
            k = np.ones(row.size, bool)
            if 1e-8 <= top_p < 1.0:
                e = self.w[order]
                remove = np.cumsum(e / e.sum()) <= 1.0 - qq
                remove[-1] = False                                   # the maximum's last member always stays
                k[order[remove]] = False
            if top_k > 0:
                sk = np.where(k, s, -np.inf)
                n = min(top_k, row.size)
                k &= sk >= np.partition(sk, row.size - n)[row.size - n]
            keep.append(k)
        self.lo, self.hi = keep
        self.sure = bool(np.array_equal(self.lo, self.hi))


def _check_dist(got, ref, zeroed, what):
    """The comparison rule of the module docstring; `zeroed`: tokens the residual must give 0."""
    lo, hi = ref.lo.copy(), ref.hi.copy()
    lo[zeroed] = hi[zeroed] = False
    kept = got > 0
    assert not (kept & ~hi).any(), (what, "kept beyond S(top_p + delta)", np.nonzero(kept & ~hi)[0][:8])
    w = np.where(kept, ref.w, 0.0)
    missed = lo & ~kept
    if missed.any():
        assert (ref.w[missed] / ref.w[lo].sum()).max() < 1e-40, (what, "dropped from S(top_p - delta)",
                                                                  np.nonzero(missed)[0][:8])
    want = w / w.sum()
    err = np.abs(got - want) - (ATOL + RTOL * want)
    assert (err <= 0).all(), (what, "values", int(err.argmax()), float(got[err.argmax()]), float(want[err.argmax()]))
    assert abs(got.sum() - 1.0) <= 1e-5, (what, "sum", got.sum())


def _check_next(got, nxt, u, what):
    """The next token's interval of the CDF of sample_p contains u.  The kernel walks the CDF in float32: a running sum
    of at most ceil(V / 256) entries after at most 256 chunk sums, each addition rounded, so the interval may be off by
    (ceil(V / 256) + 256) * 2^-24 of the mass (5.1e-5 at V = 151936; a flat row, whose roundings all go one way,
    reaches it)."""
    cdf = np.cumsum(got)
    tol = (-(-got.size // 256) + 256) * 2.0 ** -24
    assert got[nxt] > 0 and cdf[nxt] - got[nxt] - tol <= u <= cdf[nxt] + tol, (what, nxt, u, cdf[nxt] - got[nxt], cdf[nxt])


def _rejecting_offset(seed, base, p_c):
    """The first offset >= base whose draw rejects a candidate of probability p_c by a clear margin."""
    for off in range(base, base + 64):
        if O.philox_uniform(seed, off) > p_c * (1.0 + 1e-3) + 1e-7:
            return off
    raise AssertionError("no rejecting draw in 64 offsets")


def _run_residuals(E, rows, dtype, procs, V, stride=None, seed=0):
    """One launch: request b is the two-node draft (root, c_b) on rows[b] with processor procs[b].  Picks c_b (a token
    outside S(top_p + delta), else the lightest of S(top_p - delta)) and an offset whose draw rejects it; checks
    sample_p, accept_len, the draws used and the next token.  Returns the share of unambiguous requests."""
    B = len(rows)
    stride = stride or V
    host = np.full((B, 2, stride), FAR, np.float32)
    host[:, 0, :V] = np.stack(rows)
    lg = torch.as_tensor(host).to(TDT[dtype]).cuda()[:, :, :V]
    seen = lg[:, 0].float().cpu().numpy().astype(np.float64)           # what the kernel reads
    rng = np.random.default_rng(seed)
    tokens = np.zeros((B, 2), np.int32)
    seeds = rng.integers(1, 2 ** 62, size=B)
    offs = np.zeros(B, np.int64)
    refs, orders = [], {}
    for b in range(B):
        key = seen[b].tobytes()
        if key not in orders:
            orders[key] = np.argsort(seen[b], kind="stable")
        t, p, k = procs[b]
        ref = Ref(seen[b], orders[key], t, p, k)
        out_hi = np.nonzero(~ref.hi)[0]
        if out_hi.size:
            c, p_c = int(out_hi[rng.integers(out_hi.size)]), 0.0
        else:
            c = int(np.argmin(np.where(ref.lo, ref.w, np.inf)))
            p_c = ref.w[c] / ref.w[ref.lo].sum()
        tokens[b] = (int(rng.integers(V)), c)
        offs[b] = _rejecting_offset(int(seeds[b]), int(rng.integers(0, 2 ** 40)), p_c)
        refs.append(ref)
    off_t = torch.as_tensor(offs.copy()).cuda()
    out = E.Verifier(B, 2).verify_sample(
        lg, _cuda(tokens, torch.int32), None, _cuda([p[0] for p in procs], torch.float32),
        _cuda([p[1] for p in procs], torch.float32), _cuda([p[2] for p in procs], torch.int32),
        torch.as_tensor(seeds).cuda(), off_t, want_sample_p=True)
    torch.cuda.synchronize()
    sp = out["sample_p"].cpu().numpy().astype(np.float64)
    acc, nxt, used = out["accept_len"].cpu().numpy(), out["next_token"].cpu().numpy(), off_t.cpu().numpy() - offs
    for b in range(B):
        what = (dtype, V, stride, b, procs[b])
        assert acc[b] == 1 and used[b] == 2, (what, int(acc[b]), int(used[b]))
        _check_dist(sp[b], refs[b], [tokens[b, 1]], what)
        _check_next(sp[b], int(nxt[b]), O.philox_uniform(int(seeds[b]), int(offs[b]) + 1), what)
    return sum(r.sure for r in refs) / B


# ---------------------------------------------------------------------------------------------------------------------
# (a) the grid: dtypes x vocabularies x row kinds, every processor value and every top-p / top-k pairing in each launch
# ---------------------------------------------------------------------------------------------------------------------
KINDS = ("randn1", "randn4", "grid", "llm", "inf_flood", "equal")
ROWS_PER_KIND = 8


def _kind_rows(kind, V, rng):
    out = []
    for r in range(ROWS_PER_KIND):
        if kind.startswith("randn"):
            row = rng.standard_normal(V) * float(kind[5:])
        elif kind == "grid":
            row = rng.integers(-12, 13, size=V) * 0.5                   # 25 values: ties everywhere
        elif kind == "llm":
            # a flat tail holding about half the mass (1e-5 of it per token at 128k) under a few dominant logits
            row = rng.standard_normal(V) * 0.3
            row[rng.choice(V, 5, replace=False)] = np.log(V) + np.array([-2.0, -1.6, -1.2, -0.8, -0.4]) + rng.random(5)
        elif kind == "inf_flood":
            row = np.full(V, -np.inf)
            n = (1, 7, 40)[r % 3]                                        # fewer finite values than top_k = 50
            row[rng.choice(V, n, replace=False)] = rng.standard_normal(n) * 2.0
        else:
            row = np.full(V, 3.25)
        out.append(row.astype(np.float32))
    return out


def _grid_procs(V, shift):
    top_ks = (0, 1, 2, 8, 50, V, V + 5)
    pairs = [(p, k) for p in TOP_PS for k in top_ks]
    return [(TEMPS[(i + shift) % len(TEMPS)], p, k) for i, (p, k) in enumerate(pairs)]


@pytest.mark.parametrize("dtype", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("V,stride", [(997, None), (997, 1024), (32000, None), (128256, None), (151936, None)])
def test_processed_distribution_grid(E, dtype, V, stride):
    rng = np.random.default_rng(V + len(dtype))
    rows, procs = [], []
    for ki, kind in enumerate(KINDS):
        base = _kind_rows(kind, V, rng)
        ps = _grid_procs(V, ki)
        rows += [base[i % ROWS_PER_KIND] for i in range(len(ps))]
        procs += ps
    sure = _run_residuals(E, rows, dtype, procs, V, stride, seed=V)
    assert sure >= 0.8, sure


# ---------------------------------------------------------------------------------------------------------------------
# (c) constructed tie-group rows with known kept sets
# ---------------------------------------------------------------------------------------------------------------------
VC = 5000                       # chunk = ceil(5000 / 256) = 20 tokens per thread in the partial-cut owner search
HIGHS = {4000: 7.0, 10: 6.5, 2500: 6.0}


def _tie_case(name, temperature):
    """(row, top_p, top_k, expected kept indices).  Background 0, a tie group at 3 (or the maximum's group at 7), the
    top-p budget placed at (members removed + 0.5) member weights above the background's mass, in float64."""
    row = np.zeros(VC)
    t = float(np.float32(temperature))

    def top_p_for(members, cut, group_value):
        w = np.exp((row - row.max()) / t)
        below = w[row < group_value].sum()
        e = np.exp((group_value - row.max()) / t)
        tp = float(np.float32(1.0 - (below + (cut + 0.5) * e) / w.sum()))
        room = (1.0 - tp) * w.sum() - below
        assert cut + 0.4 < room / e < cut + 0.6, (name, room / e)        # unambiguous in float32 top_p as well
        return tp

    def with_highs(group):
        for i, v in HIGHS.items():
            row[i] = v
        row[group] = 3.0

    if name == "cut_in_one_chunk":                                       # members 100..107: thread 5's chunk
        g = list(range(100, 108))
        with_highs(g)
        return row, top_p_for(g, 3, 3.0), 0, sorted(g[3:] + list(HIGHS))
    if name == "cut_across_chunks":                                      # 40 members, 37 apart; member 25 at 893
        g = [5 + 37 * j for j in range(40)]
        with_highs(g)
        return row, top_p_for(g, 25, 3.0), 0, sorted(g[25:] + list(HIGHS))
    if name in ("max_group_1e-8", "max_group_cut_1"):                    # the maximum's tie group, across chunks
        g = [7, 2000, 3001]
        row[g] = 7.0
        row[[50, 60]] = 3.0
        if name == "max_group_1e-8":
            return row, 1e-8, 0, [3001]
        return row, top_p_for(g, 1, 7.0), 0, [2000, 3001]
    if name.startswith("top_k_in_group"):                                # top-k's k-th value inside a group: ties stay
        g = [300, 301, 556, 1000, 4999]
        with_highs(g)
        k = int(name[-1])
        return row, 0.0, k, sorted(list(HIGHS) + (g if k > 3 else []))
    if name.startswith("top_k_after_cut"):
        # top-k after a partial top-p cut, with the k-th survivor in the partly cut group (k = 5, 7) or above it (k = 3).
        # The cut group is always the lowest surviving one, so the kept set does not depend on whether top-k's count
        # excludes its removed members: these cases pin the two filters' composition, not that subtraction.
        g = [50 + 256 * j for j in range(6)]
        with_highs(g)
        k = int(name[-1])
        return row, top_p_for(g, 2, 3.0), k, sorted(list(HIGHS) + (g[2:] if k > 3 else []))
    raise KeyError(name)


TIE_CASES = ("cut_in_one_chunk", "cut_across_chunks", "max_group_1e-8", "max_group_cut_1", "top_k_in_group_3",
             "top_k_in_group_4", "top_k_in_group_5", "top_k_after_cut_3", "top_k_after_cut_5", "top_k_after_cut_7")


@pytest.mark.parametrize("dtype", ["fp32", "bf16", "fp16"])
def test_tie_group_cuts_keep_the_expected_members(E, dtype):
    rows, procs, expect = [], [], []
    for temperature in (1.0, 0.7):
        for name in TIE_CASES:
            row, tp, k, kept = _tie_case(name, temperature)
            got = np.nonzero(O.processed_probs(row, temperature, tp, k) > 0)[0].tolist()
            assert got == kept, (name, temperature, "oracle", got)
            rows.append(row.astype(np.float32))
            procs.append((temperature, tp, k))
            expect.append((name, temperature, kept))
    B = len(rows)
    lg = torch.as_tensor(np.stack([np.stack([r, np.full(VC, FAR, np.float32)]) for r in rows])).to(TDT[dtype]).cuda()
    tokens = np.array([[0, 4990 + b % 8] for b in range(B)], np.int32)      # background: zero probability everywhere
    seeds = np.arange(1, B + 1)
    offs = np.array([_rejecting_offset(int(s), 0, 0.0) for s in seeds], np.int64)
    out = E.Verifier(B, 2).verify_sample(
        lg, _cuda(tokens, torch.int32), None, _cuda([p[0] for p in procs], torch.float32),
        _cuda([p[1] for p in procs], torch.float32), _cuda([p[2] for p in procs], torch.int32),
        torch.as_tensor(seeds).cuda(), torch.as_tensor(offs.copy()).cuda(), want_sample_p=True)
    torch.cuda.synchronize()
    sp = out["sample_p"].cpu().numpy().astype(np.float64)
    for b, (name, temperature, kept) in enumerate(expect):
        assert np.nonzero(sp[b] > 0)[0].tolist() == kept, (dtype, name, temperature, np.nonzero(sp[b] > 0)[0][:12])
        row = rows[b].astype(np.float64)
        ref = Ref(row, np.argsort(row, kind="stable"), *procs[b])
        assert ref.sure
        _check_dist(sp[b], ref, [tokens[b, 1]], (dtype, name, temperature))


# ---------------------------------------------------------------------------------------------------------------------
# (d) levels wider than the kernel's shared list of 64 rejected candidates
# ---------------------------------------------------------------------------------------------------------------------
VD = 32000


def _star(leaves, repeat, rng, top):
    """Leaf tokens of a star tree, none of them in `top`: `leaves` distinct tokens, or with repeat, 120 distinct ones,
    then repeats of those at positions 60..119 (past the 64th), then one more new token."""
    pool = rng.permutation(np.setdiff1d(np.arange(VD), top))
    if not repeat:
        return pool[:leaves]
    return np.concatenate([pool[:120], pool[60 + rng.integers(0, 60, size=leaves - 121)], pool[120:121]])


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("leaves,repeat", [(100, False), (300, False), (300, True)])
def test_wide_levels_remember_every_rejected_candidate(E, dtype, leaves, repeat):
    """Star trees (root + `leaves` leaves, depth 2).  Requests 0-2: the leaves lie outside top-k (probability 0).
    Requests 3-5: no top-k, the leaves have probability ~1e-6 each, offsets chosen so that all are rejected.  Requests
    6-7: the last distinct leaf holds half the mass and the offset is chosen so that the walk accepts it.  Each request
    is compared with O.verify_typical on the same Philox stream."""
    B, T = 8, leaves + 1
    rng = np.random.default_rng(leaves * 2 + repeat)
    logits = (rng.standard_normal((B, T, VD)) * 1.0).astype(np.float32)
    tokens = np.zeros((B, T), np.int32)
    procs = [(0.7, 0.9, 50), (1.0, 0.0, 50), (1.5, 0.999, 20), (1.0, 0.0, 0), (1.5, 0.0, 0), (0.7, 0.0, 0),
             (1.0, 0.0, 0), (1.0, 0.0, 0)]
    for b in range(B):
        top = np.argsort(logits[b, 0])[-200:]
        leaf = _star(leaves, repeat, rng, top)
        tokens[b, 0], tokens[b, 1:] = rng.integers(VD), leaf
        if procs[b][2] == 0:
            logits[b, 0, leaf] = -3.0 - rng.random(leaf.size).astype(np.float32)      # ~1e-6 of the mass each
        if b >= 6:
            distinct = list(dict.fromkeys(leaf.tolist()))
            logits[b, 0, distinct[-1]] = np.log(np.exp(logits[b, 0].astype(np.float64)).sum())
    retrieve = np.stack([np.arange(T) * 0, np.arange(T)], axis=1)[1:].astype(np.int32)          # [leaves, 2]: (0, leaf)
    lg = torch.as_tensor(logits).to(TDT[dtype]).cuda()
    seen = lg.float().cpu().numpy()
    seeds = rng.integers(1, 2 ** 62, size=B)
    offs = np.zeros(B, np.int64)
    wants = []
    for b in range(B):
        t, p, k = procs[b]
        base = int(rng.integers(0, 2 ** 40))
        for off in range(base, base + 200 * 4096, 4096):              # disjoint streams
            draws = [0]

            def draw():
                draws[0] += 1
                return O.philox_uniform(int(seeds[b]), off + draws[0] - 1)

            want = O.verify_typical(seen[b], tokens[b], retrieve.astype(np.int64), t, p, k, draw)
            if min(want["margins"][:-1]) > 1e-3 and want["accept_len"] == (2 if b >= 6 else 1):
                break
        else:
            raise AssertionError(("no offset gives the intended walk", b))
        offs[b] = off
        want["draws"] = draws[0]
        wants.append(want)
    off_t = torch.as_tensor(offs.copy()).cuda()
    out = E.Verifier(B, T).verify_sample(
        lg, _cuda(tokens, torch.int32), _cuda(retrieve, torch.int32), _cuda([p[0] for p in procs], torch.float32),
        _cuda([p[1] for p in procs], torch.float32), _cuda([p[2] for p in procs], torch.int32),
        torch.as_tensor(seeds).cuda(), off_t, want_sample_p=True)
    torch.cuda.synchronize()
    sp = out["sample_p"].cpu().numpy().astype(np.float64)
    used = off_t.cpu().numpy() - offs
    for b, want in enumerate(wants):
        what = (dtype, leaves, repeat, b)
        assert out["best"][b].item() == want["best"] and out["accept_len"][b].item() == want["accept_len"], what
        n = want["accept_len"]
        assert out["tokens"][b, :n].tolist() == want["tokens"] and out["indices"][b, :n].tolist() == want["indices"], what
        assert int(used[b]) == want["draws"], (what, "draws", int(used[b]), want["draws"])
        if n == 1:                                                      # the residual of the root's processed row
            row = seen[b, 0].astype(np.float64)
            ref = Ref(row, np.argsort(row, kind="stable"), *procs[b])
            rejected = np.unique(tokens[b, 1:])
        else:                                                           # the plain softmax of the accepted leaf's row
            row = seen[b, want["indices"][1]].astype(np.float64)
            ref = Ref(row, None, 1.0, 0.0, 0)
            rejected = []
        _check_dist(sp[b], ref, rejected, what)
        _check_next(sp[b], out["next_token"][b].item(), O.philox_uniform(int(seeds[b]), int(offs[b]) + want["draws"] - 1),
                    what)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_wide_table_computes_what_a_narrow_one_does(E, dtype):
    """A path table with more than 64 paths runs the kernel's wide instantiation.  With per-request n_paths of at most
    30, every output must be bit for bit that of the same paths in a 30-path table (the common instantiation)."""
    from samd_b200 import synth
    tree = synth.token_recycle_tree()
    ri = synth.tree_retrieve_indices(tree).astype(np.int32)             # [30, 6]
    B, T, V = 64, len(tree), 32000
    rng = np.random.default_rng(17)
    logits = (rng.standard_normal((B, T, V)) * 2.0).astype(np.float32)
    tokens = rng.integers(0, V, size=(B, T)).astype(np.int32)
    for c, ch in enumerate(tree):
        for k in ch:
            logits[np.arange(B), c, tokens[:, k]] += 8.0 + rng.random(B).astype(np.float32) * 6.0
    lg = torch.as_tensor(logits).to(TDT[dtype]).cuda()
    n_paths = rng.integers(1, ri.shape[0] + 1, size=B).astype(np.int32)
    narrow = np.repeat(ri[None], B, axis=0)
    wide = np.full((B, 80, ri.shape[1]), -1, np.int32)
    wide[:, :ri.shape[0]] = narrow
    procs = [(TEMPS[b % 6], TOP_PS[b % 8], (0, 1, 8, 50)[b % 4]) for b in range(B)]
    outs = []
    for table in (narrow, wide):
        offs = torch.arange(B, dtype=torch.int64).cuda() * 1000
        out = E.Verifier(B, T).verify_sample(
            lg, _cuda(tokens, torch.int32), _cuda(table, torch.int32), _cuda([p[0] for p in procs], torch.float32),
            _cuda([p[1] for p in procs], torch.float32), _cuda([p[2] for p in procs], torch.int32),
            torch.arange(1, B + 1).cuda(), offs, n_paths=_cuda(n_paths, torch.int32), want_sample_p=True)
        torch.cuda.synchronize()
        outs.append({k: v.cpu() for k, v in out.items()} | {"offsets": offs.cpu()})
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), k
    assert (outs[0]["accept_len"] > 1).sum() >= B // 4                  # the walks accept, the levels reject


# ---------------------------------------------------------------------------------------------------------------------
# (e) the greedy branch of the same kernel at V = 151936 and 256 rows
# ---------------------------------------------------------------------------------------------------------------------
VG, TG = 151936, 256


def _special_rows(g):
    """Rows whose argmax needs torch.argmax's rule: NaN is the maximum (the first NaN), +0 == -0, the lowest index among
    equal maxima, here placed so that the lowest is owned by a later thread or warp of the strided partition."""
    nan, inf = float("nan"), float("inf")
    g[1, [5000, 777]] = nan
    g[1, 3] = inf
    g[2, [100000, 773]] = inf
    g[3] = -inf
    g[4] = -1.0
    g[4, 1234], g[4, 1000] = 0.0, -0.0
    g[5] = -1.0
    g[5, 1234], g[5, 1000] = -0.0, 0.0
    g[6, [255, 256, 513, VG - 1]] = 7.5                    # thread 255 (warp 7) holds the first, thread 0 the next
    g[7, [511, 300, 40000]] = 7.5                          # thread 44 holds the first
    g[8, VG - 1] = nan
    g[9] = -inf
    g[9, 77777] = -1e30
    g[10] = -g[10].abs() - 1.0                             # all negative


def _greedy_rows(B, dtype, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    lg = torch.randn(B, TG, VG, generator=gen, device="cuda") * 2.0
    for b in range(B):
        _special_rows(lg[b, 10 * b:])                       # the special rows at different node rows per request
    lg = lg.to(TDT[dtype])
    am = torch.argmax(lg.float().cpu(), dim=-1).numpy()
    return lg, am


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_greedy_chain_checks_every_row_argmax(E, dtype):
    """Identity paths whose token j + 1 is the reference argmax of row j: the walk accepts everything only if every
    row's argmax is right.  Request 3 breaks its chain at node 100; requests 2-3 have fewer rows than the table."""
    B = 4
    lg, am = _greedy_rows(B, dtype, 5)
    n_nodes = np.array([TG, TG, 200, 129], np.int32)
    tokens = np.zeros((B, TG), np.int32)
    tokens[:, 1:] = am[:, :-1]
    tokens[3, 100] = (am[3, 99] + 1) % VG
    offs = torch.zeros(B, dtype=torch.int64).cuda()
    out = E.Verifier(B, TG).verify_sample(lg, _cuda(tokens, torch.int32), None, 1.0, 0.0, 0,
                                          torch.arange(1, B + 1).cuda(), offs, greedy=torch.ones(B, dtype=torch.bool).cuda(),
                                          n_nodes=_cuda(n_nodes, torch.int32))
    torch.cuda.synchronize()
    assert (offs == 0).all()
    for b in range(B):
        T = int(n_nodes[b])
        want = O.verify_greedy(am[b, :T], tokens[b, :T], np.arange(T, dtype=np.int64)[None])
        assert want["accept_len"] == (100 if b == 3 else T)
        assert out["accept_len"][b].item() == want["accept_len"] and out["next_token"][b].item() == want["next_token"], b
        n = want["accept_len"]
        assert out["tokens"][b, :n].tolist() == want["tokens"].tolist() and (out["tokens"][b, n:] == -1).all(), b


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_greedy_tree_walk_matches_oracle(E, dtype):
    """Random trees of up to 256 nodes (per-request n_nodes and n_paths, -1 padded paths), children that copy their
    parent row's argmax 80 % of the time."""
    B = 4
    lg, am = _greedy_rows(B, dtype, 9)
    rng = np.random.default_rng(3)
    n_nodes = np.array([TG, TG, 200, 97], np.int32)
    parent = np.array([-1] + [int(rng.integers(max(0, c - 6), c)) for c in range(1, TG)])
    tokens = rng.integers(0, VG, size=(B, TG)).astype(np.int32)
    paths = []
    for b in range(B):
        T = int(n_nodes[b])
        for c in range(1, T):
            if rng.random() < 0.8:
                tokens[b, c] = am[b, parent[c]]
        leaves = sorted(set(range(T)) - set(parent[1:T].tolist()))
        ps = []
        for leaf in leaves:
            p, n = [], leaf
            while n >= 0:
                p.append(n)
                n = parent[n]
            ps.append(p[::-1])
        paths.append(ps)
    P, D = max(len(p) for p in paths), max(len(q) for p in paths for q in p)
    retrieve = np.full((B, P, D), -1, np.int32)
    for b, ps in enumerate(paths):
        for i, q in enumerate(ps):
            retrieve[b, i, :len(q)] = q
    n_paths = np.array([len(p) for p in paths], np.int32)
    offs = torch.zeros(B, dtype=torch.int64).cuda()
    out = E.Verifier(B, TG).verify_sample(lg, _cuda(tokens, torch.int32), _cuda(retrieve, torch.int32), 1.0, 0.0, 0,
                                          torch.arange(1, B + 1).cuda(), offs, n_paths=_cuda(n_paths, torch.int32),
                                          greedy=torch.ones(B, dtype=torch.bool).cuda(), n_nodes=_cuda(n_nodes, torch.int32))
    torch.cuda.synchronize()
    assert (offs == 0).all()
    deep = 0
    for b in range(B):
        T = int(n_nodes[b])
        want = O.verify_greedy(am[b, :T], tokens[b, :T], retrieve[b, :n_paths[b]].astype(np.int64))
        assert out["best"][b].item() == want["best"] and out["accept_len"][b].item() == want["accept_len"], b
        assert out["next_token"][b].item() == want["next_token"], b
        n = want["accept_len"]
        assert out["tokens"][b, :n].tolist() == want["tokens"].tolist(), b
        assert out["indices"][b, :n].tolist() == want["indices"].tolist() and (out["indices"][b, n:] == -1).all(), b
        deep += n >= 4
    assert deep >= 2                                        # the walks go several levels deep
