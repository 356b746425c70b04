"""CPU checks of penalties=: Penalties.problem() refuses bad values, the decoders name the request of a bad or missing
entry when it is pulled, and engine.apply_penalties refuses bad arguments before anything reaches the device."""
from types import SimpleNamespace

import pytest
import torch

INF, NAN = float("inf"), float("nan")


@pytest.mark.parametrize("bad, msg", [
    (dict(repetition_penalty=0.0), "repetition_penalty must be > 0"),
    (dict(repetition_penalty=-1.1), "repetition_penalty must be > 0"),
    (dict(repetition_penalty=NAN), "repetition_penalty must be a finite float"),
    (dict(repetition_penalty=INF), "repetition_penalty must be a finite float"),
    (dict(repetition_penalty=True), "repetition_penalty must be a finite float"),
    (dict(repetition_penalty="1.1"), "repetition_penalty must be a finite float"),
    (dict(presence_penalty=2.5), r"presence_penalty must be in \[-2, 2\]"),
    (dict(presence_penalty=-2.01), r"presence_penalty must be in \[-2, 2\]"),
    (dict(presence_penalty=NAN), "presence_penalty must be a finite float"),
    (dict(presence_penalty=-INF), "presence_penalty must be a finite float"),
    (dict(presence_penalty=False), "presence_penalty must be a finite float"),
    (dict(frequency_penalty=3), r"frequency_penalty must be in \[-2, 2\]"),
    (dict(frequency_penalty=NAN), "frequency_penalty must be a finite float"),
    (dict(frequency_penalty=True), "frequency_penalty must be a finite float"),
    (dict(frequency_penalty=None), "frequency_penalty must be a finite float"),
])
def test_problem_names_each_bad_value(bad, msg):
    import re
    from samd_b200.batched import Penalties
    got = Penalties(**bad).problem()
    assert got is not None and re.match(msg, got), got


def test_good_values_pass():
    from samd_b200.batched import Penalties
    for ok in (Penalties(), Penalties(1.3), Penalties(0.5, -2.0, 2.0), Penalties(repetition_penalty=2, presence_penalty=1),
               Penalties(frequency_penalty=-0.25)):
        assert ok.problem() is None, ok


def _decoder():
    from samd_b200.batched import BatchedSamdDecoder
    dec = BatchedSamdDecoder.__new__(BatchedSamdDecoder)              # no device: only the host-side checks are used
    dec.T, dec.cache, dec.dyn, dec.tree = 8, SimpleNamespace(max_len=512), SimpleNamespace(max_tokens=1024), None
    return dec


def _pull(prompts, penalties):
    dec = _decoder()
    return dec._with_penalties(dec._with_sampling(dec._requests(iter(prompts), 8), None), penalties)


def test_per_request_entries_name_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import Penalties
    pn = Penalties(1.2)
    with pytest.raises(K.SamdError, match="request 2: penalties has 2 values, fewer than the prompts"):
        list(_pull([[3], [4], [5]], [pn, pn]))
    with pytest.raises(K.SamdError, match="request 1: penalties must be a Penalties, got dict"):
        list(_pull([[3], [4]], [pn, dict(repetition_penalty=1.2)]))
    with pytest.raises(K.SamdError, match="request 1: penalties must be a Penalties, got float"):
        list(_pull([[3], [4]], [pn, 1.2]))
    with pytest.raises(K.SamdError, match="request 0: presence_penalty must be in"):
        list(_pull([[3], [4]], Penalties(presence_penalty=4.0)))
    with pytest.raises(K.SamdError, match="penalties must be None, a Penalties or a sequence of them, got float"):
        list(_pull([[3]], 1.2))
    # the requests before a bad one are handed out unchanged
    pulled = []
    with pytest.raises(K.SamdError, match="request 2: repetition_penalty must be > 0"):
        for r in _pull([[3], [4], [5]], [pn, Penalties(), Penalties(0.0)]):
            pulled.append(r)
    assert [(r[0], r[4]) for r in pulled] == [(0, pn), (1, Penalties())]


def test_shared_and_absent_penalties():
    from samd_b200.batched import Penalties
    pn = Penalties(presence_penalty=0.5)
    assert [r[4] for r in _pull([[3], [4], [5]], pn)] == [pn] * 3
    assert [r[4] for r in _pull([[3], [4]], None)] == [None, None]
    assert [r[4] for r in _pull([[3], [4]], (pn, Penalties()))] == [pn, Penalties()]


def _args(B=2, T=4, V=16, S=2):
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32)
    f32 = lambda *s: torch.ones(*s, dtype=torch.float32)
    return dict(logits=torch.zeros(B, T, V), counts=i32(S, V), repetition=f32(S), presence=f32(S), frequency=f32(S),
                tokens=i32(B, T), retrieve=i32(B, 3, T), n_nodes=i32(B), n_paths=i32(B), done=torch.zeros(B, dtype=torch.bool))


@pytest.mark.parametrize("change, msg", [
    (dict(logits=torch.zeros(2, 16)), r"logits must be \[B, T, V\]"),
    (dict(logits=torch.zeros(2, 16, 4).transpose(1, 2)), r"logits must be \[B, T, V\] with unit stride"),
    (dict(logits=torch.zeros(2, 4, 16, dtype=torch.float64)), "unsupported logits dtype"),
    (dict(logits=torch.zeros(2, 300, 16), tokens=torch.zeros(2, 300, dtype=torch.int32), retrieve=None, n_paths=None),
     "at most 256 rows per request"),
    (dict(counts=torch.zeros(2, 15, dtype=torch.int32)), r"counts must be \[S, 16\]"),
    (dict(counts=torch.zeros(2, 16, dtype=torch.int64)), "counts must be a contiguous"),
    (dict(counts=torch.zeros(16, 2, dtype=torch.int32).T), "counts must be a contiguous"),
    (dict(counts=torch.zeros(3, 16, dtype=torch.int32)), "without slots counts needs one row per request"),
    (dict(repetition=torch.ones(2, dtype=torch.float64)), "repetition must be a contiguous"),
    (dict(presence=torch.ones(3)), "presence must be a contiguous"),
    (dict(frequency=torch.ones(2, 1)), "frequency must be a contiguous"),
    (dict(tokens=None), "a path table needs the node tokens"),
    (dict(tokens=torch.zeros(2, 3, dtype=torch.int32)), "tokens must be a contiguous"),
    (dict(tokens=torch.zeros(2, 4, dtype=torch.int64)), "tokens must be a contiguous"),
    (dict(retrieve=torch.zeros(3, 3, 4, dtype=torch.int32)), r"retrieve must be \[2, P, D\]"),
    (dict(retrieve=torch.zeros(3, 4, dtype=torch.int32)), r"retrieve must be \[2, P, D\]"),
    (dict(retrieve=torch.zeros(2, 3, 4, dtype=torch.int64)), "retrieve must be a contiguous"),
    (dict(retrieve=None), "n_paths needs a path table"),
    (dict(n_nodes=torch.zeros(2, 1, dtype=torch.int32)), "n_nodes must be a contiguous"),
    (dict(n_paths=torch.zeros(2, dtype=torch.float32)), "n_paths must be a contiguous"),
    (dict(done=torch.zeros(2, dtype=torch.int32)), "done must be a contiguous"),
    (dict(slots=torch.zeros(2, dtype=torch.int64)), "slots must be a contiguous"),
    (dict(slots=torch.zeros(3, dtype=torch.int32)), "slots must be a contiguous"),
    ({}, "every tensor must be on the logits' GPU"),
])
def test_apply_penalties_argument_checks(change, msg):
    from samd_b200 import _cabi as K, engine as E
    kw = _args()
    kw.update(change)
    with pytest.raises(K.SamdError, match=msg):
        E.apply_penalties(**kw)


def test_symbol_is_exported():
    from samd_b200 import _cabi as K
    assert K.SYMBOLS["samd_apply_penalties"][1][0] is not None
    assert [f for f, _ in K.PenaltyArgs._fields_][:5] == ["logits_dev", "dtype", "batch", "n_nodes", "vocab"]
