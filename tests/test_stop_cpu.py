"""CPU checks of stop=: StopSequences.problem() refuses bad sequences, serve() and generate() name the request of a bad or
missing entry when it is pulled, and engine.match_stops refuses bad arguments before anything reaches the device."""
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

V = 100


@pytest.mark.parametrize("seqs, msg", [
    ([[]], "sequence 0 must have 1 to 16 token ids, got 0"),
    (((1, 2), ()), "sequence 1 must have 1 to 16 token ids, got 0"),
    ([list(range(17))], "sequence 0 must have 1 to 16 token ids, got 17"),
    ([[1]] * 17, "at most 16 sequences, got 17"),
    ([[1, V]], r"sequence 0: token ids must be ints in \[0, 100\), got 100"),
    ([[3], [-1]], r"sequence 1: token ids must be ints in \[0, 100\), got -1"),
    ([[True]], r"sequence 0: token ids must be ints in \[0, 100\), got True"),
    ([[1, 2.0]], r"sequence 0: token ids must be ints in \[0, 100\), got 2.0"),
    ([["7"]], r"sequence 0: token ids must be ints in \[0, 100\), got '7'"),
    ([[None]], r"sequence 0: token ids must be ints in \[0, 100\), got None"),
    ([5, 6], "sequence 0 must be a list or tuple of token ids, got int"),
    (["</s>"], "sequence 0 must be a list or tuple of token ids, got str"),
    ("stop", "sequences must be a list or tuple of token id sequences, got str"),
    (None, "sequences must be a list or tuple of token id sequences, got NoneType"),
])
def test_problem_names_each_bad_value(seqs, msg):
    from samd_b200.batched import StopSequences
    got = StopSequences(seqs).problem(V)
    assert got is not None and re.match(msg, got), got


def test_good_values_pass():
    from samd_b200.batched import StopSequences
    for ok in (StopSequences(), StopSequences(()), StopSequences([[0]]), StopSequences(((V - 1,) * 16,) * 16),
               StopSequences([[1, 2], [1, 2]]), StopSequences([np.array([3, 4]).tolist(), (np.int64(5),)])):
        assert ok.problem(V) is None, ok


def _decoder():
    from samd_b200.batched import BatchedSamdDecoder
    dec = BatchedSamdDecoder.__new__(BatchedSamdDecoder)              # no device: only the host-side checks are used
    dec.T, dec.B, dec.cache, dec.dyn, dec.tree = 8, 3, SimpleNamespace(max_len=512), SimpleNamespace(max_tokens=1024), None
    dec.lm = SimpleNamespace(config=SimpleNamespace(vocab_size=V))

    def drain(requests, *args, **kw):                                 # the decode loop pulls every request
        for _ in requests:
            pass
        return
        yield
    dec._run = drain
    return dec


def _pull(prompts, stop):
    dec = _decoder()
    return dec._with_stops(dec._with_penalties(dec._with_sampling(dec._requests(iter(prompts), 8), None), None), stop, V)


def test_per_request_entries_name_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import StopSequences
    ss = StopSequences([[1, 2]])
    with pytest.raises(K.SamdError, match="request 2: stop has 2 values, fewer than the prompts"):
        list(_pull([[3], [4], [5]], [ss, ss]))
    with pytest.raises(K.SamdError, match="request 1: stop must be a StopSequences, got list"):
        list(_pull([[3], [4]], [ss, [[1, 2]]]))
    with pytest.raises(K.SamdError, match="request 0: sequence 0 must have 1 to 16 token ids"):
        list(_pull([[3], [4]], StopSequences([[]])))
    with pytest.raises(K.SamdError, match="stop must be None, a StopSequences or a sequence of them, got int"):
        list(_pull([[3]], 7))
    pulled = []
    with pytest.raises(K.SamdError, match=r"request 2: sequence 0: token ids must be ints in \[0, 100\)"):
        for r in _pull([[3], [4], [5]], [ss, StopSequences(), StopSequences([[V]])]):
            pulled.append(r)
    assert [(r[0], r[5]) for r in pulled] == [(0, ss), (1, StopSequences())]


def test_shared_and_absent_stops():
    from samd_b200.batched import StopSequences
    ss = StopSequences([[9], [1, 2, 3]])
    assert [r[5] for r in _pull([[3], [4], [5]], ss)] == [ss] * 3
    assert [r[5] for r in _pull([[3], [4]], None)] == [None, None]
    assert [r[5] for r in _pull([[3], [4]], (ss, StopSequences()))] == [ss, StopSequences()]


def test_serve_and_generate_name_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import StopSequences
    ok, bad = StopSequences([[1]]), StopSequences([[1], list(range(17))])
    with pytest.raises(K.SamdError, match="request 1: sequence 1 must have 1 to 16 token ids, got 17"):
        list(_decoder().serve([[3], [4], [5]], 8, stop=[ok, bad, ok]))
    with pytest.raises(K.SamdError, match="request 2: stop has 2 values, fewer than the prompts"):
        list(_decoder().serve([[3], [4], [5]], 8, stop=[ok, ok]))
    with pytest.raises(K.SamdError, match="request 0: stop must be a StopSequences, got tuple"):
        _decoder().generate([[3], [4], [5]], 8, stop=[((1, 2),), ok, ok])
    with pytest.raises(K.SamdError, match=r"request 2: sequence 0: token ids must be ints in \[0, 100\), got 100"):
        _decoder().generate([[3], [4], [5]], 8, stop=[ok, ok, StopSequences([[V]])])


def _args(B=2, W=4, H=8):
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32)
    return dict(tokens=i32(B, W), count=i32(B), hist=i32(B, H), hist_len=i32(B), stop_tokens=i32(B, 16, 16),
                stop_len=i32(B, 16), done=torch.zeros(B, dtype=torch.bool), out_count=i32(B), out_hit=i32(B))


@pytest.mark.parametrize("change, msg", [
    (dict(tokens=torch.zeros(2, dtype=torch.int32)), r"tokens must be \[B, W\] with 1 <= W <= 256"),
    (dict(tokens=torch.zeros(2, 257, dtype=torch.int32)), r"tokens must be \[B, W\] with 1 <= W <= 256"),
    (dict(tokens=torch.zeros(2, 0, dtype=torch.int32)), r"tokens must be \[B, W\] with 1 <= W <= 256"),
    (dict(tokens=torch.zeros(2, 4, dtype=torch.int64)), "tokens must be a contiguous"),
    (dict(tokens=torch.zeros(4, 2, dtype=torch.int32).T), "tokens must be a contiguous"),
    (dict(count=torch.zeros(3, dtype=torch.int32)), "count must be a contiguous"),
    (dict(count=torch.zeros(2, dtype=torch.int64)), "count must be a contiguous"),
    (dict(hist=torch.zeros(3, 8, dtype=torch.int32)), r"hist must be \[2, H\] with H >= 1"),
    (dict(hist=torch.zeros(2, 0, dtype=torch.int32)), r"hist must be \[2, H\] with H >= 1"),
    (dict(hist=torch.zeros(2, 8, dtype=torch.int16)), "hist must be a contiguous"),
    (dict(hist=torch.zeros(8, 2, dtype=torch.int32).T), "hist must be a contiguous"),
    (dict(hist_len=torch.zeros(2, 1, dtype=torch.int32)), "hist_len must be a contiguous"),
    (dict(stop_tokens=torch.zeros(2, 17, 16, dtype=torch.int32)), "stop_tokens must be a contiguous"),
    (dict(stop_tokens=torch.zeros(2, 16, 17, dtype=torch.int32)), "stop_tokens must be a contiguous"),
    (dict(stop_tokens=torch.zeros(2, 16, 16, dtype=torch.int64)), "stop_tokens must be a contiguous"),
    (dict(stop_len=torch.zeros(2, 17, dtype=torch.int32)), "stop_len must be a contiguous"),
    (dict(stop_len=torch.zeros(2, 16, dtype=torch.uint8)), "stop_len must be a contiguous"),
    (dict(done=torch.zeros(2, dtype=torch.int32)), "done must be a contiguous"),
    (dict(out_count=torch.zeros(3, dtype=torch.int32)), "out_count must be a contiguous"),
    (dict(out_hit=torch.zeros(2, dtype=torch.int64)), "out_hit must be a contiguous"),
    ({}, "every tensor must be on the tokens' GPU"),
])
def test_match_stops_argument_checks(change, msg):
    from samd_b200 import _cabi as K, engine as E
    kw = _args()
    kw.update(change)
    with pytest.raises(K.SamdError, match=msg):
        E.match_stops(**kw)


def test_symbol_is_exported():
    from samd_b200 import _cabi as K
    assert K.SYMBOLS["samd_stop_match"][1][0] is not None
    assert K.STOP_MAX_SEQS == K.STOP_MAX_LEN == 16
    assert [f for f, _ in K.StopArgs._fields_][:4] == ["batch", "width", "tokens_dev", "count_dev"]
