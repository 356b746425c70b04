"""CPU checks of controls=: LogitControls.problem() refuses bad values, serve() and generate() name the request of a bad or
missing entry (or a min_tokens above its max_new_tokens) when it is pulled, and engine.apply_logit_controls refuses bad
arguments before anything reaches the device."""
import math
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

V = 100
INF = math.inf


@pytest.mark.parametrize("kw, msg", [
    (dict(logit_bias={V: 1.0}), r"logit_bias: token ids must be ints in \[0, 100\), got 100"),
    (dict(logit_bias={-1: 1.0}), r"logit_bias: token ids must be ints in \[0, 100\), got -1"),
    (dict(logit_bias={True: 1.0}), r"logit_bias: token ids must be ints in \[0, 100\), got True"),
    (dict(logit_bias=[(2.0, 1.0)]), r"logit_bias: token ids must be ints in \[0, 100\), got 2.0"),
    (dict(logit_bias=[(3, 1.0), (3, 2.0)]), "logit_bias: token id 3 appears more than once"),
    (dict(logit_bias={3: 100.5}), r"logit_bias: the bias of token 3 must be a float in \[-100, 100\] or -inf, got 100.5"),
    (dict(logit_bias={3: -101}), r"the bias of token 3 must be a float in \[-100, 100\] or -inf, got -101"),
    (dict(logit_bias={3: INF}), r"the bias of token 3 must be a float in \[-100, 100\] or -inf, got inf"),
    (dict(logit_bias={3: float("nan")}), r"the bias of token 3 must be a float in \[-100, 100\] or -inf, got nan"),
    (dict(logit_bias={3: True}), r"the bias of token 3 must be a float in \[-100, 100\] or -inf, got True"),
    (dict(logit_bias={3: "1"}), r"the bias of token 3 must be a float in \[-100, 100\] or -inf, got '1'"),
    (dict(logit_bias=[(3, 1.0, 2.0)]), r"logit_bias entry 0 must be a \(token_id, bias\) pair"),
    (dict(logit_bias=[3]), r"logit_bias entry 0 must be a \(token_id, bias\) pair, got 3"),
    (dict(logit_bias="3"), r"logit_bias must be a mapping or a sequence of \(token_id, bias\) pairs, got str"),
    (dict(logit_bias=None), r"logit_bias must be a mapping or a sequence of \(token_id, bias\) pairs, got NoneType"),
    (dict(logit_bias=[(t, 1.0) for t in range(257)]), None),          # (V = 300 below)
    (dict(bad_words=[[]]), "bad word 0 must have 1 to 16 token ids, got 0"),
    (dict(bad_words=[[1], list(range(17))]), "bad word 1 must have 1 to 16 token ids, got 17"),
    (dict(bad_words=[[1]] * 17), "at most 16 bad words, got 17"),
    (dict(bad_words=[[1, V]]), r"bad word 0: token ids must be ints in \[0, 100\), got 100"),
    (dict(bad_words=[[False]]), r"bad word 0: token ids must be ints in \[0, 100\), got False"),
    (dict(bad_words=[5]), "bad word 0 must be a list or tuple of token ids, got int"),
    (dict(bad_words="ab"), "bad_words must be a list or tuple of token id sequences, got str"),
    (dict(min_tokens=-1), "min_tokens must be an int >= 0, got -1"),
    (dict(min_tokens=1.0), "min_tokens must be an int >= 0, got 1.0"),
    (dict(min_tokens=True), "min_tokens must be an int >= 0, got True"),
])
def test_problem_names_each_bad_value(kw, msg):
    from samd_b200.batched import LogitControls
    if msg is None:                                                   # more than 256 distinct ids
        got = LogitControls(**kw).problem(300)
        assert got == "logit_bias: at most 256 token ids, got 257", got
        return
    got = LogitControls(**kw).problem(V)
    assert got is not None and re.search(msg, got), got


def test_good_values_pass():
    from samd_b200.batched import LogitControls
    for ok in (LogitControls(), LogitControls(logit_bias={0: -100, V - 1: 100.0, 5: -INF}),
               LogitControls(logit_bias=[(1, 0.5), (np.int64(2), np.float32(-3.5))]),
               LogitControls(bad_words=[[0]] + [[V - 1] * 16] * 15), LogitControls(min_tokens=8),
               LogitControls(min_tokens=np.int64(3)), LogitControls({1: 2.0}, ((3, 4),), 2)):
        assert ok.problem(V) is None, ok
    assert LogitControls(logit_bias=[(t, 1.0) for t in range(256)]).problem(300) is None
    assert LogitControls(logit_bias={4: 1.0, 2: -INF}).bias_items() == [(4, 1.0), (2, -INF)]
    assert LogitControls(logit_bias=((4, 1.0),)).bias_items() == [(4, 1.0)]


def test_stop_sequence_messages_are_unchanged():
    from samd_b200.batched import StopSequences
    assert StopSequences([[1]] * 17).problem(V) == "at most 16 sequences, got 17"
    assert StopSequences("x").problem(V) == "sequences must be a list or tuple of token id sequences, got str"
    assert StopSequences([[V]]).problem(V) == "sequence 0: token ids must be ints in [0, 100), got 100"


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


def _pull(prompts, controls, limits=8):
    dec = _decoder()
    reqs = dec._with_stops(dec._with_penalties(dec._with_sampling(dec._requests(iter(prompts), limits), None), None),
                           None, V)
    return dec._with_controls(reqs, controls, V)


def test_per_request_entries_name_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import LogitControls
    lc = LogitControls(logit_bias={1: 2.0})
    with pytest.raises(K.SamdError, match="request 2: controls has 2 values, fewer than the prompts"):
        list(_pull([[3], [4], [5]], [lc, lc]))
    with pytest.raises(K.SamdError, match="request 1: controls must be a LogitControls, got dict"):
        list(_pull([[3], [4]], [lc, {1: 2.0}]))
    with pytest.raises(K.SamdError, match="request 1: controls must be a LogitControls, got NoneType"):
        list(_pull([[3], [4]], [lc, None]))
    with pytest.raises(K.SamdError, match="request 0: min_tokens must be an int >= 0"):
        list(_pull([[3], [4]], LogitControls(min_tokens=-2)))
    with pytest.raises(K.SamdError, match="controls must be None, a LogitControls or a sequence of them, got int"):
        list(_pull([[3]], 7))
    pulled = []
    with pytest.raises(K.SamdError, match=r"request 2: logit_bias: token ids must be ints in \[0, 100\)"):
        for r in _pull([[3], [4], [5]], [lc, LogitControls(), LogitControls(logit_bias={V: 0.0})]):
            pulled.append(r)
    assert [(r[0], r[6]) for r in pulled] == [(0, lc), (1, LogitControls())]


def test_min_tokens_above_the_limit_names_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import LogitControls
    assert [r[6].min_tokens for r in _pull([[3], [4]], LogitControls(min_tokens=8))] == [8, 8]
    with pytest.raises(K.SamdError, match="request 1: min_tokens 9 exceeds max_new_tokens 4"):
        list(_pull([[3], [4]], LogitControls(min_tokens=9), limits=[16, 4]))
    with pytest.raises(K.SamdError, match="request 0: min_tokens 9 exceeds max_new_tokens 8"):
        list(_pull([[3], [4]], LogitControls(min_tokens=9)))


def test_shared_and_absent_controls():
    from samd_b200.batched import LogitControls
    lc = LogitControls(bad_words=[[1, 2]], min_tokens=2)
    assert [r[6] for r in _pull([[3], [4], [5]], lc)] == [lc] * 3
    assert [r[6] for r in _pull([[3], [4]], None)] == [None, None]
    assert [r[6] for r in _pull([[3], [4]], (lc, LogitControls()))] == [lc, LogitControls()]
    assert all(len(r) == 7 for r in _pull([[3]], None))


def test_serve_and_generate_name_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import LogitControls
    ok, bad = LogitControls(logit_bias={1: 1.0}), LogitControls(bad_words=[[1], list(range(17))])
    with pytest.raises(K.SamdError, match="request 1: bad word 1 must have 1 to 16 token ids, got 17"):
        list(_decoder().serve([[3], [4], [5]], 8, controls=[ok, bad, ok]))
    with pytest.raises(K.SamdError, match="request 2: controls has 2 values, fewer than the prompts"):
        list(_decoder().serve([[3], [4], [5]], 8, controls=[ok, ok]))
    with pytest.raises(K.SamdError, match="request 1: min_tokens 6 exceeds max_new_tokens 5"):
        list(_decoder().serve([[3], [4], [5]], [8, 5, 8], controls=LogitControls(min_tokens=6)))
    with pytest.raises(K.SamdError, match="request 0: controls must be a LogitControls, got tuple"):
        _decoder().generate([[3], [4], [5]], 8, controls=[((1, 2.0),), ok, ok])
    with pytest.raises(K.SamdError, match=r"request 2: logit_bias: the bias of token 1 must be a float"):
        _decoder().generate([[3], [4], [5]], 8, controls=[ok, ok, LogitControls(logit_bias={1: float("nan")})])
    with pytest.raises(K.SamdError, match="request 0: min_tokens 9 exceeds max_new_tokens 8"):
        _decoder().generate([[3], [4], [5]], 8, controls=LogitControls(min_tokens=9))


def _args(B=2, T=4, V=50, S=2):
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32)
    return dict(logits=torch.zeros(B, T, V), bias_ids=i32(S, 256), bias=torch.zeros(S, 256), bias_n=i32(S),
                bad_tokens=i32(S, 16, 16), bad_len=i32(S, 16), min_tokens=i32(S), tokens=i32(B, T), n_nodes=i32(B),
                done=torch.zeros(B, dtype=torch.bool), hist=i32(S, 8), hist_len=i32(S), stop_tokens=i32(S, 16, 16),
                stop_len=i32(S, 16), eos=3)


@pytest.mark.parametrize("change, msg", [
    (dict(logits=torch.zeros(2, 4)), r"logits must be \[B, T, V\] with unit stride over V"),
    (dict(logits=torch.zeros(2, 50, 4).transpose(1, 2)), r"logits must be \[B, T, V\] with unit stride over V"),
    (dict(logits=torch.zeros(2, 4, 50, dtype=torch.float64)), "unsupported logits dtype"),
    (dict(logits=torch.zeros(2, 257, 50), tokens=None, n_nodes=None), "at most 256 rows per request, got 257"),
    (dict(min_tokens=torch.zeros(2, 1, dtype=torch.int32)), r"min_tokens must be \[S\] with S >= 1"),
    (dict(min_tokens=torch.zeros(3, dtype=torch.int32)), r"without slots the tables need one row per request \(2\)"),
    (dict(retrieve=torch.zeros(2, 3, 4, dtype=torch.int32), tokens=None), "a path table needs the node tokens"),
    (dict(retrieve=torch.zeros(3, 3, 4, dtype=torch.int32)), r"retrieve must be \[2, P, D\]"),
    (dict(retrieve=torch.zeros(2, 0, 4, dtype=torch.int32)), r"retrieve must be \[2, P, D\]"),
    (dict(n_paths=torch.zeros(2, dtype=torch.int32)), "n_paths needs a path table"),
    (dict(hist=None), r"hist_len needs hist \[2, H\] with H >= 1"),
    (dict(hist=torch.zeros(2, 0, dtype=torch.int32)), r"hist_len needs hist \[2, H\] with H >= 1"),
    (dict(stop_len=None), "stop_tokens and stop_len go together"),
    (dict(eos=50), r"eos must be None or a token id in \[0, 50\), got 50"),
    (dict(eos=True), r"eos must be None or a token id in \[0, 50\), got True"),
    (dict(bias_ids=torch.zeros(2, 255, dtype=torch.int32)), "bias_ids must be a contiguous"),
    (dict(bias_ids=torch.zeros(2, 256, dtype=torch.int64)), "bias_ids must be a contiguous"),
    (dict(bias=torch.zeros(2, 256, dtype=torch.float16)), "bias must be a contiguous"),
    (dict(bias=torch.zeros(256, 2).T), "bias must be a contiguous"),
    (dict(bias_n=torch.zeros(2, 1, dtype=torch.int32)), "bias_n must be a contiguous"),
    (dict(bad_tokens=torch.zeros(2, 16, 17, dtype=torch.int32)), "bad_tokens must be a contiguous"),
    (dict(bad_len=torch.zeros(2, 16, dtype=torch.uint8)), "bad_len must be a contiguous"),
    (dict(min_tokens=torch.zeros(2, dtype=torch.int64)), "min_tokens must be a contiguous"),
    (dict(tokens=torch.zeros(2, 5, dtype=torch.int32)), "tokens must be a contiguous"),
    (dict(n_nodes=torch.zeros(2, dtype=torch.int64)), "n_nodes must be a contiguous"),
    (dict(done=torch.zeros(2, dtype=torch.int32)), "done must be a contiguous"),
    (dict(slots=torch.zeros(2, dtype=torch.int64)), "slots must be a contiguous"),
    (dict(hist=torch.zeros(2, 8, dtype=torch.int64)), "hist must be a contiguous"),
    (dict(hist_len=torch.zeros(2, dtype=torch.int64)), "hist_len must be a contiguous"),
    (dict(stop_tokens=torch.zeros(2, 17, 16, dtype=torch.int32)), "stop_tokens must be a contiguous"),
    (dict(stop_len=torch.zeros(2, 16, dtype=torch.int64)), "stop_len must be a contiguous"),
    ({}, "every tensor must be on the logits' GPU"),
])
def test_apply_logit_controls_argument_checks(change, msg):
    from samd_b200 import _cabi as K, engine as E
    kw = _args()
    kw.update(change)
    with pytest.raises(K.SamdError, match=msg):
        E.apply_logit_controls(**kw)


def test_symbol_is_exported():
    from samd_b200 import _cabi as K
    assert K.SYMBOLS["samd_apply_logit_controls"][1][0] is not None
    assert (K.BIAS_MAX, K.BAD_MAX_SEQS, K.BAD_MAX_LEN) == (256, 16, 16)
    assert [f for f, _ in K.LogitControlArgs._fields_][:3] == ["logits_dev", "dtype", "batch"]
    assert K.LogitControlArgs._fields_[-1][0] == "eos_token"
