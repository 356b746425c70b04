"""CPU checks of logprobs=: the decoders refuse a value that is not None or an int in [0, 8] in generate() and serve(),
and Verifier.token_logprobs refuses bad arguments before anything reaches the device."""
import pytest
import torch

BAD = [True, False, -1, 9, 2.0, "3", [1]]


def _decoders():
    from samd_b200.batched import BatchedSamdDecoder, BatchedSamOnlyDecoder
    return [cls.__new__(cls) for cls in (BatchedSamdDecoder, BatchedSamOnlyDecoder)]   # no device: checks only


@pytest.mark.parametrize("bad", BAD)
def test_decoders_refuse_bad_logprobs(bad):
    from samd_b200 import _cabi as K
    for dec in _decoders():
        with pytest.raises(K.SamdError, match=r"logprobs must be None or an int in \[0, 8\]"):
            dec.generate([[3, 4]], 8, logprobs=bad)
        with pytest.raises(K.SamdError, match=r"logprobs must be None or an int in \[0, 8\]"):
            next(dec.serve([[3, 4]], 8, logprobs=bad))


def test_good_logprobs_pass_the_check():
    from samd_b200.batched import _check_logprobs
    assert [_check_logprobs(x) for x in (None, 0, 1, 8)] == [None, 0, 1, 8]


def _verifier():
    from samd_b200 import engine as E
    ver = E.Verifier.__new__(E.Verifier)
    ver.device, ver._h = torch.device("cpu"), None
    return ver


def _args(B=2, T=4, V=16, W=4):
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32)
    return dict(logits=torch.zeros(B, T, V), indices=i32(B, W), count=i32(B), tokens=i32(B, W), next_token=i32(B))


@pytest.mark.parametrize("change, msg", [
    (dict(n_top=9), r"n_top must be an int in \[0, 8\]"),
    (dict(n_top=-1), r"n_top must be an int in \[0, 8\]"),
    (dict(n_top=True), r"n_top must be an int in \[0, 8\]"),
    (dict(n_top=2.0), r"n_top must be an int in \[0, 8\]"),
    (dict(logits=torch.zeros(2, 16)), r"logits must be \[B, T, V\]"),
    (dict(logits=torch.zeros(2, 4, 16, dtype=torch.float64)), "unsupported logits dtype"),
    (dict(indices=torch.zeros(2, 3, dtype=torch.int32)), "tokens must be a contiguous"),
    (dict(indices=torch.zeros(2, 4, dtype=torch.int64)), "indices must be a contiguous"),
    (dict(count=torch.zeros(3, dtype=torch.int32)), "count must be a contiguous"),
    (dict(next_token=torch.zeros(2, dtype=torch.float32)), "next_token must be a contiguous"),
    (dict(n_nodes=torch.zeros(2, 1, dtype=torch.int32)), "n_nodes must be a contiguous"),
    (dict(done=torch.zeros(2, dtype=torch.int32)), "done must be a contiguous"),
    (dict(indices=None, tokens=torch.zeros(2, 5, dtype=torch.int32)), "identity path of width 5 needs 5 logits rows"),
    ({}, "every tensor must be on the GPU"),
])
def test_token_logprobs_argument_checks(change, msg):
    from samd_b200 import _cabi as K
    kw = _args()
    kw.update(change)
    with pytest.raises(K.SamdError, match=msg):
        _verifier().token_logprobs(**kw)
