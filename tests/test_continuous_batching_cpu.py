"""CPU checks of serve()'s request validation: each request is checked when it is pulled from the iterable, and a bad one
is refused with a SamdError naming its index."""
from types import SimpleNamespace

import pytest


def _decoder(T=8, max_len=512, max_tokens=1024):
    from samd_b200.batched import BatchedSamdDecoder
    dec = BatchedSamdDecoder.__new__(BatchedSamdDecoder)              # no device: only the host-side checks are used
    dec.T, dec.cache, dec.dyn = T, SimpleNamespace(max_len=max_len), SimpleNamespace(max_tokens=max_tokens)
    return dec


@pytest.mark.parametrize("prompts, limits, msg", [
    ([[3, 4], [], [5]], 8, "request 1: empty prompt"),
    ([[3], [4], [5]], [8, 8], "request 2: max_new_tokens has 2 values"),
    ([[3], [4]], [8, 0], "request 1: max_new_tokens must be >= 1"),
    ([[3], [4] * 505], 8, "request 1: prompt of 505 tokens"),
    ([[3] * 20, [4] * 100], [8, 1000], "request 1: prompt \\+ max_new_tokens"),
])
def test_requests_are_checked_as_they_are_pulled(prompts, limits, msg):
    from samd_b200 import _cabi as K
    dec = _decoder()
    it = dec._requests(iter(prompts), limits)
    pulled = []
    with pytest.raises(K.SamdError, match=msg):
        for r in it:
            pulled.append(r)
    bad = int(msg.split()[1].rstrip(":"))
    assert [i for i, _, _ in pulled] == list(range(bad))             # the requests before it were handed out


def test_valid_requests_keep_their_order_and_limits():
    dec = _decoder()
    prompts = ([3 + i] * (i + 1) for i in range(5))                   # any iterable, consumed lazily
    got = list(dec._requests(prompts, [8, 9, 10, 11, 12, 13]))
    assert [(i, len(p), lim) for i, p, lim in got] == [(i, i + 1, 8 + i) for i in range(5)]
    assert [lim for _, _, lim in dec._requests([[3], [4]], 7)] == [7, 7]
