"""CPU checks of prefix reuse's host side: longest-prefix matching over the registered prefixes and add_prefix's
validation, on a decoder built without a device."""
from types import SimpleNamespace

import pytest


def _decoder(prefixes, T=8, max_len=512, max_tokens=1024):
    from samd_b200.batched import BatchedSamdDecoder
    dec = BatchedSamdDecoder.__new__(BatchedSamdDecoder)              # no device: only the host-side logic is used
    dec.T, dec.cache, dec.dyn = T, SimpleNamespace(max_len=max_len), SimpleNamespace(max_tokens=max_tokens)
    dec._prefixes = None if prefixes is None else [None if p is None else dict(tokens=tuple(p)) for p in prefixes]
    return dec


def test_longest_registered_prefix_wins():
    A = [5, 6, 7, 8]
    dec = _decoder([A, None, A + [9, 10], [5, 6, 30], [40]])
    assert dec._longest_prefix(A + [9, 10, 11]) == (2, 6)
    assert dec._longest_prefix(A + [9, 10]) == (2, 6)               # a prompt equal to a prefix
    assert dec._longest_prefix(A + [9, 11]) == (0, 4)               # A2 only partly shared: A
    assert dec._longest_prefix([5, 6, 30, 1]) == (3, 3)
    assert dec._longest_prefix([5, 6, 7]) == (None, 0)              # shorter than every prefix it starts
    assert dec._longest_prefix([41, 5, 6, 7, 8]) == (None, 0)
    assert dec._longest_prefix((40, 1)) == (4, 1)                   # any sequence type
    import numpy as np
    assert dec._longest_prefix(np.array(A + [9, 10, 3])) == (2, 6)


@pytest.mark.parametrize("tokens, msg", [
    ([], "empty prefix"),
    ([3] * 505, "prefix of 505 tokens \\+ one decode step of 8 does not fit max_cache_len=512"),
    ([3] * 300, "exceeds the automaton capacity max_tokens=305"),
])
def test_add_prefix_validation(tokens, msg):
    from samd_b200 import _cabi as K
    dec = _decoder([None], max_tokens=305)
    with pytest.raises(K.SamdError, match=msg):
        dec.add_prefix(tokens)


def test_add_prefix_pool_rules():
    from samd_b200 import _cabi as K
    with pytest.raises(K.SamdError, match="no prefix pool"):
        _decoder(None).add_prefix([1, 2])
    dec = _decoder([[1, 2], None, [3]])
    assert dec._check_prefix((3,)) == 2                             # identical tokens: the existing id
    assert dec._check_prefix((1, 2, 3)) == 1                        # the first free row
    full = _decoder([[1, 2], [3]])
    assert full.add_prefix([3]) == 1                                # already registered: no device work
    with pytest.raises(K.SamdError, match="pool is full \\(2 prefixes\\)"):
        full.add_prefix([4])
    with pytest.raises(K.SamdError, match="no registered prefix 5"):
        full.drop_prefix(5)
    full.drop_prefix(0)
    assert full._longest_prefix([1, 2, 3]) == (None, 0)
    assert full._check_prefix((4,)) == 0
