"""CPU checks of the batched decoders' sampling parameters: every request's SamplingParams is checked when the request is
pulled, and a bad one - or a per-request list shorter than the prompts - is refused with a SamdError naming its index."""
from types import SimpleNamespace

import pytest


def _decoder(tree=None):
    from samd_b200.batched import BatchedSamdDecoder
    dec = BatchedSamdDecoder.__new__(BatchedSamdDecoder)              # no device: only the host-side checks are used
    dec.T, dec.cache, dec.dyn, dec.tree = 8, SimpleNamespace(max_len=512), SimpleNamespace(max_tokens=1024), tree
    return dec


def _pull(dec, prompts, sampling, limits=8):
    return dec._with_sampling(dec._requests(iter(prompts), limits), sampling)


@pytest.mark.parametrize("bad, msg", [
    (dict(temperature=0.0), "temperature must be >= 1e-5"),
    (dict(temperature=float("nan")), "temperature must be >= 1e-5"),
    (dict(top_p=1.5), "top_p must be in \\[0, 1\\]"),
    (dict(top_p=-0.1), "top_p must be in \\[0, 1\\]"),
    (dict(top_k=-1), "top_k must be an int >= 0"),
    (dict(top_k=2.5), "top_k must be an int >= 0"),
    (dict(seed=-3), "seed must be an int"),
    (dict(seed=2 ** 63), "seed must be an int"),
    (dict(greedy=1), "greedy must be a bool"),
])
def test_bad_params_are_refused_with_the_request_index(bad, msg):
    from samd_b200 import _cabi as K
    from samd_b200.batched import SamplingParams
    good = SamplingParams(temperature=0.7, top_p=0.9, top_k=5, seed=11)
    sampling = [good, good, SamplingParams(**bad), good]
    it = _pull(_decoder(), [[3], [4], [5], [6]], sampling)
    pulled = []
    with pytest.raises(K.SamdError, match="request 2: " + msg):
        for r in it:
            pulled.append(r)
    assert [r[0] for r in pulled] == [0, 1] and all(r[3] == good for r in pulled)


def test_short_lists_and_wrong_types_name_the_request():
    from samd_b200 import _cabi as K
    from samd_b200.batched import SamplingParams
    sp = SamplingParams()
    with pytest.raises(K.SamdError, match="request 2: sampling has 2 values, fewer than the prompts"):
        list(_pull(_decoder(), [[3], [4], [5]], [sp, sp]))
    with pytest.raises(K.SamdError, match="request 1: sampling must be a SamplingParams, got dict"):
        list(_pull(_decoder(), [[3], [4]], [sp, dict(temperature=1.0)]))
    # one shared SamplingParams: the seed of request i is seed + i, and its last admissible value is checked too
    with pytest.raises(K.SamdError, match="request 1: seed must be an int"):
        list(_pull(_decoder(), [[3], [4]], SamplingParams(seed=2 ** 63 - 1)))


def test_per_request_params_and_shared_seeds():
    from samd_b200.batched import SamplingParams
    shared = SamplingParams(temperature=0.7, top_p=0.9, seed=100)
    got = list(_pull(_decoder(), ([3 + i] for i in range(4)), shared, [8, 9, 10, 11]))
    assert [(i, lim, sp.seed, sp.temperature, sp.top_p) for i, _, lim, sp in got] == \
        [(i, 8 + i, 100 + i, 0.7, 0.9) for i in range(4)]
    own = [SamplingParams(seed=5), SamplingParams(greedy=True, temperature=0.0), SamplingParams(top_k=3, seed=9)]
    got = list(_pull(_decoder(), [[3], [4], [5]], own))
    assert [sp for *_, sp in got] == own                              # a greedy request needs no temperature
    assert [sp for *_, sp in _pull(_decoder(), [[3], [4]], None)] == [None, None]


def test_tree_mode_refuses_sampling():
    from samd_b200 import _cabi as K
    from samd_b200.batched import SamplingParams
    with pytest.raises(K.SamdError, match="Token-Recycle tree mode"):
        _pull(_decoder(tree=[[1], []]), [[3]], SamplingParams())
    assert list(_pull(_decoder(tree=[[1], []]), [[3]], None))[0][3] is None
