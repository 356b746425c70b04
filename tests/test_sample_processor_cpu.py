"""The float64 sampling processor of the oracle (samd_oracle.processed_probs) against the one it restates: transformers'
TemperatureLogitsWarper -> TopPLogitsWarper -> TopKLogitsWarper followed by softmax, the processor list of
SamdGenerationConfig.prepare_logits_processor.  The GPU kernel is tested against processed_probs
(tests/test_gpu_sample_processor.py), so this pins what "the reference" means there.

top-p is placed halfway between two consecutive cumulative sums (computed in float64), so that float32 rounding inside
the warpers cannot move the cut.  On tie-group rows torch.sort may order equal values either way: there the number of
removed members and their values must agree, not their indices."""
import numpy as np
import pytest
import torch
from transformers.generation.logits_process import TemperatureLogitsWarper, TopKLogitsWarper, TopPLogitsWarper

import samd_oracle as O

V = 256


def _warped(row, temperature, top_p, top_k):
    s = torch.as_tensor(row, dtype=torch.float32)[None]
    ids = torch.zeros(1, 1, dtype=torch.long)
    if temperature != 1.0:
        s = TemperatureLogitsWarper(temperature)(ids, s)
    if top_p is not None:
        s = TopPLogitsWarper(top_p)(ids, s)
    if top_k > 0:
        s = TopKLogitsWarper(top_k)(ids, s)
    return s[0].double().numpy()


def _top_p_at(row, temperature, target, inside_group):
    """A top_p whose float64 cut lies halfway between two consecutive ascending cumulative sums near 1 - target,
    and the number of tokens it removes.  inside_group: the two tokens around the cut have equal values."""
    s = row.astype(np.float64) / temperature
    order = np.argsort(s, kind="stable")
    e = np.exp(s[order] - s.max())
    cum = np.cumsum(e / e.sum())
    ok = np.zeros(V, bool)
    ok[1:] = (s[order][1:] == s[order][:-1]) == inside_group
    j = int(np.nonzero(ok & (cum > 1.0 - target))[0][0])    # cum[j - 1] <= budget < cum[j]: j tokens removed
    top_p = 1.0 - 0.5 * (cum[j - 1] + cum[j])
    assert 0.5 * (cum[j] - cum[j - 1]) > 1e-4 * cum[j]        # far beyond float32 cumsum error at V = 256
    return float(top_p), j


@pytest.mark.parametrize("temperature", [0.7, 1.0, 1.5])
@pytest.mark.parametrize("target", [0.1, 0.5, 0.9, 0.999])
@pytest.mark.parametrize("top_k", [0, 1, 8, 50, V])
def test_processed_probs_equal_transformers_without_boundary_ties(temperature, target, top_k):
    rng = np.random.default_rng(int(target * 1000) + top_k)
    for _ in range(4):
        row = (rng.standard_normal(V) * 2.0).astype(np.float32)
        top_p, removed = _top_p_at(row, temperature, target, inside_group=False)
        got = O.processed_probs(row, temperature, top_p, top_k)
        w = _warped(row, temperature, top_p, top_k)
        want = np.exp(w - w.max())
        want /= want.sum()
        assert np.array_equal(got > 0, want > 0)
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-9)
        if top_k == 0:
            assert int((got == 0).sum()) == removed


@pytest.mark.parametrize("temperature", [0.7, 1.0])
@pytest.mark.parametrize("target", [0.3, 0.6, 0.95])
@pytest.mark.parametrize("top_k", [0, 2, 20, 100])
def test_processed_probs_remove_as_many_tie_members_as_transformers(temperature, target, top_k):
    rng = np.random.default_rng(int(target * 100) + top_k)
    for _ in range(4):
        row = (rng.integers(-6, 7, size=V) * 0.5).astype(np.float32)     # 13 values: groups of ~20 equal logits
        top_p, removed = _top_p_at(row, temperature, target, inside_group=True)
        got = O.processed_probs(row, temperature, top_p, top_k)
        w = _warped(row, temperature, top_p, top_k)
        assert int((got == 0).sum()) == int(np.isneginf(w).sum())
        assert np.array_equal(np.sort(row[got == 0]), np.sort(row[np.isneginf(w)]))
        if top_k == 0:
            assert int((got == 0).sum()) == removed
        want = np.exp(w - w.max())
        want /= want.sum()
        np.testing.assert_allclose(np.sort(got), np.sort(want), rtol=1e-5, atol=1e-9)
