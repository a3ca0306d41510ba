"""The tau sweep on the GPU (ArrowSpace.search_batch_taus, asp_search_batch_taus).  Every case: idx[t], score[t] equal,
bit for bit, the stacked search_batch(queries, gl, taus[t], allowed=..., k=...) calls, and a sample of queries equals the
oracle (indices identical, scores to RTOL).  The route stats tell a shared candidate pass from the per-tau route.
Run with -m gpu."""
import numpy as np
import pytest

from test_filtered_search_gpu import RTOL, _mask, _same, _spaces
from test_large_k_gpu import TC, _oracle

pytestmark = pytest.mark.gpu


def _tc(oracle_mod, nq=None):
    n, f, topk, nq0, tau, shift, dup = TC
    return _spaces(oracle_mod, n, f, topk, 11 + n + f, nq or nq0, shift, dup)


def _check(a1, g1, s, g, q, taus, k=None, allowed=None, sample=(0, 7, -1)):
    """The sweep against the per-tau loop (bits) and, for a few queries, the oracle.  Returns (idx, score)."""
    idx, sc = a1.search_batch_taus(q, g1, taus, allowed=allowed, k=k)
    kk = g1.graph_params["topk"] if k is None else k
    assert idx.shape == sc.shape == (len(taus), q.shape[0], kk)
    for t, tau in enumerate(taus):
        i1, s1 = a1.search_batch(q, g1, float(tau), allowed=allowed, k=k)
        assert np.array_equal(idx[t], i1), "tau %r rows %s" % (tau, np.where((idx[t] != i1).any(axis=1))[0][:10])
        assert np.array_equal(sc[t], s1, equal_nan=True), tau
        pick = np.array(sample) % q.shape[0]
        qq = np.ascontiguousarray(q[pick])
        _same(idx[t][pick], sc[t][pick], *_oracle(s, g, qq, float(tau), kk, allowed), RTOL)
    return idx, sc


def _stats():
    from pyarrowspace_b200.api import stat
    return stat("sweep_fused_taus"), stat("sweep_stage1_passes")


@pytest.mark.parametrize("taus,passes", [((1.0, 0.8, 0.62), 1), ((0.62, 0.62), 1), ((1.0, 0.5, 0.2, 0.05), 2),
                                         ((1.0, 0.8, 0.62, 0.5, 0.3), 2)])
@pytest.mark.parametrize("k", [None, 1, 16])
def test_fused_sweep_equals_per_tau_search(oracle_mod, taus, passes, k):
    x, q, a1, g1, s, g = _tc(oracle_mod)
    _check(a1, g1, s, g, q, taus, k)
    assert _stats() == (len(taus), passes)


@pytest.mark.parametrize("density", ["1.0", "0.1", "0.001", "none"])
def test_fused_sweep_with_masks(oracle_mod, density):
    x, q, a1, g1, s, g = _tc(oracle_mod)
    mask = _mask(x.shape[0], density, 5)
    idx, sc = _check(a1, g1, s, g, q, (1.0, 0.8, 0.62), None, mask)
    assert _stats() == (3, 1)
    if density == "none":
        assert (idx == -1).all() and np.isnan(sc).all()


def test_duplicate_items_and_near_ties_take_the_exact_scan(oracle_mod, monkeypatch):
    """Duplicate rows: ties by index across the k-th place; the tiny emission buffers make every query overflow, so
    every tau's queries take the exact scan."""
    monkeypatch.setenv("ASP_SEARCH_STAGE1", "tc")
    from pyarrowspace_b200.api import stat
    x, q, a1, g1, s, g = _spaces(oracle_mod, 3000, 24, 12, 3035, 300, True, 300)
    _check(a1, g1, s, g, q, (1.0, 0.62, 0.3), 12)
    assert _stats() == (3, 1)
    monkeypatch.setenv("ASP_TC_CAPB", "8")
    _check(a1, g1, s, g, q, (1.0, 0.62, 0.3), 12)
    assert _stats() == (3, 1) and stat("search_slow_queries") > 0


def test_mean_zero_wide_band_takes_the_three_term_retry(oracle_mod, monkeypatch):
    monkeypatch.setenv("ASP_SEARCH_STAGE1", "tc")
    from pyarrowspace_b200.api import stat
    x, q, a1, g1, s, g = _spaces(oracle_mod, 20000, 96, 10, 20096 + 11, 600, "mean_zero", 0)
    _check(a1, g1, s, g, q, (1.0, 0.8, 0.62))
    assert _stats() == (3, 1) and stat("search_terms") in (1.0, 3.0)


def test_small_capacity_overflow_takes_the_slow_path(oracle_mod, monkeypatch):
    monkeypatch.setenv("ASP_TC_CAPB", "8")
    from pyarrowspace_b200.api import stat
    x, q, a1, g1, s, g = _tc(oracle_mod)
    _check(a1, g1, s, g, q, (1.0, 0.62))
    assert _stats() == (2, 1) and stat("search_slow_queries") > 0


@pytest.mark.parametrize("taus,k,fused,passes", [((1.0, 0.62), 17, 0, 0), ((0.62, 0.8), 100, 0, 0),
                                                 ((0.0, 1.0, 0.001, 0.62, 1.5, -0.2, 0.8), None, 3, 1),
                                                 ((0.0, 0.62), None, 0, 0), ((0.62,), None, 0, 0)])
def test_per_tau_routes(oracle_mod, taus, k, fused, passes):
    """k beyond 16, taus outside (0.001, 1] mixed with fused ones, and a lone qualifying tau: the per-tau route, in order."""
    x, q, a1, g1, s, g = _tc(oracle_mod)
    _check(a1, g1, s, g, q, taus, k)
    assert _stats() == (fused, passes)


def test_small_batch_on_a_small_space_takes_the_fp64_route(oracle_mod):
    x, q, a1, g1, s, g = _spaces(oracle_mod, 2000, 32, 8, 2043, 40, True, 0)
    _check(a1, g1, s, g, q, (1.0, 0.62, 0.3))
    assert _stats() == (0, 0)


def test_one_query_against_a_large_space_is_fused(oracle_mod):
    x, q, a1, g1, s, g = _spaces(oracle_mod, 140000, 32, 10, 140000 + 32 + 11, 1, True, 0)
    _check(a1, g1, s, g, q, (1.0, 0.8, 0.62), sample=(0,))
    assert _stats() == (3, 1)


def test_device_tensors_in_and_out(oracle_mod):
    import torch
    x, q, a1, g1, s, g = _tc(oracle_mod)
    idx, sc = a1.search_batch_taus(torch.from_numpy(q).cuda(), g1, [1.0, 0.62], k=5)
    assert idx.is_cuda and sc.is_cuda and idx.shape == (2, q.shape[0], 5)
    hi, hs = a1.search_batch_taus(q, g1, [1.0, 0.62], k=5)
    assert np.array_equal(idx.cpu().numpy(), hi) and np.array_equal(sc.cpu().numpy(), hs, equal_nan=True)


def test_panics_are_those_of_search_batch(oracle_mod):
    from arrowspace import ArrowSpaceBuilder, PanicException
    x, q, a1, g1, s, g = _tc(oracle_mod)
    bad = q.copy()
    bad[5] = 0.0
    with pytest.raises(PanicException, match="all zeros"):
        a1.search_batch_taus(bad, g1, [1.0, 0.62])
    xs = np.abs(np.random.default_rng(2).normal(size=(10, 6))) + 0.1
    a0, g0 = ArrowSpaceBuilder.build({"eps": 1.0, "k": 0, "topk": 2, "p": 2.0}, xs)
    with pytest.raises(PanicException, match="The lambdas are zero, check the magnitude of items and eps."):
        a0.search_batch_taus(np.ascontiguousarray(xs[:3]), g0, [1.0, 0.62])
    idx, _ = a1.search_batch_taus(q, g1, [1.0, 0.62])                     # usable after the failed calls
    assert np.array_equal(idx[1], a1.search_batch(q, g1, 0.62)[0])
