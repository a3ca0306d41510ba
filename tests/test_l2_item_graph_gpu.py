"""The Euclidean item graph (distance="l2" / "l2sq") on the GPU: the tcgen05 candidate pass with the -d^2 score kind and
the batched exact scan, each against the C oracle (identical CSR structure, values within 1e-9), with the knn_* stats
showing which route ran."""
import ctypes as C
import os

import numpy as np
import pytest

RTOL = 1e-9


def _assert_graph_equal(gl, g):
    ip, ix, dt = gl.csr()
    oip, oix, odt = g.csr()
    assert gl.nnodes == g.nnodes
    assert np.array_equal(ip, oip), "CSR row pointers differ"
    assert np.array_equal(ix, oix), "CSR column indices differ"
    np.testing.assert_allclose(dt, odt, rtol=RTOL, atol=0)


def _kth(x, k, distance, sample=600, seed=0):
    """k-th-neighbour distance of a row sample against all rows (numpy; only used to choose eps values)."""
    rng = np.random.default_rng(seed)
    rows = rng.choice(x.shape[0], min(sample, x.shape[0]), replace=False)
    nsq = (x * x).sum(1)
    d2 = np.maximum(nsq[rows, None] + nsq[None, :] - 2.0 * x[rows] @ x.T, 0.0)
    d2[np.arange(len(rows)), rows] = np.inf
    d = np.sqrt(d2) if distance == "l2" else d2
    return np.sort(d, axis=1)[:, k - 1]


def _build(gp, x, distance, stage1, extra_env=None):
    from arrowspace import ArrowSpaceBuilder
    env = {"ASP_KNN_STAGE1": stage1}
    env.update(extra_env or {})
    os.environ.update(env)
    try:
        return ArrowSpaceBuilder.build_item_graph(gp, x, distance=distance)
    finally:
        for k in env:
            os.environ.pop(k, None)


def _shifted(n, f, seed):                              # the C4-style data: unit rows x 100, shifted to positive entries
    from pyarrowspace_b200 import synth
    return synth.make_items(n, f, seed, n_clusters=9)


def _wide_norms(n, f, seed):                           # mean-zero, norms over two decades
    from pyarrowspace_b200 import synth
    x = synth.make_items(n, f, seed, n_clusters=9, shift=0)
    return x * 10.0 ** np.random.default_rng(seed).uniform(-1.0, 1.0, size=(n, 1))


SHAPES = {"shifted": (_shifted, 3000, 96), "wide_norms": (_wide_norms, 3000, 64), "f37": (_shifted, 2500, 37),
          "above_8192": (_wide_norms, 8300, 48)}


@pytest.mark.gpu
@pytest.mark.parametrize("stage1", ["fp64", "tc"])
@pytest.mark.parametrize("distance", ["l2", "l2sq"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_l2_item_graph_parity(oracle_mod, shape, distance, stage1):
    """eps at the median of the k-th-neighbour distance: the radius binds on about half of the rows, the cap on the rest."""
    from pyarrowspace_b200 import api
    make, n, f = SHAPES[shape]
    x = make(n, f, 40 + f)
    k = 10
    kth = _kth(x, k, distance)
    eps = float(np.quantile(kth, 0.5))
    gp = {"eps": eps, "k": k, "topk": 3, "p": 2.0, "sigma": None}
    aspace, gl = _build(gp, x, distance, stage1)
    assert api.stat("knn_stage1_is_tc") == (1.0 if stage1 == "tc" else 0.0)
    if stage1 == "fp64":
        assert api.stat("knn_slow_rows") == n                        # the exact scan on every row
    s, g = oracle_mod.build(gp, x, nodes="items", distance=distance)
    _assert_graph_equal(gl, g)
    deg = np.diff(g.csr()[0]) - 1
    assert deg.min() < k <= deg.max()                               # some rows pruned by eps, some capped


@pytest.mark.gpu
@pytest.mark.parametrize("stage1", ["fp64", "tc"])
@pytest.mark.parametrize("distance", ["l2", "l2sq"])
def test_l2_item_graph_duplicates_hubs_zero_rows(oracle_mod, distance, stage1):
    """Exact duplicates (distance 0: ties by index), a hub of 90 copies of one row, and zero rows."""
    from pyarrowspace_b200 import api, synth
    base = synth.make_items(3000, 32, 8, n_clusters=3, shift=0) * np.linspace(0.2, 5.0, 3000)[:, None]
    x = np.concatenate([base, base[:50], base[:50], np.repeat(base[7:8], 90, axis=0), np.zeros((3, 32))])
    x = np.ascontiguousarray(x)
    eps = float(np.quantile(_kth(x, 6, distance), 0.4))
    gp = {"eps": eps, "k": 6, "topk": 3, "p": 2.0, "sigma": None}
    aspace, gl = _build(gp, x, distance, stage1)
    assert api.stat("knn_stage1_is_tc") == (1.0 if stage1 == "tc" else 0.0)
    s, g = oracle_mod.build(gp, x, nodes="items", distance=distance)
    _assert_graph_equal(gl, g)
    assert np.diff(gl.csr()[0]).max() > 64


@pytest.mark.gpu
def test_l2_item_graph_dense_clusters_switch_to_two_term(oracle_mod):
    """Dense neighbourhoods with a dominant mean direction: the one-term band holds hundreds of cluster members, the
    emission lists overflow and the rows are redone with the two-term split; the graph is still the oracle's."""
    from pyarrowspace_b200 import api
    rng = np.random.default_rng(77)
    ncl, per, f = 2, 4500, 64
    centres = rng.standard_normal((ncl, f))
    centres /= np.linalg.norm(centres, axis=1, keepdims=True)
    x = np.repeat(centres, per, axis=0) * (1.0 + 6e-2 * rng.standard_normal((ncl * per, f)))
    x = x * 100.0 + 60.0
    x = np.ascontiguousarray(x[rng.permutation(ncl * per)])
    eps = float(np.quantile(_kth(x, 5, "l2"), 0.5))
    gp = {"eps": eps, "k": 5, "topk": 3, "p": 2.0, "sigma": None}
    aspace, gl = _build(gp, x, "l2", "tc", {"ASP_KNN_BATCH": "4500", "ASP_TC_CAPB": "512"})
    stats = {k: api.stat(k) for k in ("knn_rows_two_term", "knn_slow_rows", "knn_stage1_is_tc")}
    assert stats["knn_stage1_is_tc"] == 1.0 and stats["knn_rows_two_term"] > 0, stats
    s, g = oracle_mod.build(gp, x, nodes="items", distance="l2")
    _assert_graph_equal(gl, g)


@pytest.mark.gpu
@pytest.mark.parametrize("distance", ["l2", "l2sq"])
def test_l2_item_knn_rows_equal_the_full_graph(oracle_mod, distance):
    """asp_item_knn_rows on row ranges gives the rows of the whole-range lists, and the lists make the oracle's graph."""
    import torch
    from pyarrowspace_b200 import _lib
    from pyarrowspace_b200.distributed import CudaEngine
    x = _wide_norms(9000, 40, 5)
    eps = float(np.quantile(_kth(x, 8, distance), 0.5))
    gp = {"eps": eps, "k": 8, "topk": 3, "p": 2.0, "sigma": None}
    cgp = _lib.make_params(eps, 8, 3, 2.0, None)
    sw = _lib.make_switches(distance=distance)
    eng = CudaEngine(0)
    space = eng.full_space(torch.from_numpy(x).cuda())
    full = [t.cpu().numpy() for t in eng.knn_rows(space, cgp, 0, 9000, sw)]
    for r0, r1 in ((0, 1), (1234, 5678), (8990, 9000), (4000, 4000)):
        part = [t.cpu().numpy() for t in eng.knn_rows(space, cgp, r0, r1, sw)]
        assert np.array_equal(part[2], full[2][r0:r1])
        for a, b, c in zip(part[0], full[0][r0:r1], part[2]):
            assert np.array_equal(a[:c], b[:c])
        for a, b, c in zip(part[1], full[1][r0:r1], part[2]):
            assert np.array_equal(a[:c], b[:c])
    idx, dst, cnt = (torch.from_numpy(v).cuda() for v in full)
    hg = eng.graph_from_knn(9000, idx, dst, cnt, cgp, sw)
    from pyarrowspace_b200 import api
    gl = api.GraphLaplacian._wrap(hg)
    s, g = oracle_mod.build(gp, x, nodes="items", distance=distance)
    _assert_graph_equal(gl, g)
    eng.lib.asp_free_space(space)


@pytest.mark.gpu
def test_search_after_l2_item_graph_is_bit_identical(oracle_mod):
    """The operand cache is keyed by its item order: a feature graph + lambdas + search on a space that built an l2 item
    graph first (norm-ordered cache) gives bit for bit the results of a fresh space (lambda-ordered cache)."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import _lib, api, synth
    x = synth.make_items(12000, 96, 31, n_clusters=16)
    q, _ = synth.make_queries(x, 700, 31)
    fgp = {"eps": 0.5, "k": 6, "topk": 10, "p": 2.0, "sigma": 0.25}
    eps = float(np.quantile(_kth(x, 6, "l2"), 0.5))
    aspace, gl_items = _build({"eps": eps, "k": 6, "topk": 3, "p": 2.0, "sigma": None}, x, "l2", "tc")
    assert api.stat("knn_stage1_is_tc") == 1.0
    lib = _lib.load()
    cgp = _lib.make_params(0.5, 6, 10, 2.0, 0.25)
    sw = _lib.make_switches()
    hg = C.c_void_p()
    _lib.check(lib.asp_space_feature_graph(aspace._h, C.byref(cgp), C.byref(sw), C.byref(hg)))
    gl = api.GraphLaplacian._wrap(hg)
    _lib.check(lib.asp_space_compute_lambdas(aspace._h, hg))
    idx, sc = aspace.search_batch(q, gl, 0.62)
    assert api.stat("search_stage1_is_tc") == 1.0
    fresh, gl2 = ArrowSpaceBuilder.build(fgp, x)
    idx2, sc2 = fresh.search_batch(q, gl2, 0.62)
    assert np.array_equal(aspace.lambdas(), fresh.lambdas())
    assert np.array_equal(idx, idx2)
    assert np.array_equal(sc, sc2, equal_nan=True)
    s, g = oracle_mod.build(fgp, x)
    oidx, osc, _ = s.search_batch(q, g, 0.62)
    assert np.array_equal(idx, oidx)


@pytest.mark.gpu
def test_l2_item_graph_refuses_what_it_cannot_do():
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import synth
    from pyarrowspace_b200._lib import LibraryError
    x = synth.make_items(9000, 16, 3)
    with pytest.raises(LibraryError):
        ArrowSpaceBuilder.build_item_graph({"eps": 1.0, "k": 31, "topk": 31, "p": 2.0, "sigma": None}, x, distance="l2")
    with pytest.raises(LibraryError):
        ArrowSpaceBuilder.build_item_graph({"eps": 1.0, "k": 5, "topk": 3, "p": 2.0, "sigma": None}, x * 1e20, distance="l2")
