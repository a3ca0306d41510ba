"""Per-call device memory is given back on every path: the bytes in use in the device's default memory pool (where the
library's stream-ordered allocations live) are the same before and after each call, whether it succeeds or fails, and
back at the starting level once every handle is freed.

The pool is read through the driver API (cuDeviceGetDefaultMemPool + CU_MEMPOOL_ATTR_USED_MEM_CURRENT) after
asp_ctx_synchronize, since a stream-ordered free completes on the stream.  PyTorch's caching allocator does not use this
pool unless PYTORCH_CUDA_ALLOC_CONF selects its cudaMallocAsync backend; the test skips in that case."""
import ctypes as C
import gc
import os

import numpy as np
import pytest

CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif("cudaMallocAsync" in os.environ.get("PYTORCH_CUDA_ALLOC_CONF", ""),
                       reason="PyTorch allocates from the same pool"),
]


class Pool:
    """Bytes in use in the default pool of the context's device, read once the context's stream is idle."""

    def __init__(self):
        from pyarrowspace_b200 import _lib
        self.lib, self.ctx = _lib.load(), _lib.context()
        self.cu = C.CDLL("libcuda.so.1")
        dev, self.pool = C.c_int(), C.c_void_p()
        assert self.cu.cuDeviceGet(C.byref(dev), self.lib.asp_ctx_device(self.ctx)) == 0
        assert self.cu.cuDeviceGetDefaultMemPool(C.byref(self.pool), dev) == 0

    def used(self):
        gc.collect()                                          # handles of dropped Python objects are freed here
        _check(self.lib.asp_ctx_synchronize(self.ctx))
        v = C.c_uint64()
        assert self.cu.cuMemPoolGetAttribute(self.pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(v)) == 0
        return v.value

    def same_after(self, fn, raises=None, warm=False):
        """fn() leaves the pool where it found it (raises: the exception type it must raise).  warm: one call first, so
        that what a first call builds for the space's lifetime (the fp16 operands, their three-term remainders) exists."""
        if warm:
            fn()
        before = self.used()
        if raises is None:
            fn()
        else:
            with pytest.raises(raises):
                fn()
        after = self.used()
        assert after == before, f"{after - before} bytes of device memory still in use after the call"


def _check(rc):
    from pyarrowspace_b200 import _lib
    _lib.check(rc)


@pytest.fixture(scope="module")
def pool():
    return Pool()


@pytest.fixture(scope="module")
def built():
    """Mean-zero items (the wide one-term band: the search retries part of its batch with the three-term split)."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import synth
    x = synth.make_items(20000, 64, 21, 100.0, n_clusters=8, shift=0.0)
    q = synth.make_fresh_queries(64, 2048, 121, n_clusters=8)[0]
    gp = {"eps": 0.5, "k": 6, "topk": 10, "p": 2.0, "sigma": 0.25}
    a, g = ArrowSpaceBuilder.build(gp, x, tau_mode="median_abs")
    mask = np.random.default_rng(3).random(20000) < 0.5
    a.search_batch(q, g, 0.6)                                 # warm-up: the space's persistent operand cache
    return x, q, gp, a, g, mask


def test_build_and_search(pool, built):
    import torch
    from arrowspace import ArrowSpaceBuilder
    x, q, gp, a, g, mask = built
    pool.same_after(lambda: ArrowSpaceBuilder.build(gp, x, tau_mode="median_abs"))
    pool.same_after(lambda: a.search_batch(q, g, 0.6), warm=True)
    qbig = np.ascontiguousarray(np.tile(q, (17, 1)))          # >= 32768 host queries: the pipelined path
    pool.same_after(lambda: a.search_batch(qbig, g, 0.6), warm=True)
    qd = torch.from_numpy(q).cuda()
    pool.same_after(lambda: a.search_batch(qd, g, 0.6), warm=True)
    pool.same_after(lambda: a.search_batch(q, g, 0.6, allowed=mask), warm=True)
    pool.same_after(lambda: a.search_hybrid_batch(q, g, 0.6), warm=True)
    pool.same_after(lambda: a.search_range_batch(q[:64], g, 0.6, 0.5), warm=True)


def test_search_errors(pool, built):
    from arrowspace import ArrowSpaceBuilder, PanicException
    x, q, gp, a, g, mask = built
    a.search_range_batch(q[:64], g, 0.6, 0.5)                # the range route's first call builds the three-term operands
    qz = q.copy()
    qz[5] = 0.0
    pool.same_after(lambda: a.search_batch(qz, g, 0.6), PanicException)
    pool.same_after(lambda: a.search_hybrid_batch(qz, g, 0.6), PanicException)
    pool.same_after(lambda: a.search_range_batch(qz, g, 0.6, 0.5), PanicException)
    pool.same_after(lambda: a.search_range_batch(q[:64], g, 0.6, -1.0, max_results=1), ValueError)
    pool.same_after(lambda: a.search_hybrid_batch(q, g, 0.6, pool=2000), Exception)
    xs = np.abs(np.random.default_rng(2).normal(size=(50, 6))) + 0.1
    a0, g0 = ArrowSpaceBuilder.build({"eps": 1.0, "k": 0, "topk": 2, "p": 2.0}, xs)      # no edges: every lambda is 0
    pool.same_after(lambda: a0.search_batch(xs[:4].copy(), g0, 0.5), PanicException)


def test_merges(pool):
    lib, ctx = pool.lib, pool.ctx
    rng = np.random.default_rng(5)
    parts, nq, topk, m = 3, 40, 4, 6
    idx = np.ascontiguousarray(rng.permutation(1000)[: parts * nq * topk].reshape(parts, nq, topk), dtype=np.int64)
    sc = -np.sort(-rng.random((parts, nq, topk)), axis=2)
    oi, os_ = np.empty((nq, topk), np.int64), np.empty((nq, topk))
    pool.same_after(lambda: _check(lib.asp_topk_merge(ctx, idx.ctypes.data, sc.ctypes.data, parts, nq, topk, oi.ctypes.data,
                                                      os_.ctypes.data)))
    hidx = np.ascontiguousarray(rng.permutation(1000)[: parts * nq * m].reshape(parts, nq, m), dtype=np.int64)
    hcos = -np.sort(-rng.random((parts, nq, m)), axis=2)
    hsc = rng.random((parts, nq, m))
    pool.same_after(lambda: _check(lib.asp_hybrid_merge(ctx, hidx.ctypes.data, hcos.ctypes.data, hsc.ctypes.data, parts, nq, m,
                                                        topk, oi.ctypes.data, os_.ctypes.data)))
    counts = rng.integers(0, 5, size=(parts, nq)).astype(np.int64)
    total = int(counts.sum())
    ridx, rsc = [], []
    for p in range(parts):
        for qi in range(nq):
            c = int(counts[p, qi])
            ridx.append(np.sort(rng.choice(1000, c, replace=False)))
            rsc.append(-np.sort(-rng.random(c)))
    ridx, rsc = np.ascontiguousarray(np.concatenate(ridx), np.int64), np.ascontiguousarray(np.concatenate(rsc))
    ro, rs = np.empty(total, np.int64), np.empty(total)
    pool.same_after(lambda: _check(lib.asp_range_merge(ctx, parts, nq, counts.ctypes.data, ridx.ctypes.data, rsc.ctypes.data,
                                                       ro.ctypes.data, rs.ctypes.data)))


def test_item_graphs(pool):
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import _lib, synth
    lib = pool.lib
    x = synth.make_items(9000, 48, 7, n_clusters=9)
    gp = {"eps": 0.3, "k": 8, "topk": 3, "p": 2.0, "sigma": None}
    gp2 = {"eps": 40.0, "k": 8, "topk": 3, "p": 2.0, "sigma": None}
    pool.same_after(lambda: ArrowSpaceBuilder.build_item_graph(gp, x))
    pool.same_after(lambda: ArrowSpaceBuilder.build_item_graph(gp2, x, distance="l2"))

    a, _ = ArrowSpaceBuilder.build_item_graph(gp, x)
    cgp, sw = _lib.make_params(0.3, 8, 3, 2.0, None), _lib.make_switches()
    rows = x.shape[0]                                         # every row: the lists make a graph over all items
    idx, dist, cnt, kk = np.empty((rows, 8), np.int32), np.empty((rows, 8)), np.empty(rows, np.int32), C.c_int32()

    def knn_rows():
        _check(lib.asp_item_knn_rows(a._h, C.byref(cgp), C.byref(sw), 0, rows, idx.ctypes.data, dist.ctypes.data,
                                     cnt.ctypes.data, C.byref(kk)))
    knn_rows()
    pool.same_after(knn_rows)

    def from_knn():
        h = C.c_void_p()
        _check(lib.asp_graph_from_knn(pool.ctx, rows, kk.value, idx.ctypes.data, dist.ctypes.data, cnt.ctypes.data, C.byref(cgp),
                                      C.byref(sw), C.byref(h)))
        lib.asp_free_graph(h)
    pool.same_after(from_knn)


def test_l2_item_graph_out_of_range_norms(pool):
    """The Euclidean tensor-core pass refuses norms above 1e18 after the neighbour lists exist: they are freed too."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import synth
    x = synth.make_items(8192, 32, 11, n_clusters=9)
    x[17] *= 1e19
    gp = {"eps": 40.0, "k": 8, "topk": 3, "p": 2.0, "sigma": None}
    pool.same_after(lambda: ArrowSpaceBuilder.build_item_graph(gp, x, distance="l2"), Exception)


def test_every_handle_freed(pool):
    """Build, search, range search and an item graph, then drop every handle: the pool is back where it started."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import synth
    start = pool.used()
    x = synth.make_items(9000, 48, 8, n_clusters=9)
    q = synth.make_queries(x, 512, 3)[0]
    a, g = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 10, "p": 2.0, "sigma": 0.3}, x)
    a.search_batch(q, g, 0.6)
    a.search_hybrid_batch(q, g, 0.6)
    a.search_range_batch(q[:32], g, 0.6, 0.5)
    ai, gi = ArrowSpaceBuilder.build_item_graph({"eps": 40.0, "k": 8, "topk": 3, "p": 2.0, "sigma": None}, x, distance="l2")
    assert pool.used() > start
    del a, g, ai, gi
    assert pool.used() == start
