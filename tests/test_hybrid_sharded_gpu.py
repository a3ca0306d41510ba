"""search_hybrid on item-sharded spaces, on one GPU: R = 2, 4, 8 row shards live on the same device (as in
test_shards_on_one_gpu_equal_single), each answers asp_search_hybrid_shard, and asp_hybrid_merge (asp_topk_merge for the
whole set) of their lists must equal the one-GPU asp_search_hybrid_batch and orc_search_hybrid bit for bit.  Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _data(n, f, seed, nq, dup):
    rng = np.random.default_rng(seed)
    cent = rng.normal(size=(8, f))
    x = np.abs(cent[rng.integers(0, 8, n)] + 0.2 * rng.normal(size=(n, f))) + 0.05
    if dup:
        x[n - dup - 5:n - 5] = x[:dup]                       # duplicates in the first and the last shard
    q = x[rng.integers(0, n, nq)] * 1.02 + 0.01 * rng.normal(size=(nq, f))
    if dup:
        q[:3] = x[:3] * 1.5                                  # ties in cosine and score across the shard boundary
    return x, q


def _shards(x, world, a1, only=None):
    """Row shards of `world` (or only shard `only`) on cuda:0 with the one-GPU space's lambdas and norms (what regroup
    imports)."""
    from pyarrowspace_b200 import _lib, shard_rows
    lib = _lib.load()
    n, f = x.shape
    lam, nrm = a1.lambdas(), a1.norms()
    out = []
    for r in (range(world) if only is None else [only]):
        r0, r1 = shard_rows(n, world, r)
        h = C.c_void_p()
        xs = np.ascontiguousarray(x[r0:r1])
        _lib.check(lib.asp_space_create(a1._ctx, xs.ctypes.data, r1 - r0, f, n, world, r, C.byref(h)))
        _lib.check(lib.asp_space_import_lambdas(h, np.ascontiguousarray(lam[r0:r1]).ctypes.data,
                                                np.ascontiguousarray(nrm[r0:r1]).ctypes.data))
        out.append(h)
    return out


def _sharded_hybrid(shards, gl, q, tau, pool, topk, n):
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    nq = q.shape[0]
    m = lib.asp_hybrid_pool(n, topk, pool)
    whole = m >= n
    width = topk if whole else m
    parts = len(shards)
    idx = np.empty((parts, nq, width), dtype=np.int64)
    cos = np.empty((parts, nq, width))
    sc = np.empty((parts, nq, width))
    lam = np.empty((parts, nq))
    for r, h in enumerate(shards):
        _lib.check(lib.asp_search_hybrid_shard(h, gl._h, q.ctypes.data, nq, tau, pool, idx[r].ctypes.data,
                                               None if whole else cos[r].ctypes.data, sc[r].ctypes.data, lam[r].ctypes.data))
    assert all(np.array_equal(lam[r], lam[0]) for r in range(parts))
    out_idx = np.empty((nq, topk), dtype=np.int64)
    out_sc = np.empty((nq, topk))
    ctx = _lib.context()
    if whole:
        _lib.check(lib.asp_topk_merge(ctx, idx.ctypes.data, sc.ctypes.data, parts, nq, topk, out_idx.ctypes.data,
                                      out_sc.ctypes.data))
    else:
        _lib.check(lib.asp_hybrid_merge(ctx, idx.ctypes.data, cos.ctypes.data, sc.ctypes.data, parts, nq, m, topk,
                                        out_idx.ctypes.data, out_sc.ctypes.data))
    return out_idx, out_sc, lam[0], idx


@pytest.mark.parametrize("n,f,topk,pool,nq,dup", [
    (5000, 96, 10, 0, 300, 0),          # shortlist 20 on tcgen05 (batch >= 256)
    (5000, 96, 10, 0, 7, 0),            # the small-batch candidate pass
    (5000, 64, 3, 31, 257, 12),         # the longest tensor-core list, duplicated rows across shards
    (4000, 130, 20, 40, 64, 0),         # shortlist 40: the batched exact scan
    (6000, 48, 5, 1024, 40, 12),        # shortlist 1024: shards of 8 are smaller than m (padded lists)
    (1500, 48, 4, 5000, 33, 0),         # pool >= n: the whole set (asp_topk_merge of plain-search lists)
])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_hybrid_equals_one_gpu_and_oracle(oracle_mod, world, n, f, topk, pool, nq, dup):
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import _lib
    x, q = _data(n, f, n + f + topk, nq, dup)
    gp = {"eps": 0.6, "k": 5, "topk": topk, "p": 2.0, "sigma": 0.3}
    a1, g1 = ArrowSpaceBuilder.build(gp, x)
    s, g = oracle_mod.build(gp, x)
    shards = _shards(x, world, a1)
    try:
        for tau in (0.62, 0.0):
            if pool >= n and tau == 0.0:
                continue                                  # the plain search needs tau > 0 on its tensor-core route
            idx, sc, lq, lists = _sharded_hybrid(shards, g1, q, tau, pool, topk, n)
            i1, s1, l1 = a1.search_hybrid_batch(q, g1, tau, pool=pool or None, want_lambda=True)
            assert np.array_equal(lq, l1)
            assert np.array_equal(idx, i1), "rows %s" % np.where((idx != i1).any(axis=1))[0][:10]
            ok = i1 >= 0
            assert np.array_equal(sc[ok], s1[ok]) and np.isnan(sc[~ok]).all()
            oidx, osc, olq = s.search_hybrid_batch(q, g, tau, pool)
            assert np.array_equal(idx, oidx)
            np.testing.assert_allclose(sc[ok], osc[ok], rtol=1e-9, atol=0)
            if pool < n:                                  # each shard lists min(m, its rows) entries, then -1 padding
                from pyarrowspace_b200 import shard_rows
                for r in range(world):
                    r0, r1 = shard_rows(n, world, r)
                    assert ((lists[r] >= 0).sum(axis=1) == min(lists.shape[2], r1 - r0)).all()
                    assert ((lists[r] >= r0) & (lists[r] < r1) | (lists[r] == -1)).all()
    finally:
        lib = _lib.load()
        for h in shards:
            lib.asp_free_space(h)


def test_shard_call_contract(oracle_mod):
    """asp_search_hybrid_batch still refuses a row shard; asp_search_hybrid_shard refuses a shortlist above 1024 and
    reports a zero query vector; asp_hybrid_pool is the one-GPU rule."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    x, q = _data(3000, 32, 4, 5, 0)
    a1, g1 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 4, "p": 2.0, "sigma": 0.3}, x)
    assert [lib.asp_hybrid_pool(3000, 4, p) for p in (0, 2, 50, 5000)] == [8, 4, 50, 3000]
    assert lib.asp_hybrid_pool(3000, 20, 0) == 31 and lib.asp_hybrid_pool(6, 4, 0) == 6
    shards = _shards(x, 2, a1)
    try:
        idx = np.empty((5, 2000), dtype=np.int64)
        sc = np.empty((5, 2000))
        assert lib.asp_search_hybrid_batch(shards[0], g1._h, q.ctypes.data, 5, 0.5, 0, idx.ctypes.data, sc.ctypes.data,
                                           None) == _lib.ASP_ERR_UNSUPPORTED
        cos = np.empty((5, 2000))
        assert lib.asp_search_hybrid_shard(shards[0], g1._h, q.ctypes.data, 5, 0.5, 2000, idx.ctypes.data, cos.ctypes.data,
                                           sc.ctypes.data, None) == _lib.ASP_ERR_UNSUPPORTED
        qz = q.copy()
        qz[2] = 0.0
        assert lib.asp_search_hybrid_shard(shards[1], g1._h, qz.ctypes.data, 5, 0.5, 0, idx.ctypes.data, cos.ctypes.data,
                                           sc.ctypes.data, None) == _lib.ASP_ERR_ZERO_VECTOR
    finally:
        for h in shards:
            lib.asp_free_space(h)


def _api_worker(rank, world, item_shards, port, out):
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        from arrowspace import ArrowSpaceBuilder, PanicException
        from pyarrowspace_b200 import api
        from pyarrowspace_b200.distributed import grid_groups, grid_layout
        x, q = _data(3000, 64, 8, 300, 12)
        a1, g1 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 6, "p": 2.0, "sigma": 0.3}, x, device=0)
        r_, c_, r, c = grid_layout(world, rank, item_shards)
        grid = dict(R=r_, C=c_, r=r, c=c, item_group=None, merge_group=None)
        if c_ > 1:
            item_groups, merge_groups = grid_groups(world, r_)
            grid["item_group"], grid["merge_group"] = item_groups[r], merge_groups[c]
        sp = api.ArrowSpace._wrap(_shards(x, r_, a1, only=r)[0], a1._ctx, grid["merge_group"], grid)
        same = {}
        for pool in (None, 40, 5000):
            hi, hs, hl = sp.search_hybrid_batch(q, g1, 0.62, pool=pool, want_lambda=True)
            i1, s1, l1 = a1.search_hybrid_batch(q, g1, 0.62, pool=pool, want_lambda=True)
            same[pool] = bool(np.array_equal(hi, i1) and np.array_equal(hs, s1, equal_nan=True) and np.array_equal(hl, l1))
        hits = sp.search_hybrid(q[7].copy(), g1, 0.62)
        same["single"] = [i for i, _ in hits] == list(a1.search_hybrid_batch(q[7:8], g1, 0.62)[0][0])
        qz = q.copy()
        qz[-1] = 0.0                                          # in the last query slot only
        try:
            sp.search_hybrid_batch(qz, g1, 0.62)
            raised = None
        except PanicException as e:
            raised = "PanicException"
        out.put((rank, same, raised))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        out.put((rank, "error", repr(e)))
        raise


@pytest.mark.parametrize("world,item_shards", [(2, 2), (4, 4), (4, 2)])
def test_public_search_hybrid_on_item_shards(world, item_shards):
    """ArrowSpace.search_hybrid_batch / search_hybrid on item shards through the product path (CudaEngine, the
    orchestration, the C ABI): `world` processes share cuda:0 and exchange over gloo.  Every rank returns the one-GPU answer
    bit for bit (default shortlist, pool 40, whole set), and a zero query raises PanicException on every rank."""
    import socket
    import torch.multiprocessing as mp
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_api_worker, args=(r, world, item_shards, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[1] != "error" for r in res), res
    for rank, same, raised in res:
        assert all(same.values()), (rank, same)
        assert raised == "PanicException", rank
