"""Search with a per-call k on the GPU (search_batch / search_hybrid_batch k=, asp_search_batch_k and the hybrid _k entry
points).  The reference is the unchanged oracle: orc_scores of every item ranked by (score desc, index asc) and cut to k
(test_filtered_search_cpu.want_search); indices identical, scores to the tolerance the other oracle comparisons use (the
oracle's lambdas differ from the GPU's in the last bits).  Against the GPU's own graph-topk path the bits are identical.
Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

from test_filtered_search_cpu import want_hybrid, want_search
from test_filtered_search_gpu import RTOL, _mask, _same, _spaces
from test_hybrid_sharded_gpu import _data as _shard_data
from test_hybrid_sharded_gpu import _shards

pytestmark = pytest.mark.gpu

KS = [20, 32, 33, 64, 100, 128, 129, 300]
TC = (20000, 64, 10, 300, 0.62, True, 0)          # n, f, graph topk, nq, tau, shift, dup: qualifies for the tensor-core pass
DUP = (3000, 24, 12, 300, 0.62, True, 300)         # duplicate rows: exact ties across the k-th place


def _oracle(s, g, q, tau, k, mask=None):
    lq = s.search_batch(q, g, tau)[2]
    return want_search(s, q, lq, tau, np.ones(len(s.lambdas()), dtype=bool) if mask is None else mask, k)


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("case", ["tc", "dup"])
def test_search_k_equals_oracle(oracle_mod, case, k):
    from pyarrowspace_b200.api import stat
    n, f, topk, nq, tau, shift, dup = TC if case == "tc" else DUP
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    idx, sc = a1.search_batch(q, g1, tau, k=k)
    assert idx.shape == (nq, k)
    _same(idx, sc, *_oracle(s, g, q, tau, k), RTOL)
    if 32 <= k <= 64:                                          # the wide tensor-core route, not the exact scan of every query
        assert stat("search_stage1_is_tc") == 1 and stat("search_slow_queries") < nq // 4


@pytest.mark.parametrize("density", ["1.0", "0.5", "0.01", "fewer"])
@pytest.mark.parametrize("k", [33, 64, 100])
def test_search_k_with_masks(oracle_mod, density, k):
    n, f, topk, nq, tau, shift, dup = TC
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    if density == "fewer":                                     # fewer allowed items than k
        mask = np.zeros(n, dtype=bool)
        mask[np.random.default_rng(k).permutation(n)[:k - 5]] = True
    else:
        mask = _mask(n, density, k)
    idx, sc = a1.search_batch(q, g1, tau, allowed=mask, k=k)
    oi, osc = _oracle(s, g, q, tau, k, mask)
    _same(idx, sc, oi, osc, RTOL)
    assert (oi >= 0).sum(axis=1).tolist() == [min(k, int(mask.sum()))] * nq


def test_k_matches_a_graph_built_with_topk_k_bit_for_bit(oracle_mod):
    """The same answer, bit for bit, as the graph-topk call of a graph built with topk = k (default switches: topk does not
    change the graph), and k equal to the graph's topk is the call without k."""
    from arrowspace import ArrowSpaceBuilder
    n, f, topk, nq, tau, shift, dup = TC
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    i0, s0 = a1.search_batch(q, g1, tau)
    ik, sk = a1.search_batch(q, g1, tau, k=topk)
    assert np.array_equal(i0, ik) and np.array_equal(s0, sk, equal_nan=True)
    for k in (48, 100):
        a2, g2 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": k, "p": 2.0, "sigma": 0.3}, x)
        i2, s2 = a2.search_batch(q, g2, tau)
        ik, sk = a1.search_batch(q, g1, tau, k=k)
        assert np.array_equal(i2, ik) and np.array_equal(s2, sk, equal_nan=True)


def test_prefix_property(oracle_mod):
    n, f, topk, nq, tau, shift, dup = TC
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    i10, s10 = a1.search_batch(q, g1, tau, k=10)
    for k in (33, 64, 100):
        ik, sk = a1.search_batch(q, g1, tau, k=k)
        assert np.array_equal(ik[:, :10], i10) and np.array_equal(sk[:, :10], s10)


@pytest.mark.parametrize("case", ["mean_zero", "small_tau", "large_shard_one_query", "k_beyond_n", "device"])
def test_search_k_other_routes(oracle_mod, monkeypatch, case):
    import torch
    k = 48
    if case == "mean_zero":                                    # the wide one-term band, then the three-term retry
        monkeypatch.setenv("ASP_SEARCH_STAGE1", "tc")
        x, q, a1, g1, s, g = _spaces(oracle_mod, 20000, 96, 10, 20096 + 11, 600, "mean_zero", 0)
        tau = 0.62
    elif case == "small_tau":                                  # tau <= 0.001: not the tensor-core pass
        x, q, a1, g1, s, g = _spaces(oracle_mod, *TC[:3], 11 + TC[0] + TC[1], *TC[3:4], *TC[5:])
        tau = 0.001
    elif case == "large_shard_one_query":
        x, q, a1, g1, s, g = _spaces(oracle_mod, 140000, 32, 10, 140000 + 32 + 11, 1, True, 0)
        tau = 0.62
    elif case == "k_beyond_n":
        x, q, a1, g1, s, g = _spaces(oracle_mod, 40, 16, 5, 67, 300, True, 0)
        tau = 0.62
    else:
        x, q, a1, g1, s, g = _spaces(oracle_mod, *TC[:3], 11 + TC[0] + TC[1], *TC[3:4], *TC[5:])
        tau = 0.62
    for kk in ((k, 300) if case == "k_beyond_n" else (k,)):
        if case == "device":
            qd = torch.from_numpy(q).cuda()
            idx, sc = a1.search_batch(qd, g1, tau, k=kk)
            assert idx.is_cuda and idx.shape == (q.shape[0], kk)
            idx, sc = idx.cpu().numpy(), sc.cpu().numpy()
        else:
            idx, sc = a1.search_batch(q, g1, tau, k=kk)
        _same(idx, sc, *_oracle(s, g, q, tau, kk), RTOL)


def test_pipelined_host_batch(oracle_mod, monkeypatch):
    """32768 host queries or more: the two-piece pipeline; the same bits as one shot, a sample against the oracle."""
    from pyarrowspace_b200 import synth
    n, f, topk, nq, tau, shift, dup = TC
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    qq = np.ascontiguousarray(np.concatenate([q] * 110)[:32800] * (1.0 + 1e-3 * np.arange(32800)[:, None] / 32800))
    ip, sp = a1.search_batch(qq, g1, tau, k=40)
    monkeypatch.setenv("ASP_NO_PIPELINE", "1")
    i1, s1 = a1.search_batch(qq, g1, tau, k=40)
    assert np.array_equal(ip, i1) and np.array_equal(sp, s1, equal_nan=True)
    pick = np.arange(0, 32800, 997)
    _same(ip[pick], sp[pick], *_oracle(s, g, np.ascontiguousarray(qq[pick]), tau, 40), RTOL)


@pytest.mark.parametrize("k,pool", [(20, None), (50, None), (100, None), (40, 64)])
def test_hybrid_k_equals_oracle_on_a_graph_of_topk_k(oracle_mod, k, pool):
    n, f, topk, nq, tau, shift, dup = TC
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    s2, g2 = oracle_mod.build({"eps": 0.6, "k": 5, "topk": k, "p": 2.0, "sigma": 0.3}, x)
    oi, osc, _ = s2.search_hybrid_batch(q, g2, tau, pool or 0)
    idx, sc = a1.search_hybrid_batch(q, g1, tau, pool=pool, k=k)
    assert idx.shape == (nq, k)
    _same(idx, sc, oi, osc, RTOL)
    mask = _mask(n, "0.5", k)
    idx, sc = a1.search_hybrid_batch(q, g1, tau, pool=pool, k=k, allowed=mask)
    _same(idx, sc, *want_hybrid(s2, q, s2.search_hybrid_batch(q, g2, tau, 0)[2], tau, pool or 0, mask, k), RTOL)
    one = a1.search_hybrid(q[3].copy(), g1, tau, pool=pool, k=k)
    assert [i for i, _ in one] == [i for i in oi[3] if i >= 0]


# ----------------------------------------------------------------------------- item shards

@pytest.mark.parametrize("world", [2, 4])
def test_shards_on_one_gpu_equal_one_gpu(world):
    """Row shards on cuda:0: asp_search_batch_k per shard + asp_topk_merge, and asp_search_hybrid_shard_k +
    asp_hybrid_merge, equal the one-GPU calls bit for bit."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    x, q = _shard_data(6000, 32, 4, 300, 12)
    a1, g1 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 6, "p": 2.0, "sigma": 0.3}, x, device=0)
    n, nq = x.shape[0], q.shape[0]
    shards = _shards(x, world, a1)
    try:
        for k in (40, 64, 130):
            parts_i = np.empty((world, nq, k), dtype=np.int64)
            parts_s = np.empty((world, nq, k))
            lam = np.empty(nq)
            for r, h in enumerate(shards):
                _lib.check(lib.asp_search_batch_k(h, g1._h, q.ctypes.data, nq, 0.62, k, parts_i[r].ctypes.data,
                                                  parts_s[r].ctypes.data, lam.ctypes.data, None))
            oi, osc = np.empty((nq, k), dtype=np.int64), np.empty((nq, k))
            _lib.check(lib.asp_topk_merge(a1._ctx, parts_i.ctypes.data, parts_s.ctypes.data, world, nq, k, oi.ctypes.data,
                                          osc.ctypes.data))
            i1, s1 = a1.search_batch(q, g1, 0.62, k=k)
            assert np.array_equal(oi, i1) and np.array_equal(osc, s1, equal_nan=True)
        for k, pool in ((50, 0), (20, 0), (40, 100)):
            m = lib.asp_hybrid_pool(n, k, pool)
            pi, pc, ps = np.empty((world, nq, m), dtype=np.int64), np.empty((world, nq, m)), np.empty((world, nq, m))
            lam = np.empty(nq)
            for r, h in enumerate(shards):
                _lib.check(lib.asp_search_hybrid_shard_k(h, g1._h, q.ctypes.data, nq, 0.62, pool, k, pi[r].ctypes.data,
                                                         pc[r].ctypes.data, ps[r].ctypes.data, lam.ctypes.data, None))
            oi, osc = np.empty((nq, k), dtype=np.int64), np.empty((nq, k))
            _lib.check(lib.asp_hybrid_merge(a1._ctx, pi.ctypes.data, pc.ctypes.data, ps.ctypes.data, world, nq, m, k,
                                            oi.ctypes.data, osc.ctypes.data))
            i1, s1 = a1.search_hybrid_batch(q, g1, 0.62, pool=pool or None, k=k)
            assert np.array_equal(oi, i1) and np.array_equal(osc, s1, equal_nan=True)
    finally:
        for h in shards:
            lib.asp_free_space(h)


def _api_worker(rank, world, item_shards, port, out):
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        from arrowspace import ArrowSpaceBuilder
        from pyarrowspace_b200 import api
        from pyarrowspace_b200.distributed import grid_groups, grid_layout
        x, q = _shard_data(3000, 64, 8, 300, 12)
        a1, g1 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 6, "p": 2.0, "sigma": 0.3}, x, device=0)
        r_, c_, r, c = grid_layout(world, rank, item_shards)
        grid = dict(R=r_, C=c_, r=r, c=c, item_group=None, merge_group=None)
        if c_ > 1:
            item_groups, merge_groups = grid_groups(world, r_)
            grid["item_group"], grid["merge_group"] = item_groups[r], merge_groups[c]
        sp = api.ArrowSpace._wrap(_shards(x, r_, a1, only=r)[0], a1._ctx, grid["merge_group"], grid)
        mask = np.random.default_rng(3).random(3000) < 0.5
        same = {}
        for k, pool in ((40, None), (64, None), (100, None), (50, 5000)):
            for allowed in (None, mask):
                hi, hs = sp.search_hybrid_batch(q, g1, 0.62, k=k, pool=pool, allowed=allowed)
                h1, hs1 = a1.search_hybrid_batch(q, g1, 0.62, k=k, pool=pool, allowed=allowed)
                same[(k, pool, allowed is None)] = bool(np.array_equal(hi, h1) and np.array_equal(hs, hs1, equal_nan=True))
        hits = sp.search_hybrid(q[7].copy(), g1, 0.62, k=48)
        same["single"] = [i for i, _ in hits] == [i for i in a1.search_hybrid_batch(q[7:8], g1, 0.62, k=48)[0][0] if i >= 0]
        out.put((rank, same))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        out.put((rank, "error", repr(e)))
        raise


@pytest.mark.parametrize("world,item_shards", [(2, 2), (4, 4), (4, 2)])
def test_public_k_on_item_shards(world, item_shards):
    """search_hybrid_batch(k=) / search_hybrid(k=) on item shards through the product path (CudaEngine, the orchestration,
    asp_search_hybrid_shard_k, gloo, processes sharing cuda:0): every rank returns the one-GPU answer bit for bit, with and
    without a mask, for shortlists and for the whole set (pool 5000: the lists merge with asp_topk_merge at width k).
    search_batch's per-shard lists at width k and their merge are covered on one device above."""
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
    for rank, same in res:
        assert all(same.values()), (rank, same)
