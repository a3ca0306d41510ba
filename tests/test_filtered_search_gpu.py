"""Filtered search (allowed=) on the GPU: indices identical to the definition over the oracle (test_filtered_search_cpu:
the oracle's scores of the allowed items, ranked and cut) and scores equal on every candidate route (tcgen05 batch, tcgen05 small batch on a large shard, the three-term retry, FP64 DMMA, GEMV,
the exact scan), at mask densities 1.0, 0.5, 0.01, one item and none.  Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

from test_filtered_search_cpu import want_hybrid, want_search

pytestmark = pytest.mark.gpu

DENSITIES = ["1.0", "0.5", "0.01", "one", "none"]


def _data(n, f, seed, nq, shift=True, dup=0):
    rng = np.random.default_rng(seed)
    cent = rng.normal(size=(16, f))
    x = cent[rng.integers(0, 16, n)] + 0.25 * rng.normal(size=(n, f))
    if shift:
        x = np.abs(x) + 0.05
    if dup:
        x[n - dup:] = x[:dup]                                 # exact duplicates: ties across the mask
    q = x[rng.integers(0, n, nq)] * 1.02 + 0.01 * rng.normal(size=(nq, f))
    if dup:
        q[:3] = x[:3] * 1.5
    return np.ascontiguousarray(x), np.ascontiguousarray(q)


def _mask(n, density, seed):
    rng = np.random.default_rng(seed)
    if density == "none":
        return np.zeros(n, dtype=bool)
    if density == "one":
        m = np.zeros(n, dtype=bool)
        m[int(rng.integers(0, n))] = True
        return m
    return rng.random(n) < float(density)


RTOL = 1e-9          # the oracle's f64 outputs (its lambdas differ from the GPU's in the last bits), as in test_gpu_parity


def _same(idx, sc, oidx, osc, rtol=0.0):
    """Indices identical, padding where the reference pads, scores equal (bitwise when rtol = 0)."""
    assert np.array_equal(idx, oidx), "rows %s" % np.where((idx != oidx).any(axis=1))[0][:10]
    ok = oidx >= 0
    assert np.isnan(sc[~ok]).all()
    if rtol:
        np.testing.assert_allclose(sc[ok], osc[ok], rtol=rtol, atol=0)
    else:
        assert np.array_equal(sc[ok], osc[ok])


_BUILT = {}


def _spaces(oracle_mod, n, f, topk, seed, nq, shift=True, dup=0):
    key = (n, f, topk, seed, nq, shift, dup)
    if key not in _BUILT:
        from arrowspace import ArrowSpaceBuilder
        _BUILT.clear()
        gp, sw = {"eps": 0.6, "k": 5, "topk": topk, "p": 2.0, "sigma": 0.3}, {}
        if shift == "mean_zero":                              # synth's mean-zero regime: the wide one-term band, the retry
            from pyarrowspace_b200 import synth
            x = synth.make_items(n, f, 21, 100.0, n_clusters=8, shift=0.0)
            q = synth.make_fresh_queries(f, nq, 121, n_clusters=8)[0]
            gp, sw = {"eps": 0.5, "k": 6, "topk": topk, "p": 2.0, "sigma": 0.25}, {"tau_mode": "median_abs"}
        else:
            x, q = _data(n, f, seed, nq, shift, dup)
        a1, g1 = ArrowSpaceBuilder.build(gp, x, **sw)
        s, g = oracle_mod.build(gp, x, **sw)
        _BUILT[key] = (x, q, a1, g1, s, g)
    return _BUILT[key]


# (route, n, f, topk, nq, tau, shift, dup, env)
ROUTES = {
    "tc_batch": (20000, 64, 10, 300, 0.62, True, 0, {}),
    "tc_small_large_shard": (140000, 32, 10, 5, 0.62, True, 0, {}),
    "tc_retry_mean_zero": (20000, 96, 10, 600, 0.62, "mean_zero", 0, {"ASP_SEARCH_STAGE1": "tc"}),
    "fp64_forced": (8000, 48, 10, 300, 0.62, True, 0, {"ASP_SEARCH_STAGE1": "fp64"}),
    "fp64_small_tau": (8000, 48, 10, 300, 0.001, True, 0, {}),
    "gemv": (5000, 40, 10, 5, 0.62, True, 0, {}),
    "exact_scan": (6000, 48, 40, 70, 0.62, True, 0, {}),
    "exact_scan_ties": (3000, 24, 12, 40, 0.62, True, 300, {"ASP_SEARCH_STAGE1": "tc", "ASP_TC_CAPB": "8"}),
}


@pytest.mark.parametrize("density", DENSITIES)
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_filtered_search_equals_oracle(oracle_mod, monkeypatch, route, density):
    n, f, topk, nq, tau, shift, dup, env = ROUTES[route]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    mask = _mask(n, density, 5 + len(route))
    if dup:
        mask[:dup // 2] = False                               # one copy of a duplicate masked, the other not
        mask[n - dup:n - dup // 2] = True
    idx, sc = a1.search_batch(q, g1, tau, allowed=mask)
    oidx, osc = want_search(s, q, s.search_batch(q, g, tau)[2], tau, mask, topk)
    _same(idx, sc, oidx, osc, RTOL)
    assert (oidx >= 0).sum(axis=1).tolist() == [min(topk, int(mask.sum()))] * nq


@pytest.mark.parametrize("route", ["tc_batch", "gemv", "fp64_forced", "tc_small_large_shard"])
def test_adversarial_mask_removes_the_unfiltered_answers(oracle_mod, monkeypatch, route):
    """Every item the unfiltered search returns for the batch is masked out, so every answer lies beyond the unfiltered
    lists.  A threshold raised by a masked item would drop true answers here."""
    n, f, topk, nq, tau, shift, dup, env = ROUTES[route]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    base, _ = a1.search_batch(q, g1, tau)
    mask = np.ones(n, dtype=bool)
    mask[base[base >= 0]] = False
    idx, sc = a1.search_batch(q, g1, tau, allowed=mask)
    oidx, osc = want_search(s, q, s.search_batch(q, g, tau)[2], tau, mask, topk)
    _same(idx, sc, oidx, osc, RTOL)
    assert not np.isin(idx, base[base >= 0]).any()


def test_all_true_is_bit_identical_to_none_and_launches(oracle_mod):
    from pyarrowspace_b200.api import launch_count
    n, f, topk, nq, tau, shift, dup, _ = ROUTES["tc_batch"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    a1.search_batch(q, g1, tau)                                # the operand cache exists before counting
    c0 = launch_count()
    i0, s0 = a1.search_batch(q, g1, tau)
    c1 = launch_count()
    i1, s1 = a1.search_batch(q, g1, tau)
    c2 = launch_count()
    it, st = a1.search_batch(q, g1, tau, allowed=np.ones(n, dtype=bool))
    c3 = launch_count()
    assert c1 - c0 == c2 - c1                                  # allowed=None: the same launches every call
    assert c3 - c2 == (c2 - c1) + 1                            # all-true: the same kernels + the visiting-order mask
    assert np.array_equal(i0, it) and np.array_equal(s0, st, equal_nan=True)
    assert np.array_equal(i0, i1) and np.array_equal(s0, s1, equal_nan=True)


def test_device_batch_out_and_one_query(oracle_mod):
    import torch
    n, f, topk, nq, tau, shift, dup, _ = ROUTES["tc_batch"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    mask = _mask(n, "0.5", 3)
    oidx, osc = want_search(s, q, s.search_batch(q, g, tau)[2], tau, mask, topk)
    di, ds = a1.search_batch(torch.from_numpy(q).cuda(), g1, tau, allowed=mask)
    assert di.is_cuda
    _same(di.cpu().numpy(), ds.cpu().numpy(), oidx, osc, RTOL)
    out = (np.empty((nq, topk), dtype=np.int64), np.empty((nq, topk)))
    ri, rs = a1.search_batch(q, g1, tau, out=out, allowed=mask)
    assert ri is out[0] and rs is out[1]
    _same(ri, rs, oidx, osc, RTOL)
    one_i, one_s = a1.search_batch(q[:1], g1, tau, allowed=mask)
    _same(one_i, one_s, oidx[:1], osc[:1], RTOL)
    none_i, none_s = a1.search_batch(q[:1], g1, tau, allowed=np.zeros(n, dtype=bool))
    assert (none_i == -1).all() and np.isnan(none_s).all()


def test_pipelined_host_batch_equals_single_shot(oracle_mod, monkeypatch):
    from arrowspace import ArrowSpaceBuilder
    x, _ = _data(20000, 32, 9, 1)
    rng = np.random.default_rng(2)
    q = x[rng.integers(0, 20000, 40000)] * 1.01 + 0.01 * rng.normal(size=(40000, 32))
    a1, g1 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 10, "p": 2.0, "sigma": 0.3}, x)
    mask = _mask(20000, "0.5", 4)
    pi, ps = a1.search_batch(q, g1, 0.62, allowed=mask)
    monkeypatch.setenv("ASP_NO_PIPELINE", "1")
    si, ss = a1.search_batch(q, g1, 0.62, allowed=mask)
    assert np.array_equal(pi, si) and np.array_equal(ps, ss, equal_nan=True)
    assert not np.isin(pi[pi >= 0], np.where(~mask)[0]).any()


def test_c4_sample_one_percent(oracle_mod):
    """C4 (1M x 384) at 1 % density against the oracle on 64 queries."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200 import synth
    cfg = synth.config("C4")
    x = synth.make_items(cfg["n"], cfg["f"], cfg["seed"], scale=cfg["scale"])
    q = synth.make_queries(x, 64, 2, scale=cfg["scale"])[0]
    a1, g1 = ArrowSpaceBuilder.build(cfg["graph_params"], x)
    s, g = oracle_mod.build(cfg["graph_params"], x)
    mask = _mask(x.shape[0], "0.01", 6)
    idx, sc = a1.search_batch(q, g1, cfg["tau"], allowed=mask)
    oidx, osc = want_search(s, q, s.search_batch(q, g, cfg["tau"])[2], cfg["tau"], mask, cfg["graph_params"]["topk"])
    _same(idx, sc, oidx, osc, RTOL)


# ---------------------------------------------------------------------------------------------------------- hybrid

@pytest.mark.parametrize("density", ["0.5", "0.01", "one", "none"])
@pytest.mark.parametrize("pool", [0, 40, 1024, 100000])
def test_filtered_hybrid_one_gpu(oracle_mod, pool, density):
    n, f, topk, nq = 6000, 48, 8, 300
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 77, nq)
    mask = _mask(n, density, 8)
    i1, s1 = a1.search_hybrid_batch(q, g1, 0.62, pool=pool or None, allowed=mask)
    oi, os_ = want_hybrid(s, q, s.search_hybrid_batch(q, g, 0.62, pool)[2], 0.62, pool, mask, topk)
    assert np.array_equal(i1, oi)
    ok = oi >= 0
    np.testing.assert_allclose(s1[ok], os_[ok], rtol=1e-9, atol=0)
    assert np.isnan(s1[~ok]).all()
    hits = a1.search_hybrid(q[1].copy(), g1, 0.62, pool=pool or None, allowed=mask)
    assert [i for i, _ in hits] == [int(i) for i in i1[1] if i >= 0]


@pytest.mark.parametrize("pool", [0, 40, 1024, 100000])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_filtered_hybrid_and_search_on_emulated_shards(oracle_mod, world, pool):
    """R row shards on one device, each given its slice of the mask (one shard has no allowed row): the merged filtered
    shard lists equal the one-GPU filtered hybrid search bit for bit, and the merged filtered searches (asp_topk_merge)
    equal the one-GPU filtered search."""
    from test_hybrid_sharded_gpu import _shards
    from pyarrowspace_b200 import _lib, shard_rows
    from pyarrowspace_b200.distributed import pack_allowed
    lib = _lib.load()
    n, f, topk, nq = 5000, 48, 6, 260
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 91, nq)
    mask = _mask(n, "0.5", 12)
    r0, r1 = shard_rows(n, world, world - 1)
    mask[r0:r1] = False
    shards = _shards(x, world, a1)
    ctx = _lib.context()
    try:
        m = lib.asp_hybrid_pool(n, topk, pool)
        whole = m >= n
        width = topk if whole else m
        idx = np.empty((world, nq, width), dtype=np.int64)
        cos = np.empty((world, nq, width))
        sc = np.empty((world, nq, width))
        sidx = np.empty((world, nq, topk), dtype=np.int64)
        ssc = np.empty((world, nq, topk))
        for r, h in enumerate(shards):
            a, b = shard_rows(n, world, r)
            bits = pack_allowed(mask, a, b - a)
            _lib.check(lib.asp_search_hybrid_shard_filtered(h, g1._h, q.ctypes.data, nq, 0.62, pool, idx[r].ctypes.data,
                                                            None if whole else cos[r].ctypes.data, sc[r].ctypes.data, None,
                                                            bits.ctypes.data))
            _lib.check(lib.asp_search_batch_filtered(h, g1._h, q.ctypes.data, nq, 0.62, sidx[r].ctypes.data,
                                                     ssc[r].ctypes.data, None, bits.ctypes.data))
        out_idx = np.empty((nq, topk), dtype=np.int64)
        out_sc = np.empty((nq, topk))
        if whole:
            _lib.check(lib.asp_topk_merge(ctx, idx.ctypes.data, sc.ctypes.data, world, nq, topk, out_idx.ctypes.data,
                                          out_sc.ctypes.data))
        else:
            _lib.check(lib.asp_hybrid_merge(ctx, idx.ctypes.data, cos.ctypes.data, sc.ctypes.data, world, nq, m, topk,
                                            out_idx.ctypes.data, out_sc.ctypes.data))
        i1, s1 = a1.search_hybrid_batch(q, g1, 0.62, pool=pool or None, allowed=mask)
        _same(out_idx, out_sc, i1, s1)
        mi = np.empty((nq, topk), dtype=np.int64)
        ms = np.empty((nq, topk))
        _lib.check(lib.asp_topk_merge(ctx, sidx.ctypes.data, ssc.ctypes.data, world, nq, topk, mi.ctypes.data, ms.ctypes.data))
        bi, bs = a1.search_batch(q, g1, 0.62, allowed=mask)
        _same(mi, ms, bi, bs)
    finally:
        for h in shards:
            lib.asp_free_space(h)


def _api_worker(rank, world, item_shards, port, out):
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        from arrowspace import ArrowSpaceBuilder
        from pyarrowspace_b200 import api, shard_rows
        from pyarrowspace_b200.distributed import grid_groups, grid_layout
        from test_hybrid_sharded_gpu import _shards
        x, q = _data(3000, 64, 8, 300)
        a1, g1 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 6, "p": 2.0, "sigma": 0.3}, x, device=0)
        r_, c_, r, c = grid_layout(world, rank, item_shards)
        grid = dict(R=r_, C=c_, r=r, c=c, item_group=None, merge_group=None)
        if c_ > 1:
            item_groups, merge_groups = grid_groups(world, r_)
            grid["item_group"], grid["merge_group"] = item_groups[r], merge_groups[c]
        sp = api.ArrowSpace._wrap(_shards(x, r_, a1, only=r)[0], a1._ctx, grid["merge_group"], grid)
        mask = _mask(3000, "0.5", 21)
        a, b = shard_rows(3000, r_, 0)
        mask[a:b] = False                                     # item shard 0 has no allowed row
        same = {}
        for pool in (None, 40, 5000):
            hi, hs = sp.search_hybrid_batch(q, g1, 0.62, pool=pool, allowed=mask)
            i1, s1 = a1.search_hybrid_batch(q, g1, 0.62, pool=pool, allowed=mask)
            same[pool] = bool(np.array_equal(hi, i1) and np.array_equal(hs, s1, equal_nan=True))
        try:
            sp.search_hybrid_batch(q, g1, 0.62, allowed=mask[:-1])
            raised = None
        except ValueError:
            raised = "ValueError"
        out.put((rank, same, raised))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        out.put((rank, "error", repr(e)))
        raise


@pytest.mark.parametrize("world,item_shards", [(2, 2), (4, 4), (4, 2)])
def test_public_filtered_hybrid_on_item_shards(world, item_shards):
    """search_hybrid_batch(allowed=) through the product path with `world` processes sharing cuda:0 over gloo: every rank
    returns the one-GPU filtered answer, and a wrong mask raises ValueError on every rank before any collective."""
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
        assert raised == "ValueError", rank


def test_argument_errors(oracle_mod):
    import torch
    n, f, topk, nq, tau, shift, dup, _ = ROUTES["gemv"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, topk, 11 + n + f, nq, shift, dup)
    for bad, exc in ((np.ones(n, dtype=np.uint8), TypeError), (np.ones(n), TypeError), ([True] * n, TypeError),
                     (torch.ones(n, dtype=torch.bool), TypeError), (np.ones(n - 1, dtype=bool), ValueError),
                     (np.ones((1, n), dtype=bool), ValueError)):
        with pytest.raises(exc):
            a1.search_batch(q, g1, tau, allowed=bad)
        with pytest.raises(exc):
            a1.search_hybrid(q[0].copy(), g1, tau, allowed=bad)
        with pytest.raises(exc):
            a1.search_hybrid_batch(q, g1, tau, allowed=bad)
