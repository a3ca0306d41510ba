"""Range search on the GPU: indices identical to the definition over the oracle (test_range_search_cpu.want_range: every
item whose oracle score is >= min_score, (score desc, index asc)) and scores within RTOL, on every route (tcgen05 batch,
tcgen05 small batch on a large shard, mean-zero data, forced emission overflow into the scan, tau = 0.001 and tau = 0 on the
scan), at thresholds giving about 0, 1, 10 and 1000 hits per query, with masks, on emulated item shards and through the
product orchestration over gloo.  Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

from test_range_search_cpu import want_range

pytestmark = pytest.mark.gpu

RTOL = 1e-9          # the oracle's f64 outputs (its lambdas differ from the GPU's in the last bits), as in test_gpu_parity


def _data(n, f, seed, nq, dup=0):
    rng = np.random.default_rng(seed)
    cent = rng.normal(size=(16, f))
    x = np.abs(cent[rng.integers(0, 16, n)] + 0.25 * rng.normal(size=(n, f))) + 0.05
    if dup:
        x[n - dup:] = x[:dup]                                 # exact duplicates: ties, resolved by index
    q = x[rng.integers(0, n, nq)] * 1.02 + 0.01 * rng.normal(size=(nq, f))
    if dup:
        q[:3] = x[:3] * 1.5
    return np.ascontiguousarray(x), np.ascontiguousarray(q)


_BUILT = {}


def _spaces(oracle_mod, n, f, seed, nq, kind="plain", dup=0):
    key = (n, f, seed, nq, kind, dup)
    if key not in _BUILT:
        from arrowspace import ArrowSpaceBuilder
        _BUILT.clear()
        gp, sw = {"eps": 0.6, "k": 5, "topk": 10, "p": 2.0, "sigma": 0.3}, {}
        if kind == "mean_zero":                               # synth's mean-zero regime: the wide one-term band
            from pyarrowspace_b200 import synth
            x = synth.make_items(n, f, 21, 100.0, n_clusters=8, shift=0.0)
            q = synth.make_fresh_queries(f, nq, 121, n_clusters=8)[0]
            gp, sw = {"eps": 0.5, "k": 6, "topk": 10, "p": 2.0, "sigma": 0.25}, {"tau_mode": "median_abs"}
        else:
            x, q = _data(n, f, seed, nq, dup)
        a1, g1 = ArrowSpaceBuilder.build(gp, x, **sw)
        s, g = oracle_mod.build(gp, x, **sw)
        _BUILT[key] = (x, q, a1, g1, s, g)
    return _BUILT[key]


def _oracle_scores(s, g, q, tau):
    lq = s.search_batch(q, g, tau)[2]
    return lq, np.stack([s.scores(q[i], lq[i], tau) for i in range(len(q))])


def _threshold(scores, level):
    """A min_score giving about `level` hits per query: midway between the level-th and the next best score of the median
    query (a midpoint, so that no score sits on the threshold up to the last bits the GPU's lambdas may differ in)."""
    if level == 0:
        return float(np.nextafter(scores.max(), np.inf)) + 1e-9
    srt = -np.sort(-scores, axis=1)
    k = min(level, scores.shape[1] - 1)
    a, b = np.median(srt[:, k - 1]), np.median(srt[:, k])
    return float(0.5 * (a + b)) if a != b else float(a)


def _want(s, q, lq, tau, thr, mask=None):
    rows = [want_range(s, q[i], lq[i], tau, thr, mask) for i in range(len(q))]
    indptr = np.concatenate([[0], np.cumsum([len(r[0]) for r in rows])]).astype(np.int64)
    return indptr, np.concatenate([r[0] for r in rows]), np.concatenate([r[1] for r in rows])


def _same(got, want, rtol=RTOL):
    gp, gi, gs = got
    wp, wi, ws = want
    assert np.array_equal(gp, wp), "counts differ at queries %s" % np.nonzero(np.diff(gp) != np.diff(wp))[0][:10]
    assert np.array_equal(gi, wi)
    np.testing.assert_allclose(gs, ws, rtol=rtol, atol=0)


def _mask(n, density, seed):
    rng = np.random.default_rng(seed)
    if density == "none":
        return np.zeros(n, dtype=bool)
    if density == "one":
        m = np.zeros(n, dtype=bool)
        m[int(rng.integers(0, n))] = True
        return m
    return rng.random(n) < float(density)


# (n, f, nq, tau, kind, dup, env)
ROUTES = {
    "tc_batch": (20000, 64, 300, 0.62, "plain", 0, {}),
    "tc_small_large_shard": (140000, 32, 5, 0.62, "plain", 0, {}),
    "tc_mean_zero": (20000, 96, 300, 0.62, "mean_zero", 0, {}),
    "tc_overflow_to_scan": (3000, 24, 40, 0.62, "plain", 300, {"ASP_TC_CAPB": "8"}),
    "scan_tau_0p001": (6000, 48, 70, 0.001, "plain", 0, {}),
    "scan_tau_0": (6000, 48, 70, 0.0, "plain", 0, {}),
}
LEVELS = [0, 1, 10, 1000]


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_range_equals_definition(oracle_mod, monkeypatch, route, level):
    from pyarrowspace_b200 import stat
    n, f, nq, tau, kind, dup, env = ROUTES[route]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    lq, scores = _oracle_scores(s, g, q, tau)
    thr = _threshold(scores, level)
    got = a1.search_range_batch(q, g1, tau, thr)
    _same(got, _want(s, q, lq, tau, thr))
    is_tc = stat("range_stage1_is_tc")
    assert is_tc == (1.0 if route.startswith("tc") else 0.0)
    if route == "tc_overflow_to_scan" and level >= 10:
        assert stat("search_slow_queries") > 0


@pytest.mark.parametrize("route", ["tc_batch", "tc_mean_zero", "tc_overflow_to_scan"])
def test_scan_route_is_bit_identical(oracle_mod, monkeypatch, route):
    """ASP_RANGE_STAGE1=scan against the tensor-core route: the same hits, the same bits."""
    n, f, nq, tau, kind, dup, env = ROUTES[route]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    _, scores = _oracle_scores(s, g, q[:20], tau)
    mask = _mask(n, "0.5", 3)
    for level in (1, 10, 1000):
        thr = _threshold(scores, level)
        for allowed in (None, mask):
            monkeypatch.delenv("ASP_RANGE_STAGE1", raising=False)
            tc = a1.search_range_batch(q, g1, tau, thr, allowed=allowed)
            monkeypatch.setenv("ASP_RANGE_STAGE1", "scan")
            sc = a1.search_range_batch(q, g1, tau, thr, allowed=allowed)
            assert all(np.array_equal(u, v) for u, v in zip(tc, sc))


@pytest.mark.parametrize("density", ["1.0", "0.5", "0.01", "one", "none"])
@pytest.mark.parametrize("route", ["tc_batch", "scan_tau_0"])
def test_masks(oracle_mod, route, density):
    n, f, nq, tau, kind, dup, _ = ROUTES[route]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    lq, scores = _oracle_scores(s, g, q, tau)
    thr = _threshold(scores, 1000)
    mask = _mask(n, density, 7)
    _same(a1.search_range_batch(q, g1, tau, thr, allowed=mask), _want(s, q, lq, tau, thr, mask))


def test_thresholds_at_the_edges(oracle_mod):
    """Inclusive at an item's exact score; -inf returns every item; > 1 returns empty rows; a segment longer than one CTA's
    sort (8192) and one that needs several merge passes."""
    from arrowspace import ArrowSpaceBuilder
    n, f, nq, tau, kind, dup, _ = ROUTES["tc_batch"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    idx, sc = a1.search_batch(q, g1, tau)
    for qi in (0, 5, 77):                                     # min_score = the GPU's own score of the 10th hit: included
        indptr, ri, rs = a1.search_range_batch(q[qi:qi + 1], g1, tau, sc[qi, -1])
        assert indptr[1] >= 10 and ri[9] == idx[qi, 9] and rs[9] == sc[qi, -1]
        assert np.array_equal(ri[:10], idx[qi]) and np.array_equal(rs[:10], sc[qi])
    lq, scores = _oracle_scores(s, g, q[:4], tau)
    thr = float(np.median(np.quantile(scores, 0.3, axis=1)))  # ~14000 hits per query: the long-segment sort
    got = a1.search_range_batch(q[:4], g1, tau, thr)
    assert np.diff(got[0]).min() > 8192
    _same(got, _want(s, q[:4], lq, tau, thr))
    for big in (1.0000001, 2.0, 1e300, float("inf")):
        indptr, ri, rs = a1.search_range_batch(q, g1, tau, big)
        assert indptr.tolist() == [0] * (nq + 1) and len(ri) == 0 and len(rs) == 0
    xs, qs = _data(500, 16, 3, 6)
    a2, g2 = ArrowSpaceBuilder.build({"eps": 0.6, "k": 5, "topk": 4, "p": 2.0, "sigma": 0.3}, xs)
    s2, gg2 = oracle_mod.build({"eps": 0.6, "k": 5, "topk": 4, "p": 2.0, "sigma": 0.3}, xs)
    lq2 = s2.search_batch(qs, gg2, 0.62)[2]
    _same(a2.search_range_batch(qs, g2, 0.62, float("-inf")), _want(s2, qs, lq2, 0.62, float("-inf")))
    # several merge passes: every item of a 140k shard
    n, f, nq, tau, kind, dup, _ = ROUTES["tc_small_large_shard"]
    x, q, a3, g3, s3, gg3 = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    lq3 = s3.search_batch(q[:2], gg3, tau)[2]
    got = a3.search_range_batch(q[:2], g3, tau, float("-inf"))
    assert np.diff(got[0]).tolist() == [n, n]
    _same(got, _want(s3, q[:2], lq3, tau, float("-inf")))


def test_cross_check_with_search_batch(oracle_mod):
    """Where search_batch's k-th score clears min_score, its row equals the range row's first k entries bit for bit."""
    n, f, nq, tau, kind, dup, _ = ROUTES["tc_batch"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    idx, sc = a1.search_batch(q, g1, tau)
    thr = float(np.median(sc[:, -1]))
    indptr, ri, rs = a1.search_range_batch(q, g1, tau, thr)
    checked = 0
    for qi in range(nq):
        if sc[qi, -1] >= thr:
            a = indptr[qi]
            assert np.array_equal(ri[a:a + 10], idx[qi]) and np.array_equal(rs[a:a + 10], sc[qi])
            checked += 1
    assert checked >= nq // 3


def test_device_batch_single_query_and_errors(oracle_mod):
    import torch
    from arrowspace import ArrowSpaceBuilder, PanicException
    n, f, nq, tau, kind, dup, _ = ROUTES["tc_batch"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    _, scores = _oracle_scores(s, g, q[:10], tau)
    thr = _threshold(scores, 10)
    host = a1.search_range_batch(q, g1, tau, thr)
    dev = a1.search_range_batch(torch.from_numpy(q).cuda(), g1, tau, thr)
    assert all(t.is_cuda for t in dev)
    assert all(np.array_equal(h, t.cpu().numpy()) for h, t in zip(host, dev))
    one = a1.search_range(q[4].copy(), g1, tau, thr)
    a, b = host[0][4], host[0][5]
    assert [i for i, _ in one] == host[1][a:b].tolist() and [v for _, v in one] == host[2][a:b].tolist()
    total = int(host[0][-1])
    with pytest.raises(ValueError, match="max_hits = %d" % (total - 1)):
        a1.search_range_batch(q, g1, tau, thr, max_results=total - 1)
    assert a1.search_range_batch(q, g1, tau, thr, max_results=total)[0][-1] == total
    with pytest.raises(ValueError):
        a1.search_range_batch(q, g1, tau, float("nan"))
    qz = q.copy()
    qz[3] = 0.0
    with pytest.raises(PanicException):
        a1.search_range_batch(qz, g1, tau, thr)
    xs = np.abs(np.random.default_rng(2).normal(size=(50, 6))) + 0.1
    a0, g0 = ArrowSpaceBuilder.build({"eps": 1.0, "k": 0, "topk": 2, "p": 2.0}, xs)      # no edges: every lambda is 0
    with pytest.raises(PanicException, match="The lambdas are zero"):
        a0.search_range(xs[0].copy(), g0, 0.5, 0.1)


def _shards(x, world, a1, only=None):
    """Row shards of `world` (or only shard `only`) on cuda:0 with the one-GPU space's lambdas and norms."""
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


@pytest.mark.parametrize("world", [2, 4, 8])
def test_emulated_item_shards_equal_one_gpu(oracle_mod, world):
    """Each row shard's asp_search_range_batch (its slice of the mask) merged with asp_range_merge: bitwise the one-GPU
    answer, with and without a mask."""
    from pyarrowspace_b200 import _lib
    from pyarrowspace_b200.distributed import pack_allowed
    lib = _lib.load()
    n, f, nq, tau, kind, dup, _ = ROUTES["tc_batch"]
    x, q, a1, g1, s, g = _spaces(oracle_mod, n, f, 11 + n + f, nq, kind, dup)
    _, scores = _oracle_scores(s, g, q[:20], tau)
    shards = _shards(x, world, a1)
    try:
        for level, allowed in ((10, None), (1000, _mask(n, "0.5", 9))):
            thr = _threshold(scores, level)
            want = a1.search_range_batch(q, g1, tau, thr, allowed=allowed)
            counts, idx, sc = [], [], []
            for h in shards:
                n_local, row0 = C.c_int64(), C.c_int64()
                _lib.check(lib.asp_space_dims(h, C.byref(n_local), C.byref(C.c_int32()), C.byref(row0), C.byref(C.c_int64())))
                bits = None if allowed is None else pack_allowed(allowed, row0.value, n_local.value)
                cnt, lam, res = np.empty(nq, np.int64), np.empty(nq), C.c_void_p()
                _lib.check(lib.asp_search_range_batch(h, g1._h, q.ctypes.data, nq, tau, thr,
                                                      None if bits is None else bits.ctypes.data, 0, cnt.ctypes.data,
                                                      lam.ctypes.data, C.byref(res)))
                ii, ss = np.empty(int(cnt.sum()), np.int64), np.empty(int(cnt.sum()))
                _lib.check(lib.asp_range_result_fetch(res, ii.ctypes.data, ss.ctypes.data))
                lib.asp_range_result_free(res)
                counts.append(cnt), idx.append(ii), sc.append(ss)
            counts = np.ascontiguousarray(np.stack(counts))
            ii, ss = np.concatenate(idx), np.concatenate(sc)
            oi, os_ = np.empty_like(ii), np.empty_like(ss)
            _lib.check(lib.asp_range_merge(a1._ctx, world, nq, counts.ctypes.data, ii.ctypes.data, ss.ctypes.data,
                                           oi.ctypes.data, os_.ctypes.data))
            assert np.array_equal(np.concatenate([[0], np.cumsum(counts.sum(axis=0))]), want[0])
            assert np.array_equal(oi, want[1]) and np.array_equal(os_, want[2])
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
        mask = np.random.default_rng(4).random(3000) < 0.5
        for thr, allowed in ((0.9, None), (0.8, mask), (5.0, None)):
            got = sp.search_range_batch(q, g1, 0.62, thr, allowed=allowed)
            want = a1.search_range_batch(q, g1, 0.62, thr, allowed=allowed)
            same[(thr, allowed is None)] = all(np.array_equal(u, v) for u, v in zip(got, want))
        hits = sp.search_range(q[7].copy(), g1, 0.62, 0.9)
        same["single"] = hits == a1.search_range(q[7].copy(), g1, 0.62, 0.9)
        total = int(a1.search_range_batch(q, g1, 0.62, 0.9)[0][-1])
        try:
            sp.search_range_batch(q, g1, 0.62, 0.9, max_results=total - 1)
            limit = None
        except ValueError:
            limit = "ValueError"
        qz = q.copy()
        qz[-1] = 0.0
        try:
            sp.search_range_batch(qz, g1, 0.62, 0.9)
            raised = None
        except PanicException:
            raised = "PanicException"
        out.put((rank, same, (limit, raised)))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        out.put((rank, "error", repr(e)))
        raise


def test_public_search_range_on_item_shards():
    """ArrowSpace.search_range_batch / search_range through the product path (CudaEngine, the orchestration, the C ABI):
    2 processes share cuda:0 over gloo, item_shards = 2.  Every rank returns the one-GPU answer bit for bit, the cap raises
    ValueError and a zero query PanicException on every rank."""
    import socket
    import torch.multiprocessing as mp
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    world = 2
    procs = [ctx.Process(target=_api_worker, args=(r, world, 2, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[1] != "error" for r in res), res
    for rank, same, raised in res:
        assert all(same.values()), (rank, same)
        assert raised == ("ValueError", "PanicException"), rank
