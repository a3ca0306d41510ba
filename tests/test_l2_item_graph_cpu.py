"""The Euclidean item graph (distance="l2" / "l2sq", nodes = items) without a GPU: the C oracle against the independent
numpy one, the raw-accumulator threshold of the tensor-core candidate pass (csrc/l2_bound.cuh, compiled with g++) against
the f32 score it guards, and the multi-rank orchestration over gloo with an l2-aware numpy engine."""
import ctypes as C
import math
import os
import socket
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ragged_items(n, f, seed):
    """Clusters at different scales (norms over two decades), exact duplicates, zero rows."""
    rng = np.random.default_rng(seed)
    centres = rng.normal(size=(4, f)) * np.array([0.05, 0.5, 1.0, 5.0])[:, None]
    lab = rng.integers(0, 4, n)
    x = centres[lab] * (1.0 + 0.2 * rng.normal(size=(n, f)))
    x[n // 2:n // 2 + 5] = x[:5]                                      # exact duplicates: distance 0, ties by index
    x[n - 2:] = 0.0                                                   # zero rows
    return x


def _oracle_np_csr(x, gp, distance):
    from oracle import oracle_np
    W, L, edges = oracle_np.build_graph(x, gp["eps"], gp["k"], gp["p"], gp["sigma"], topk=gp["topk"], distance=distance)
    return L, edges


def _kth_distances(x, k, distance):
    """Distance of every row to its k-th nearest other row (numpy, only to choose eps values that bind on some rows)."""
    nsq = (x * x).sum(1)
    d2 = np.maximum(nsq[:, None] + nsq[None, :] - 2.0 * x @ x.T, 0.0)
    np.fill_diagonal(d2, np.inf)
    d = np.sqrt(d2) if distance == "l2" else d2
    return np.sort(d, axis=1)[:, k - 1]


@pytest.mark.parametrize("distance", ["l2", "l2sq"])
@pytest.mark.parametrize("n,f,k,q", [(37, 5, 4, 0.5), (64, 13, 6, 0.3), (90, 7, 3, 0.7), (9, 3, 8, 0.5)])
def test_oracle_item_graph_equals_numpy(oracle_mod, distance, n, f, k, q):
    """Ragged shapes, duplicates, zero rows, and an eps at a quantile of the k-th-neighbour distance: the radius binds on
    some rows and the cap on the others."""
    x = _ragged_items(n, f, 11 * n + f)
    kth = _kth_distances(x, min(k, n - 1), distance)
    eps = float(np.quantile(kth, q))
    assert (kth > eps).any() and (kth <= eps).any()
    gp = {"eps": eps, "k": k, "topk": 3, "p": 2.0, "sigma": None}
    s, g = oracle_mod.build(gp, x, nodes="items", distance=distance)
    L, edges = _oracle_np_csr(x, dict(gp, sigma=eps * 0.5), distance)
    got = [tuple(int(v) for v in e) for e in g.edges()]
    assert got == sorted(tuple(e) for e in edges)
    ip, ix, dt = g.csr()
    dense = np.zeros((n, n))
    for r in range(n):
        dense[r, ix[ip[r]:ip[r + 1]]] = dt[ip[r]:ip[r + 1]]
    np.testing.assert_allclose(dense, L, rtol=1e-12, atol=1e-300)


# ----------------------------------------------------------------------------- the threshold of the tensor-core pass

@pytest.fixture(scope="module")
def bound():
    import tempfile
    out = os.path.join(tempfile.mkdtemp(prefix="l2b"), "libl2_bound_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "host_emul", "l2_bound_host.cpp")])
    lib = C.CDLL(out)
    lib.l2_score.argtypes = [C.c_float] * 3
    lib.l2_score.restype = C.c_float
    lib.l2_threshold.argtypes = [C.c_float] * 4
    lib.l2_threshold.restype = C.c_float
    return lib


def _f32(v):
    return float(np.float32(v))


def _check_tile(bound, A, lo, hi, theta, bs, accs):
    """No column with B in [lo, hi] whose f32 score reaches theta is rejected by the threshold."""
    thr = bound.l2_threshold(A, lo, hi, theta)
    for B in bs:
        for a in accs:
            sc = bound.l2_score(A, B, a)
            if sc >= theta:
                assert a >= thr, (A, lo, hi, theta, B, a, sc, thr)
    return thr


from hypothesis import HealthCheck, given, settings              # noqa: E402
from hypothesis import strategies as st                           # noqa: E402

PROP = settings(max_examples=400, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])


@PROP
@given(st.floats(-20, 18), st.floats(-8, 8), st.floats(0, 3), st.floats(-1.0, 1.0), st.booleans(), st.sampled_from([0, 1, 2, 3]),
       st.integers(0, 2 ** 31 - 1))
def test_threshold_never_rejects_a_passing_column(bound, log_a, log_ratio, log_width, theta_pos, lo_zero, theta_kind, seed):
    """Random row norm A (1e-20 .. 1e18 in log: the library refuses larger norms on this route), tile intervals from 1e-8 A
    to 1e8 A (extreme ratios, capped at 1e18), lo = 0, thresholds
    around the tile's own scores (A^2 <= D^2 and A^2 > D^2), positive thresholds and exact-zero rows; columns at the interval
    ends, at the analytic minimiser and random inside, with accumulators around the value at which they reach theta."""
    rng = np.random.default_rng(seed)
    A = _f32(10.0 ** log_a) if theta_kind != 3 else 0.0
    lo = _f32(max(A, 1e-20) * 10.0 ** log_ratio)
    hi = _f32(min(lo * 10.0 ** log_width, 1e18))
    if lo > hi:
        return
    if lo_zero:
        lo = 0.0
    # theta: around -(A - B)^2 .. -(A + B)^2 for a B of the tile, or positive (the k-th best of exact duplicates)
    Bm = _f32(lo + (hi - lo) * rng.uniform())
    if theta_kind == 0:
        theta = _f32(-((A - Bm) ** 2 + 2 * A * Bm * (1 - theta_pos)))
    elif theta_kind == 1:
        theta = _f32(-(A * A) * (1.0 + theta_pos))                  # D^2 around A^2
    elif theta_kind == 2:
        theta = _f32(abs(theta_pos) * 1e-3 * (A * A + Bm * Bm))       # > 0
    else:
        theta = _f32(-(Bm * Bm) * (1.0 + 1e-3 * theta_pos))          # zero row: d^2 = B^2
    if not math.isfinite(theta):
        return
    bs = {lo, hi, Bm, _f32(np.nextafter(np.float32(hi), np.float32(0))), _f32(np.nextafter(np.float32(lo), np.float32(np.inf)))}
    e2 = A * A + theta
    if e2 > 0:
        bs.add(_f32(min(max(math.sqrt(e2), lo), hi)))
    bs = [b for b in bs if lo <= b <= hi and math.isfinite(b)]
    accs = set()
    for B in bs:
        if A > 0 and B > 0:
            c0 = (A * A + B * B + theta) / (2 * A * B)               # cos at which the score reaches theta
            for dc in (0.0, 1e-7, -1e-7, 1e-6, -1e-6, 3e-5, -3e-5):
                v = (c0 + dc) * 16384.0
                if abs(v) < 2.0 * 16384.0:
                    a = np.float32(v)
                    for _ in range(3):
                        accs.add(float(a))
                        a = np.nextafter(a, np.float32(-np.inf))
    accs |= {float(np.float32(v)) for v in rng.uniform(-1.05, 1.05, 8) * 16384.0}
    accs.add(0.0)
    _check_tile(bound, A, lo, hi, theta, bs, sorted(accs))


def test_threshold_special_cases(bound):
    inf = float("inf")
    assert bound.l2_threshold(1.0, 0.5, 2.0, -inf) == -inf                    # no threshold yet
    assert bound.l2_threshold(0.0, 3.0, 4.0, -1.0) == inf                     # zero row: d^2 = B^2 >= 9 > 1
    assert bound.l2_threshold(0.0, 0.5, 4.0, -1.0) == -inf                    # ... or some B^2 <= 1: every column
    assert bound.l2_threshold(1.0, 0.0, 2.0, -4.0) == -inf                    # A^2 <= D^2 and lo = 0: no pruning
    assert bound.l2_threshold(5.0, 0.0, 0.0, -1.0) == inf                     # only zero columns, d^2 = 25 > 1
    t = bound.l2_threshold(1.0, 0.9, 1.1, -1e-4)                              # tight tile: cos >= ~1 - 5e-5 needed
    assert 0.999 * 16384 < t < 16384
    assert bound.l2_threshold(1.0, 100.0, 200.0, -1.0) == inf                 # |A - B| > D for the whole tile
    # the pruned case of a tight tile keeps every column whose score passes
    _check_tile(bound, 1.0, 0.9, 1.1, -1e-4, [0.9, 0.95, 1.0, 1.05, 1.1],
                [float(np.float32(16384 * (1 - e))) for e in (0, 1e-6, 1e-5, 4e-5, 5e-5, 6e-5, 1e-4)])


def test_score_zero_rows_and_columns(bound):
    assert bound.l2_score(0.0, 3.0, 0.0) == -9.0
    assert bound.l2_score(2.0, 0.0, 0.0) == -4.0
    assert bound.l2_score(2.0, 2.0, 16384.0) == 0.0                            # cos = 1, same norm: d = 0
    assert bound.l2_score(1.0, 1.0, 0.0) == -2.0                               # orthogonal unit vectors


# ----------------------------------------------------------------------------- gloo orchestration with an l2 engine

class NumpyL2KnnEngine:
    """Stands in for CudaEngine in `sharded_item_graph`: the oracle's Euclidean distance (left-to-right sums,
    d2 = (saa + sbb) - 2 dot clamped at 0, sqrt for l2) and selection rule, numpy symmetrise + weights."""

    def __init__(self, distance):
        import torch
        self.torch = torch
        self.distance = distance

    def full_space(self, x_full):
        return {"x": x_full.numpy().copy()}

    def knn_rows(self, space, cgp, r0, r1, sw=None):
        x = space["x"]
        n, f = x.shape
        kk = min(int(cgp.k), n - 1)

        def seq(a, b):
            s = 0.0
            for u, v in zip(a, b):
                s += u * v
            return s
        nsq = [seq(x[i], x[i]) for i in range(n)]
        idx = np.full((r1 - r0, kk), -1, dtype=np.int32)
        dst = np.zeros((r1 - r0, kk))
        cnt = np.zeros(r1 - r0, dtype=np.int32)
        for i in range(r0, r1):
            cand = []
            for j in range(n):
                if j == i:
                    continue
                d2 = max(0.0, (nsq[i] + nsq[j]) - 2.0 * seq(x[i], x[j]))
                d = math.sqrt(d2) if self.distance == "l2" else d2
                if d <= cgp.eps:
                    cand.append((d, j))
            cand.sort()
            for e, (dj, j) in enumerate(cand[:kk]):
                idx[i - r0, e], dst[i - r0, e] = j, dj
            cnt[i - r0] = min(len(cand), kk)
        t = self.torch
        return t.from_numpy(idx), t.from_numpy(dst), t.from_numpy(cnt)

    def graph_from_knn(self, n, idx, dist, cnt, cgp, sw):
        idx, dist, cnt = idx.numpy(), dist.numpy(), cnt.numpy()
        sigma = cgp.sigma if cgp.has_sigma else cgp.eps * 0.5
        w = np.zeros((n, n))
        for i in range(n):
            for e in range(cnt[i]):
                j = idx[i, e]
                wij = 1.0 / (1.0 + (dist[i, e] / sigma) ** cgp.p)
                w[i, j] = max(w[i, j], wij)
                w[j, i] = max(w[j, i], wij)
        return {"edges": sorted((i, j) for i in range(n) for j in range(i + 1, n) if w[i, j] > 0)}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


N_G, F_G, K_G = 150, 6, 4


def _gloo_items():
    return _ragged_items(N_G, F_G, 2024)


def _gloo_eps(distance):
    return float(np.quantile(_kth_distances(_gloo_items(), K_G, distance), 0.5))


def _l2_worker(rank, world, port, distance, q):
    import torch
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        from pyarrowspace_b200 import _lib
        from pyarrowspace_b200.distributed import sharded_item_graph
        cuts = [0] + [int(N_G * (r + 1) / world) + (2 if r % 2 == 0 and r + 1 < world else 0) for r in range(world)]
        cuts[-1] = N_G
        r0, r1 = cuts[rank], cuts[rank + 1]
        shard = torch.from_numpy(_gloo_items()[r0:r1].copy())
        cgp = _lib.make_params(_gloo_eps(distance), K_G, 3, 2.0, None)
        sw = _lib.make_switches(distance=distance)
        space, graph = sharded_item_graph(NumpyL2KnnEngine(distance), shard, N_G, r0, cgp, sw, None)
        q.put((rank, graph["edges"], space["x"].shape))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        q.put((rank, "error", repr(e)))
        raise


@pytest.mark.parametrize("distance", ["l2", "l2sq"])
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_l2_item_graph_over_gloo(world, distance, oracle_mod):
    """Ragged item shards, halo all-gather and the all-gather of the per-rank Euclidean neighbour lists reproduce the
    single-process oracle's item graph on every rank."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_l2_worker, args=(r, world, port, distance, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[1] != "error" for r in res), res
    x = _gloo_items()
    s, g = oracle_mod.build({"eps": _gloo_eps(distance), "k": K_G, "topk": 3, "p": 2.0, "sigma": None}, x, nodes="items",
                            distance=distance)
    want = [tuple(int(v) for v in e) for e in g.edges()]
    assert len(want) > 0
    for r in res:
        assert r[2] == (N_G, F_G)
        assert [tuple(e) for e in r[1]] == want
