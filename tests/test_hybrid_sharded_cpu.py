"""search_hybrid on item-sharded spaces without a GPU.

- The cross-shard merge of csrc/hybrid.cuh (hybrid_merge_kernel + hybrid_select_kernel, as asp_hybrid_merge runs them) is
  compiled with g++ and walked on the CPU: per-shard shortlists built from the oracle's cosines and H3 scores, merged, must
  equal orc_search_hybrid on the whole item set bit for bit.
- distributed.sharded_search_hybrid is driven over gloo with an oracle-backed engine for every item-sharded layout of 2 and 4
  ranks: every rank must return the oracle's answer, and a failure on any rank must raise the same error on every rank."""
import ctypes as C
import os
import socket
import subprocess

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _compile_emul(out):
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "host_emul", "hybrid_merge_host.cpp")])


def _load_emul(path):
    lib = C.CDLL(path)
    vp, i64 = C.c_void_p, C.c_int64
    lib.hyb_merge_emulate.argtypes = [C.c_int, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.hyb_merge_emulate.restype = None
    return lib


@pytest.fixture(scope="module")
def emul_path(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hybm") / "libhybrid_merge_host.so")
    _compile_emul(out)
    return out


@pytest.fixture(scope="module")
def emul(emul_path):
    return _load_emul(emul_path)


def merge(lib, idx, cos, score, topk):
    """asp_hybrid_merge on the CPU: [parts, nq, m] shortlists -> (idx, score) [nq, topk]."""
    parts, nq, m = idx.shape
    idx, cos, score = (np.ascontiguousarray(a) for a in (idx, cos, score))
    pool_idx = np.empty((nq, max(m, 1)), dtype=np.int64)
    pool_score = np.empty((nq, max(m, 1)))
    out_idx = np.full((nq, topk), 99, dtype=np.int64)
    out_sc = np.full((nq, topk), 99.0)
    lib.hyb_merge_emulate(parts, nq, m, topk, idx.ctypes.data, cos.ctypes.data, score.ctypes.data, pool_idx.ctypes.data,
                          pool_score.ctypes.data, out_idx.ctypes.data, out_sc.ctypes.data)
    return out_idx, out_sc


def pool_len(n_total, topk, pool):
    """asp_hybrid_pool (include/arrowspace_b200.h)."""
    m = pool if pool > 0 else min(2 * topk, 31)
    return min(max(m, topk), n_total)


def shard_lists(cos, h3, cuts, m):
    """Each shard's top-m by (cosine desc, index asc) as asp_search_hybrid_shard returns them: [parts, nq, m] global
    indices, cosines and H3 scores, padded with -1 / NaN.  cos / h3: [nq, n] over all items."""
    nq = cos.shape[0]
    parts = len(cuts) - 1
    idx = np.full((parts, nq, m), -1, dtype=np.int64)
    cs = np.full((parts, nq, m), np.nan)
    sc = np.full((parts, nq, m), np.nan)
    for r in range(parts):
        a, b = cuts[r], cuts[r + 1]
        ids = np.arange(a, b)
        for qi in range(nq):
            order = np.lexsort((ids, -cos[qi, a:b]))[:m]
            k = len(order)
            idx[r, qi, :k] = ids[order]
            cs[r, qi, :k] = cos[qi, a:b][order]
            sc[r, qi, :k] = h3[qi, a:b][order]
    return idx, cs, sc


def _data(n, f, seed, dup_at=None, nq=23):
    rng = np.random.default_rng(seed)
    centres = rng.normal(size=(5, f))
    x = centres[rng.integers(0, 5, n)] + 0.3 * rng.normal(size=(n, f)) + 0.4
    if dup_at is not None:
        x[dup_at:dup_at + 12] = x[:12]                       # exact duplicates in another shard: ties across shards
    q = x[rng.integers(0, n, nq)] * 1.03 + 0.02 * rng.normal(size=(nq, f))
    q[:4] = x[:4] * 2.0                                      # queries that tie the duplicates exactly
    return x, q


def _oracle_scores(s, q, lq, tau):
    """The oracle's cosines (the score at tau = 1) and H3 scores at tau of every item, [nq, n]."""
    return np.stack([s.scores(q[i], lq[i], 1.0) for i in range(len(q))]), np.stack([s.scores(q[i], lq[i], tau) for i in range(len(q))])


def _cuts(n, parts, ragged=False):
    if not ragged:
        return [n * r // parts for r in range(parts + 1)]
    c = [0] + [n * (r + 1) // parts + (5 if r % 2 == 0 else -3) for r in range(parts - 1)] + [n]
    c[1] = 3                                                 # the first shard holds 3 rows: fewer than m
    return c


@pytest.mark.parametrize("n,f,topk,pool,parts,ragged,tau", [
    (300, 24, 5, 0, 2, False, 0.62),          # default pool (10)
    (300, 24, 5, 0, 8, True, 0.62),           # 8 shards, one of 3 rows
    (300, 24, 5, 2, 4, False, 0.3),           # pool < topk: raised to topk
    (300, 24, 1, 0, 3, True, 0.9),            # topk = 1
    (240, 16, 6, 31, 8, False, 0.0),          # the longest tensor-core list; tau = 0: pure lambda proximity
    (2100, 12, 10, 1024, 2, False, 0.62),     # m = 1024 (exact-scan shortlist), shards larger than m
    (2100, 12, 10, 1024, 8, False, 0.62),     # m = 1024, 8 shards smaller than m
    (200, 16, 6, 1000, 4, True, 0.62),        # pool >= n_total: the whole set
    (9, 5, 4, 0, 2, False, 0.62),             # shortlist (8) cut to n = 9
])
def test_merge_kernel_on_the_cpu_equals_the_oracle(oracle_mod, emul, n, f, topk, pool, parts, ragged, tau):
    x, q = _data(n, f, n + f + parts, dup_at=n // 2 + 7 if n > 40 else None)
    gp = {"eps": 0.7, "k": 4, "topk": topk, "p": 2.0, "sigma": 0.3}
    s, g = oracle_mod.build(gp, x)
    oidx, osc, lq = s.search_hybrid_batch(q, g, tau, pool)
    cos, h3 = _oracle_scores(s, q, lq, tau)
    m = pool_len(n, topk, pool)
    cuts = _cuts(n, parts, ragged)
    idx, cs, sc = shard_lists(cos, h3, cuts, m)
    out_idx, out_sc = merge(emul, idx, cs, sc, topk)
    assert np.array_equal(out_idx, oidx)
    ok = oidx >= 0
    assert np.array_equal(out_sc[ok], osc[ok]) and np.isnan(out_sc[~ok]).all()
    # the shards in any order give the same answer
    rev_idx, rev_sc = merge(emul, idx[::-1], cs[::-1], sc[::-1], topk)
    assert np.array_equal(rev_idx, out_idx) and np.array_equal(rev_sc[ok], out_sc[ok])


def test_duplicates_across_a_shard_boundary_tie_by_index(oracle_mod, emul):
    """Rows 0..11 are repeated at 150..161 (the second shard): the queries q[:4] = 2 x[:4] tie both copies in cosine and in
    score; the smaller global index must come first, as on one GPU."""
    n, f, topk = 300, 24, 6
    x, q = _data(n, f, 77, dup_at=150)
    s, g = oracle_mod.build({"eps": 0.7, "k": 4, "topk": topk, "p": 2.0, "sigma": 0.3}, x)
    oidx, osc, lq = s.search_hybrid_batch(q, g, 0.62, 0)
    cos, h3 = _oracle_scores(s, q, lq, 0.62)
    idx, cs, sc = shard_lists(cos, h3, [0, 150, 300], pool_len(n, topk, 0))
    out_idx, out_sc = merge(emul, idx, cs, sc, topk)
    assert np.array_equal(out_idx, oidx) and np.array_equal(out_sc, osc)
    for qi in range(4):
        row = list(out_idx[qi])
        assert qi in row and qi + 150 in row and row.index(qi) < row.index(qi + 150)


FAST = settings(max_examples=60, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])


@FAST
@given(st.integers(1, 60), st.integers(1, 8), st.integers(1, 12), st.integers(0, 70), st.integers(0, 2 ** 31 - 1))
def test_merge_over_random_splits(emul, n, parts, topk, pool, seed):
    """Random contiguous splits (empty shards included), heavy ties in cosine and score (values on a coarse grid): the merge
    equals H2-H3 on the whole set -- the m best cosines by (cosine desc, index asc), then the best topk of them by
    (score desc, index asc)."""
    rng = np.random.default_rng(seed)
    nq = int(rng.integers(1, 5))
    cos = np.round(rng.uniform(-1, 1, (nq, n)), 1)
    h3 = np.round(rng.uniform(0, 1, (nq, n)), 1)
    cuts = [0] + sorted(int(c) for c in rng.integers(0, n + 1, parts - 1)) + [n]
    m = pool_len(n, topk, pool)
    idx, cs, sc = shard_lists(cos, h3, cuts, m)
    out_idx, out_sc = merge(emul, idx, cs, sc, topk)
    ids = np.arange(n)
    for qi in range(nq):
        short = np.lexsort((ids, -cos[qi]))[:m]
        order = np.lexsort((short, -h3[qi, short]))[:topk]
        want = np.full(topk, -1)
        want[:len(order)] = short[order]
        assert list(out_idx[qi]) == list(want)
        assert np.array_equal(out_sc[qi, :len(order)], h3[qi, short[order]]) and np.isnan(out_sc[qi, len(order):]).all()


# ----------------------------------------------------------------------------- the orchestration over gloo

class OracleHybridEngine:
    """Stands in for CudaEngine in sharded_search_hybrid: the oracle's lambdas, cosines and scores restricted to the item
    shard's rows, the g++ build of the merge kernel, a numpy asp_topk_merge; CPU tensors for the collectives."""

    def __init__(self, s, g, emul_path, fail=False):
        import torch
        self.torch = torch
        self.device = torch.device("cpu")
        self.s, self.g = s, g
        self.emul = _load_emul(emul_path)
        self.fail = fail

    def hybrid_pool(self, n_total, topk, pool):
        return pool_len(n_total, topk, pool)

    def hybrid_shard(self, space, graph, q, tau, pool, idx, cos, score, lam):
        from pyarrowspace_b200._lib import ASP_ERR_NOMEM, ASP_ERR_ZERO_VECTOR, LibraryError
        if self.fail:
            raise LibraryError(ASP_ERR_NOMEM, "out of device memory in the hybrid search")
        if not q.any(axis=1).all():
            raise LibraryError(ASP_ERR_ZERO_VECTOR, "a query vector is all zeros: its Rayleigh quotient is undefined")
        a, b = space
        topk = self.g.params.topk
        _, _, lq = self.s.search_hybrid_batch(q, self.g, tau, pool)
        c_all, h_all = _oracle_scores(self.s, q, lq, tau)
        lam.numpy()[:] = lq
        if cos is None:                                      # whole set: the shard's best topk by score
            ids = np.arange(a, b)
            for qi in range(len(q)):
                order = np.lexsort((ids, -h_all[qi, a:b]))[:topk]
                idx.numpy()[qi, :len(order)] = ids[order]
                score.numpy()[qi, :len(order)] = h_all[qi, a:b][order]
            return
        i, c, h = shard_lists(c_all[:, a:b], h_all[:, a:b], [0, b - a], idx.shape[1])
        idx.numpy()[:] = np.where(i[0] >= 0, i[0] + a, -1)
        cos.numpy()[:] = c[0]
        score.numpy()[:] = h[0]

    def hybrid_merge(self, idx, cos, score, m, topk):
        out_idx, out_sc = merge(self.emul, idx.numpy(), cos.numpy(), score.numpy(), topk)
        return self.torch.from_numpy(out_idx), self.torch.from_numpy(out_sc)

    def topk_merge(self, idx, score):
        parts, nq, topk = idx.shape
        ii, ss = idx.numpy().transpose(1, 0, 2).reshape(nq, -1), score.numpy().transpose(1, 0, 2).reshape(nq, -1)
        out_idx = np.full((nq, topk), -1, dtype=np.int64)
        out_sc = np.full((nq, topk), np.nan)
        for qi in range(nq):
            keep = ii[qi] >= 0
            order = np.lexsort((ii[qi][keep], -ss[qi][keep]))[:topk]
            out_idx[qi, :len(order)] = ii[qi][keep][order]
            out_sc[qi, :len(order)] = ss[qi][keep][order]
        return self.torch.from_numpy(out_idx), self.torch.from_numpy(out_sc)


def _grid(world, rank, item_shards):
    """The grid dict of distributed.regroup for a search on CPU ranks."""
    from pyarrowspace_b200.distributed import grid_groups, grid_layout
    r_, c_, r, c = grid_layout(world, rank, item_shards)
    grid = dict(R=r_, C=c_, r=r, c=c, item_group=None, merge_group=None)
    if c_ > 1:
        item_groups, merge_groups = grid_groups(world, r_)
        grid["item_group"], grid["merge_group"] = item_groups[r], merge_groups[c]
    return grid


def _worker(rank, world, port, item_shards, case, emul_path, q):
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        import oracle
        from pyarrowspace_b200._lib import LibraryError
        from pyarrowspace_b200.distributed import sharded_search_hybrid
        n, f, topk, pool, tau, nq, zero_row, fail_rank = case
        x, qs = _data(n, f, 31 + n, dup_at=n // 2, nq=nq)
        if zero_row is not None:
            qs[zero_row] = 0.0
        s, g = oracle.build({"eps": 0.7, "k": 4, "topk": topk, "p": 2.0, "sigma": 0.3}, x)
        grid = _grid(world, rank, item_shards)
        cuts = [0, 3] + [n * (r + 1) // item_shards for r in range(1, item_shards)] if item_shards > 1 else [0, n]
        eng = OracleHybridEngine(s, g, emul_path, fail=(rank == fail_rank))
        try:
            out = sharded_search_hybrid(eng, (cuts[grid["r"]], cuts[grid["r"] + 1]), g, qs, tau, pool, topk, n, grid)
            q.put((rank, "ok", out))
        except LibraryError as e:
            q.put((rank, "raised", e.code))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        q.put((rank, "error", repr(e)))
        raise


def _free_port():
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    p = sk.getsockname()[1]
    sk.close()
    return p


def _run(world, item_shards, case, emul_path):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, item_shards, case, emul_path, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[1] != "error" for r in res), res
    return sorted(res, key=lambda r: r[0])


# (n, f, topk, pool, tau, nq, zero query row, failing rank); the first shard always holds only 3 rows
CASES = {"default": (300, 16, 5, 0, 0.62, 21, None, None),
         "pool40": (300, 16, 4, 40, 0.3, 10, None, None),
         "whole": (120, 8, 6, 500, 0.62, 9, None, None)}


@pytest.mark.parametrize("world,item_shards", [(2, 2), (4, 4), (4, 2)])
@pytest.mark.parametrize("case", sorted(CASES))
def test_sharded_search_hybrid_over_gloo(oracle_mod, emul_path, world, item_shards, case):
    """Every item-sharded layout of 2 and 4 ranks (R = world: one query slot; R = 2 of 4: two slots, each merging over its
    own R ranks, finished slices all-gathered): every rank returns the whole batch, equal to orc_search_hybrid bit for
    bit, lambda_q included."""
    n, f, topk, pool, tau, nq, _, _ = CASES[case]
    res = _run(world, item_shards, CASES[case], emul_path)
    x, qs = _data(n, f, 31 + n, dup_at=n // 2, nq=nq)
    s, g = oracle_mod.build({"eps": 0.7, "k": 4, "topk": topk, "p": 2.0, "sigma": 0.3}, x)
    oidx, osc, olq = s.search_hybrid_batch(qs, g, tau, pool)
    ok = oidx >= 0
    for rank, tag, out in res:
        assert tag == "ok", (rank, tag, out)
        idx, sc, lq = out
        assert np.array_equal(idx, oidx)
        assert np.array_equal(sc[ok], osc[ok]) and np.isnan(sc[~ok]).all()
        assert np.array_equal(lq, olq)


@pytest.mark.parametrize("world,item_shards,zero_row,fail_rank", [
    (4, 2, 1, None),          # a zero query in query slot 0 only: the ranks of slot 1 raise too
    (4, 2, None, 3),          # one rank fails on its own
    (2, 2, 0, None),
    (4, 4, None, 0),
])
def test_sharded_search_hybrid_same_error_on_every_rank(emul_path, world, item_shards, zero_row, fail_rank):
    from pyarrowspace_b200._lib import ASP_ERR_NOMEM, ASP_ERR_ZERO_VECTOR
    case = (200, 8, 3, 0, 0.62, 9, zero_row, fail_rank)
    res = _run(world, item_shards, case, emul_path)
    want = ASP_ERR_ZERO_VECTOR if zero_row is not None else ASP_ERR_NOMEM
    assert [(tag, code) for _, tag, code in res] == [("raised", want)] * world
