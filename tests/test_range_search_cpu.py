"""Range search without a GPU.

- The definition: per query every (allowed) item whose oracle score (orc_scores, the reference order) is >= min_score,
  ordered by (score desc, index asc).  With min_score set to the oracle search's k-th score, its first k entries are
  orc_search's answer bit for bit (ties at the boundary included).
- The cross-shard merge of csrc/range.cuh (asp_range_merge's host tables + range_merge_kernel) is compiled with g++ and
  walked on the CPU: per-shard pieces merged must equal the one-shard order.
- distributed.sharded_search_range is driven over gloo with an oracle-backed engine for the grid layouts of 2 and 4 ranks.
- Argument errors that need no library."""
import ctypes as C
import os
import socket
import subprocess

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def want_range(s, q, lq, tau, min_score, mask=None):
    """The definition: (idx, score) of every item with orc score >= min_score (and allowed), (score desc, index asc)."""
    sc = s.scores(q, lq, tau)
    ids = np.arange(len(sc))
    keep = sc >= min_score
    if mask is not None:
        keep &= mask
    ids, sc = ids[keep], sc[keep]
    order = np.lexsort((ids, -sc))
    return ids[order], sc[order]


def _data(n, f, seed, nq=17, dup=True):
    rng = np.random.default_rng(seed)
    centres = rng.normal(size=(5, f))
    x = centres[rng.integers(0, 5, n)] + 0.3 * rng.normal(size=(n, f)) + 0.4
    if dup:
        x[n // 2:n // 2 + 10] = x[:10]                       # exact duplicates: ties in score, resolved by index
    q = x[rng.integers(0, n, nq)] * 1.03 + 0.02 * rng.normal(size=(nq, f))
    q[:3] = x[:3] * 2.0                                      # queries that tie the duplicates exactly
    return x, q


GP = {"eps": 0.7, "k": 4, "topk": 7, "p": 2.0, "sigma": 0.3}


@pytest.mark.parametrize("tau", [0.0, 0.62, 1.0])
def test_definition_prefix_is_the_oracle_search(oracle_mod, tau):
    x, q = _data(300, 16, 5)
    s, g = oracle_mod.build(GP, x)
    oidx, osc, lq = s.search_batch(q, g, tau)
    k = GP["topk"]
    for qi in range(len(q)):
        idx, sc = want_range(s, q[qi], lq[qi], tau, osc[qi, k - 1])
        assert len(idx) >= k
        assert np.array_equal(idx[:k], oidx[qi]) and np.array_equal(sc[:k], osc[qi])
        assert (sc >= osc[qi, k - 1]).all() and (sc[k:] == osc[qi, k - 1]).all()   # beyond k: only boundary ties


def test_boundary_ties_are_all_included(oracle_mod):
    """q[:3] = 2 x[:3] and rows n/2 .. n/2 + 9 repeat rows 0..9: both copies score the same, so a threshold at that score
    returns both, the smaller index first."""
    x, q = _data(300, 16, 9)
    s, g = oracle_mod.build(GP, x)
    _, _, lq = s.search_batch(q, g, 1.0)
    for qi in range(3):
        sc_all = s.scores(q[qi], lq[qi], 1.0)
        assert sc_all[qi] == sc_all[150 + qi]
        idx, sc = want_range(s, q[qi], lq[qi], 1.0, sc_all[qi])
        assert qi in idx and 150 + qi in idx and list(idx).index(qi) < list(idx).index(150 + qi)


FAST = settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])


@FAST
@given(st.integers(20, 120), st.sampled_from([0.0, 0.3, 0.62, 1.0]), st.floats(0.0, 1.0), st.integers(0, 2 ** 31 - 1))
def test_definition_property(oracle_mod, n, tau, frac, seed):
    """Random data and thresholds: the range answer is the set {score >= min_score}, sorted; its prefix of length k is the
    oracle's top-k whenever the k-th score clears the threshold."""
    x, q = _data(n, 8, seed, nq=4, dup=False)
    gp = dict(GP, topk=min(5, n))
    s, g = oracle_mod.build(gp, x)
    oidx, osc, lq = s.search_batch(q, g, tau)
    for qi in range(len(q)):
        sc_all = s.scores(q[qi], lq[qi], tau)
        thr = float(np.quantile(sc_all, frac))
        idx, sc = want_range(s, q[qi], lq[qi], tau, thr)
        assert set(idx) == set(np.nonzero(sc_all >= thr)[0])
        assert all((sc[i] > sc[i + 1]) or (sc[i] == sc[i + 1] and idx[i] < idx[i + 1]) for i in range(len(idx) - 1))
        k = gp["topk"]
        if osc[qi, k - 1] >= thr:
            assert np.array_equal(idx[:k], oidx[qi]) and np.array_equal(sc[:k], osc[qi])


# ----------------------------------------------------------------------------- the merge body, walked on the CPU

def _compile_emul(out):
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "host_emul", "range_merge_host.cpp")])


def _load_emul(path):
    lib = C.CDLL(path)
    vp, i64 = C.c_void_p, C.c_int64
    lib.range_merge_emulate.argtypes = [C.c_int, i64, vp, vp, vp, vp, vp]
    lib.range_merge_emulate.restype = None
    lib.range_desc_key.argtypes = [C.c_double]
    lib.range_desc_key.restype = C.c_uint64
    lib.range_key_score.argtypes = [C.c_uint64]
    lib.range_key_score.restype = C.c_double
    return lib


@pytest.fixture(scope="module")
def emul_path(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("rngm") / "librange_merge_host.so")
    _compile_emul(out)
    return out


@pytest.fixture(scope="module")
def emul(emul_path):
    return _load_emul(emul_path)


def merge(lib, counts, idx, score):
    """asp_range_merge on the CPU: counts [parts, nq], concatenated parts -> merged (idx, score)."""
    counts = np.ascontiguousarray(counts, dtype=np.int64)
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    score = np.ascontiguousarray(score, dtype=np.float64)
    total = int(counts.sum())
    out_idx = np.full(max(total, 1), -7, dtype=np.int64)
    out_sc = np.full(max(total, 1), 99.0)
    lib.range_merge_emulate(counts.shape[0], counts.shape[1], counts.ctypes.data, idx.ctypes.data, score.ctypes.data,
                            out_idx.ctypes.data, out_sc.ctypes.data)
    return out_idx[:total], out_sc[:total]


def shard_pieces(scores, keep, cuts):
    """Per-shard CSR pieces as asp_search_range_batch returns them on shard [cuts[r], cuts[r+1]): counts [parts, nq] and the
    concatenated parts' hits (GLOBAL indices), each query's hits by (score desc, index asc)."""
    nq = scores.shape[0]
    parts = len(cuts) - 1
    counts = np.zeros((parts, nq), dtype=np.int64)
    idx, sc = [], []
    for r in range(parts):
        a, b = cuts[r], cuts[r + 1]
        ids = np.arange(a, b)
        for qi in range(nq):
            k = keep[qi, a:b]
            i, s = ids[k], scores[qi, a:b][k]
            order = np.lexsort((i, -s))
            counts[r, qi] = len(order)
            idx.append(i[order])
            sc.append(s[order])
    return counts, np.concatenate(idx) if idx else np.empty(0, np.int64), np.concatenate(sc) if sc else np.empty(0)


def one_shard(scores, keep):
    idx, sc = [], []
    ids = np.arange(scores.shape[1])
    for qi in range(scores.shape[0]):
        i, s = ids[keep[qi]], scores[qi][keep[qi]]
        order = np.lexsort((i, -s))
        idx.append(i[order])
        sc.append(s[order])
    return np.concatenate(idx), np.concatenate(sc)


@pytest.mark.parametrize("parts", [2, 3, 4, 5, 8])
def test_merge_equals_one_shard_order(oracle_mod, emul, parts):
    x, q = _data(300, 16, parts)
    s, g = oracle_mod.build(GP, x)
    _, osc, lq = s.search_batch(q, g, 0.62)
    scores = np.stack([s.scores(q[i], lq[i], 0.62) for i in range(len(q))])
    thr = np.quantile(scores, 0.9, axis=1)[:, None]
    thr[5] = 5.0                                              # a query with no hit anywhere
    keep = scores >= thr
    cuts = [300 * r // parts for r in range(parts + 1)]
    cuts[1] = 0 if parts > 2 else cuts[1]                     # an empty shard
    counts, idx, sc = shard_pieces(scores, keep, cuts)
    out_idx, out_sc = merge(emul, counts, idx, sc)
    want_idx, want_sc = one_shard(scores, keep)
    assert np.array_equal(out_idx, want_idx) and np.array_equal(out_sc, want_sc)


def test_cross_shard_duplicate_scores_tie_by_index(oracle_mod, emul):
    x, q = _data(300, 16, 3)
    s, g = oracle_mod.build(GP, x)
    _, _, lq = s.search_batch(q, g, 1.0)
    scores = np.stack([s.scores(q[i], lq[i], 1.0) for i in range(len(q))])
    keep = scores >= np.quantile(scores, 0.8, axis=1)[:, None]
    counts, idx, sc = shard_pieces(scores, keep, [0, 150, 300])      # rows 150.. repeat rows 0..9 across the boundary
    out_idx, out_sc = merge(emul, counts, idx, sc)
    want_idx, want_sc = one_shard(scores, keep)
    assert np.array_equal(out_idx, want_idx) and np.array_equal(out_sc, want_sc)
    # the shards in the other order: the same answer
    ca, ia, sa = shard_pieces(scores, keep, [150, 300])
    cb, ib, sb = shard_pieces(scores, keep, [0, 150])
    rev = merge(emul, np.vstack([ca, cb]), np.concatenate([ia, ib]), np.concatenate([sa, sb]))
    assert np.array_equal(rev[0], want_idx) and np.array_equal(rev[1], want_sc)


def test_merge_with_nothing(emul):
    out_idx, out_sc = merge(emul, np.zeros((3, 4), dtype=np.int64), np.empty(0, np.int64), np.empty(0))
    assert len(out_idx) == 0 and len(out_sc) == 0


@FAST
@given(st.integers(1, 60), st.integers(1, 8), st.integers(1, 5), st.integers(0, 2 ** 31 - 1))
def test_merge_over_random_splits(emul, n, parts, nq, seed):
    """Random contiguous splits (empty shards included) and heavy ties (scores on a coarse grid)."""
    rng = np.random.default_rng(seed)
    scores = np.round(rng.uniform(-1, 1, (nq, n)), 1)
    keep = rng.uniform(size=(nq, n)) < rng.uniform()
    cuts = [0] + sorted(int(c) for c in rng.integers(0, n + 1, parts - 1)) + [n]
    counts, idx, sc = shard_pieces(scores, keep, cuts)
    out_idx, out_sc = merge(emul, counts, idx, sc)
    want_idx, want_sc = one_shard(scores, keep)
    assert np.array_equal(out_idx, want_idx) and np.array_equal(out_sc, want_sc)


def test_sort_key_orders_scores_descending(emul):
    vals = [float("-inf"), -1.5, -1.0, -1e-300, -0.0, 0.0, 5e-324, 1e-300, 0.25, 1.0, 2.0, float("inf")]
    keys = [emul.range_desc_key(v) for v in vals]
    assert keys == sorted(keys, reverse=True)
    assert keys[4] == keys[5]                                # -0.0 and 0.0 tie, as they do as doubles
    for v in vals:
        back = emul.range_key_score(emul.range_desc_key(v))
        assert back == v and (v != 0.0 or np.signbit(back) == False)   # noqa: E712


# ----------------------------------------------------------------------------- the orchestration over gloo

class OracleRangeEngine:
    """Stands in for CudaEngine in sharded_search_range: the oracle's lambdas and scores restricted to the item shard's
    rows, the g++ build of the merge kernel; CPU tensors for the collectives."""

    def __init__(self, s, g, emul_path, fail=False):
        import torch
        self.torch = torch
        self.device = torch.device("cpu")
        self.s, self.g = s, g
        self.emul = _load_emul(emul_path)
        self.fail = fail

    def range_shard(self, space, graph, q, tau, min_score, allowed, max_hits):
        from pyarrowspace_b200._lib import ASP_ERR_LIMIT, ASP_ERR_NOMEM, ASP_ERR_ZERO_VECTOR, LibraryError
        if self.fail:
            raise LibraryError(ASP_ERR_NOMEM, "out of device memory in the range search")
        if not q.any(axis=1).all():
            raise LibraryError(ASP_ERR_ZERO_VECTOR, "a query vector is all zeros: its Rayleigh quotient is undefined")
        a, b = space
        _, _, lq = self.s.search_batch(q, self.g, tau)
        scores = np.stack([self.s.scores(q[i], lq[i], tau) for i in range(len(q))])
        keep = scores >= min_score
        if allowed is not None:
            keep &= allowed[None, :]
        keep[:, :a] = False
        keep[:, b:] = False
        counts, idx, sc = shard_pieces(scores, keep, [0, scores.shape[1]])
        if max_hits > 0 and counts.sum() > max_hits:
            raise LibraryError(ASP_ERR_LIMIT, "range search: %d hits, more than max_hits = %d" % (counts.sum(), max_hits))
        return self.torch.from_numpy(idx), self.torch.from_numpy(sc), counts[0], lq

    def range_merge(self, counts, idx, score):
        out_idx, out_sc = merge(self.emul, counts, idx.numpy(), score.numpy())
        return self.torch.from_numpy(out_idx), self.torch.from_numpy(out_sc)


def _grid(world, rank, item_shards):
    from pyarrowspace_b200.distributed import grid_groups, grid_layout
    r_, c_, r, c = grid_layout(world, rank, item_shards)
    grid = dict(R=r_, C=c_, r=r, c=c, item_group=None, merge_group=None)
    if c_ > 1:
        item_groups, merge_groups = grid_groups(world, r_)
        grid["item_group"], grid["merge_group"] = item_groups[r], merge_groups[c]
    return grid


def _cuts(n, item_shards):
    return [0, 3] + [n * (r + 1) // item_shards for r in range(1, item_shards)] if item_shards > 1 else [0, n]


def _mask(n, kind):
    if kind is None:
        return None
    m = np.ones(n, dtype=bool)
    m[::3] = False
    m[:3] = False                                            # the 3-row first shard has no allowed row
    return m


def _worker(rank, world, port, item_shards, case, emul_path, q):
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        import oracle
        from pyarrowspace_b200._lib import LibraryError
        from pyarrowspace_b200.distributed import sharded_search_range
        n, f, tau, frac, nq, zero_row, fail_rank, mask_kind, max_hits = case
        x, qs = _data(n, f, 31 + n, nq=nq)
        if zero_row is not None:
            qs[zero_row] = 0.0
        s, g = oracle.build(GP, x)
        grid = _grid(world, rank, item_shards)
        cuts = _cuts(n, item_shards)
        eng = OracleRangeEngine(s, g, emul_path, fail=(rank == fail_rank))
        try:
            out = sharded_search_range(eng, (cuts[grid["r"]], cuts[grid["r"] + 1]), g, qs, tau, frac, n, grid,
                                       allowed=_mask(n, mask_kind), max_hits=max_hits)
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


# (n, f, tau, min_score, nq, zero query row, failing rank, mask, max_hits); the first item shard holds only 3 rows
CASES = {"plain": (300, 16, 0.62, 0.8, 13, None, None, None, 1 << 26),
         "masked": (300, 16, 0.62, 0.7, 9, None, None, "thirds", 1 << 26),
         "tau0": (200, 8, 0.0, 0.9, 7, None, None, None, 1 << 26)}


@pytest.mark.parametrize("world,item_shards", [(2, 2), (4, 4), (4, 2), (4, 1)])
@pytest.mark.parametrize("case", sorted(CASES))
def test_sharded_search_range_over_gloo(oracle_mod, emul_path, world, item_shards, case):
    """R = 2 of 2, 4 of 4 (one query slot), 2 of 4 (two slots, each merging over its R ranks) and 1 of 4 (four slots, no
    merge): every rank returns the whole batch, equal to the definition bit for bit, lambda_q included."""
    n, f, tau, thr, nq, _, _, mask_kind, _ = CASES[case]
    res = _run(world, item_shards, CASES[case], emul_path)
    x, qs = _data(n, f, 31 + n, nq=nq)
    s, g = oracle_mod.build(GP, x)
    _, _, olq = s.search_batch(qs, g, tau)
    mask = _mask(n, mask_kind)
    want = [want_range(s, qs[i], olq[i], tau, thr, mask) for i in range(nq)]
    want_ptr = np.concatenate([[0], np.cumsum([len(w[0]) for w in want])])
    for rank, tag, out in res:
        assert tag == "ok", (rank, tag, out)
        indptr, idx, sc, lq = out
        assert np.array_equal(indptr, want_ptr)
        assert np.array_equal(idx, np.concatenate([w[0] for w in want]))
        assert np.array_equal(sc, np.concatenate([w[1] for w in want]))
        assert np.array_equal(lq, olq)


@pytest.mark.parametrize("world,item_shards,zero_row,fail_rank,max_hits", [
    (4, 2, 1, None, 1 << 26),  # a zero query in query slot 0 only: the ranks of slot 1 raise too
    (4, 2, None, 3, 1 << 26),  # one rank fails on its own
    (2, 2, 0, None, 1 << 26),
    (4, 4, None, 0, 1 << 26),
    (4, 2, None, None, 40),    # the merged total passes the cap while no shard does on its own
    (2, 2, None, None, 5),     # a shard passes the cap by itself
])
def test_sharded_search_range_same_error_on_every_rank(emul_path, world, item_shards, zero_row, fail_rank, max_hits):
    from pyarrowspace_b200._lib import ASP_ERR_LIMIT, ASP_ERR_NOMEM, ASP_ERR_ZERO_VECTOR
    case = (200, 8, 0.62, 0.5, 9, zero_row, fail_rank, None, max_hits)
    res = _run(world, item_shards, case, emul_path)
    want = ASP_ERR_ZERO_VECTOR if zero_row is not None else ASP_ERR_NOMEM if fail_rank is not None else ASP_ERR_LIMIT
    assert [(tag, code) for _, tag, code in res] == [("raised", want)] * world


# ----------------------------------------------------------------------------- argument errors (no library needed)

def test_argument_checks():
    from pyarrowspace_b200.api import DEFAULT_MAX_RESULTS, _check_allowed, _check_max_results, _check_min_score
    assert _check_min_score(0.5) == 0.5 and _check_min_score(np.float32(0.25)) == 0.25 and _check_min_score(1) == 1.0
    assert _check_min_score(float("-inf")) == float("-inf") and _check_min_score(3.0) == 3.0
    with pytest.raises(ValueError):
        _check_min_score(float("nan"))
    for bad in ("0.5", None, True, 1 + 2j, [0.5]):
        with pytest.raises(TypeError):
            _check_min_score(bad)
    assert _check_max_results(None) == DEFAULT_MAX_RESULTS == 1 << 26 and _check_max_results(np.int64(7)) == 7
    for bad, exc in ((0, ValueError), (-3, ValueError), (2.0, TypeError), (True, TypeError), ("9", TypeError)):
        with pytest.raises(exc):
            _check_max_results(bad)
    with pytest.raises(TypeError):
        _check_allowed(np.ones(5, dtype=np.int8), 5)
    with pytest.raises(ValueError):
        _check_allowed(np.ones(4, dtype=bool), 5)
