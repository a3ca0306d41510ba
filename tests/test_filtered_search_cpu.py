"""Filtered search (allowed=) without a GPU.

The reference of a filtered search is its definition, built here from the unchanged oracle: the oracle's scores
(orc_scores, the expression orc_search ranks by) of every item, ordered by (score desc, index asc), restricted to the
allowed items and cut to topk; for the hybrid search the shortlist is the m allowed items of largest cosine (m from the
whole item count), re-ranked by the oracle's H3 score.  With an all-true mask these definitions must give orc_search /
orc_search_hybrid bit for bit, which checks the helpers against the oracle itself; the GPU tests import them.

Also here:
- distributed.pack_allowed, the per-rank slice of the mask that the library takes;
- distributed.sharded_search_hybrid with a mask, over gloo, with an oracle-backed engine (R = 2 of 2, 4 of 4, 2 of 4; one
  item shard has no allowed row).  The -1-padded shard lists go through the unchanged merges."""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

import test_hybrid_sharded_cpu as hs

GP = {"eps": 0.7, "k": 4, "topk": 6, "p": 2.0, "sigma": 0.3}


def want_search(s, q, lq, tau, mask, topk):
    """The filtered search by definition over the oracle space s: (idx, score) [nq, topk] padded with -1 / NaN.  lq: the
    queries' lambdas as orc_search computes them."""
    ids = np.flatnonzero(mask)
    idx = np.full((len(q), topk), -1, dtype=np.int64)
    sc = np.full((len(q), topk), np.nan)
    for i in range(len(q)):
        v = s.scores(q[i], lq[i], tau)[ids]
        order = np.lexsort((ids, -v))[:topk]
        idx[i, :len(order)] = ids[order]
        sc[i, :len(order)] = v[order]
    return idx, sc


def want_hybrid(s, q, lq, tau, pool, mask, topk):
    """The filtered hybrid search by definition: H2 over the allowed items (m from the whole item count), then H3."""
    m = hs.pool_len(s.nitems, topk, pool)
    ids = np.flatnonzero(mask)
    idx = np.full((len(q), topk), -1, dtype=np.int64)
    sc = np.full((len(q), topk), np.nan)
    for i in range(len(q)):
        c = s.scores(q[i], lq[i], 1.0)[ids]                  # the score at tau = 1 is the cosine
        short = ids[np.lexsort((ids, -c))][:m]
        h = s.scores(q[i], lq[i], tau)[short]
        order = np.lexsort((short, -h))[:topk]
        idx[i, :len(order)] = short[order]
        sc[i, :len(order)] = h[order]
    return idx, sc


def _data(n, f, seed, nq=9, dup=0):
    rng = np.random.default_rng(seed)
    cent = rng.normal(size=(4, f))
    x = np.abs(cent[rng.integers(0, 4, n)] + 0.3 * rng.normal(size=(n, f))) + 0.1
    if dup:
        x[n - dup:] = x[:dup]
    q = x[rng.integers(0, n, nq)] * 1.02 + 0.01 * rng.normal(size=(nq, f))
    if dup:
        q[:3] = x[:3] * 1.5                                  # ties between the copies
    return x, q


def _eq(a_idx, a_sc, b_idx, b_sc):
    assert np.array_equal(a_idx, b_idx)
    ok = b_idx >= 0
    assert np.array_equal(a_sc[ok], b_sc[ok]) and np.isnan(a_sc[~ok]).all()


FAST = settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])


@pytest.mark.parametrize("tau", [0.0, 0.62, 1.0])
def test_definitions_with_every_item_allowed_are_the_oracle(oracle_mod, tau):
    x, q = _data(300, 12, 3, dup=40)
    s, g = oracle_mod.build(GP, x)
    every = np.ones(300, dtype=bool)
    oi, osc, lq = s.search_batch(q, g, tau)
    _eq(*want_search(s, q, lq, tau, every, GP["topk"]), oi, osc)
    for pool in (0, 2, 9, 40, 300, 1000):
        hi, hsc, hlq = s.search_hybrid_batch(q, g, tau, pool)
        _eq(*want_hybrid(s, q, hlq, tau, pool, every, GP["topk"]), hi, hsc)


@FAST
@given(st.integers(0, 2 ** 31 - 1), st.sampled_from([0.0, 0.3, 0.62, 1.0]), st.integers(0, 40))
def test_definitions_with_every_item_allowed_random(oracle_mod, seed, tau, pool):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(5, 80))
    x, q = _data(n, 6, seed % 1000, nq=3, dup=min(4, n // 2))
    s, g = oracle_mod.build(GP, x)
    every = np.ones(n, dtype=bool)
    hi, hsc, hlq = s.search_hybrid_batch(q, g, tau, pool)
    _eq(*want_hybrid(s, q, hlq, tau, pool, every, GP["topk"]), hi, hsc)
    if (hlq != 0.0).all():
        oi, osc, _ = s.search_batch(q, g, tau)
        _eq(*want_search(s, q, hlq, tau, every, GP["topk"]), oi, osc)


@pytest.mark.parametrize("n_total,world", [(37, 4), (1001, 8), (8, 8), (5, 2), (129, 4), (301, 8)])
def test_pack_allowed_slices_and_packs_lsb_first(n_total, world):
    from pyarrowspace_b200.distributed import pack_allowed, shard_rows
    mask = np.random.default_rng(n_total).random(n_total) < 0.4
    for rank in range(world):
        a, b = shard_rows(n_total, world, rank)
        bits = pack_allowed(mask, a, b - a)
        assert bits.dtype == np.uint8 and bits.shape == ((b - a + 7) // 8,)
        for i in range(b - a):
            assert bool((bits[i // 8] >> (i % 8)) & 1) == mask[a + i]
        assert not (np.unpackbits(bits, bitorder="little")[b - a:]).any()
    for a, b in ((3, 20), (5, 6), (11, 11), (13, 37)):       # offsets that are not multiples of 8
        if b > n_total:
            continue
        bits = pack_allowed(mask, a, b - a)
        assert np.array_equal(np.unpackbits(bits, bitorder="little")[:b - a].astype(bool), mask[a:b])


# ----------------------------------------------------------------------------- the orchestration over gloo

class FilteredOracleEngine(hs.OracleHybridEngine):
    """OracleHybridEngine whose shard lists come from the allowed rows of the shard only."""

    def hybrid_shard(self, space, graph, q, tau, pool, idx, cos, score, lam, allowed=None):
        if allowed is None:
            return super().hybrid_shard(space, graph, q, tau, pool, idx, cos, score, lam)
        a, b = space
        topk = self.g.params.topk
        _, _, lq = self.s.search_hybrid_batch(q, self.g, tau, pool)
        c_all, h_all = hs._oracle_scores(self.s, q, lq, tau)
        lam.numpy()[:] = lq
        ids = np.arange(a, b)[allowed[a:b]]
        key = h_all if cos is None else c_all
        width = topk if cos is None else idx.shape[1]
        for qi in range(len(q)):
            order = ids[np.lexsort((ids, -key[qi, ids]))][:width]
            idx.numpy()[qi, :len(order)] = order
            score.numpy()[qi, :len(order)] = h_all[qi, order]
            if cos is not None:
                cos.numpy()[qi, :len(order)] = c_all[qi, order]


def _case_mask(n, cuts):
    mask = np.random.default_rng(n).random(n) < 0.5
    mask[cuts[1]:cuts[2]] = False                             # the second item shard has no allowed row
    return mask


def _cuts(n, item_shards):
    return [0, 3] + [n * (r + 1) // item_shards for r in range(1, item_shards)] if item_shards > 1 else [0, n]


def _worker(rank, world, port, item_shards, case, emul_path, q):
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        import oracle
        from pyarrowspace_b200.distributed import sharded_search_hybrid
        n, f, topk, pool, tau, nq = case
        x, qs = hs._data(n, f, 31 + n, dup_at=n // 2, nq=nq)
        s, g = oracle.build({"eps": 0.7, "k": 4, "topk": topk, "p": 2.0, "sigma": 0.3}, x)
        grid = hs._grid(world, rank, item_shards)
        cuts = _cuts(n, item_shards)
        cuts = cuts + [n] if len(cuts) < 3 else cuts
        mask = _case_mask(n, cuts)
        eng = FilteredOracleEngine(s, g, emul_path)
        out = sharded_search_hybrid(eng, (cuts[grid["r"]], cuts[grid["r"] + 1]), g, qs, tau, pool, topk, n, grid,
                                    allowed=mask)
        q.put((rank, "ok", out))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                              # pragma: no cover
        q.put((rank, "error", repr(e)))
        raise


def _run(world, item_shards, case, emul_path):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = hs._free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, item_shards, case, emul_path, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[1] != "error" for r in res), res
    return sorted(res, key=lambda r: r[0])


CASES = {"default": (300, 16, 5, 0, 0.62, 21), "pool40": (300, 16, 4, 40, 0.3, 10), "whole": (120, 8, 6, 500, 0.62, 9)}


@pytest.mark.parametrize("world,item_shards", [(2, 2), (4, 4), (4, 2)])
@pytest.mark.parametrize("case", sorted(CASES))
def test_filtered_sharded_search_hybrid_over_gloo(oracle_mod, emul_path, world, item_shards, case):
    """Every rank returns the filtered hybrid search over all items by definition, bit for bit, although one item shard contributes only
    -1 padding: the merges (asp_hybrid_merge, asp_topk_merge) take such lists unchanged."""
    n, f, topk, pool, tau, nq = CASES[case]
    res = _run(world, item_shards, CASES[case], emul_path)
    x, qs = hs._data(n, f, 31 + n, dup_at=n // 2, nq=nq)
    s, g = oracle_mod.build({"eps": 0.7, "k": 4, "topk": topk, "p": 2.0, "sigma": 0.3}, x)
    cuts = _cuts(n, item_shards)
    cuts = cuts + [n] if len(cuts) < 3 else cuts
    mask = _case_mask(n, cuts)
    _, _, olq = s.search_hybrid_batch(qs, g, tau, pool)
    oidx, osc = want_hybrid(s, qs, olq, tau, pool, mask, topk)
    for rank, tag, out in res:
        assert tag == "ok", (rank, tag, out)
        idx, sc, lq = out
        _eq(idx, sc, oidx, osc)
        assert np.array_equal(lq, olq)
        assert mask[idx[idx >= 0]].all()


@pytest.fixture(scope="module")
def emul_path(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hybm_f") / "libhybrid_merge_host.so")
    hs._compile_emul(out)
    return out
