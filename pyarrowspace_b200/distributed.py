"""Multi-GPU host logic: one process per GPU, ``torch.distributed`` (NCCL over NVLink) for the plumbing.

The path shards by rows (SURVEY.md section 8(e)): rank r owns the rows of Gram segments
[r*8/world, (r+1)*8/world).  Exchange steps, and nothing else:

  build   1. all-gather of the per-segment partial Grams (8 x F x F f64: 9.4 MB at F = 384)
          2. (rare) rank-ordered continuation of left-to-right column sums for the pairs whose
             distance falls inside the rounding band: rank r continues rank r-1's sums
  search  3. all-gather of the per-shard top-k lists (16 * Q * topk bytes per rank) + merge kernel
  item graph (nodes = items)
          4. all-gather of the item shards (the "halo rows": every rank scores ITS rows against ALL items)
          5. all-gather of the per-rank neighbour lists (12 * N * k bytes), Laplacian assembled on every rank
  regrouping (item_shards = R < world = G; `regroup`)
          6. the build is always row-partitioned G ways; for the search the G ranks form an R x C grid (C = G / R): the C
             consecutive ranks of item shard r all-gather their rows, lambdas and norms (once, at build time), and every
             rank then answers 1/C of each query batch against item shard r.  Per-query work (lambda_q, operand
             projection, stage 2, merge) is divided by C instead of being replicated G times; R = 1 needs no cross-GPU
             merge at all.  R = G is the fully item-sharded layout (every rank scores every query).
  hybrid search (R > 1; `sharded_search_hybrid`)
          7. all-gather of the per-shard cosine shortlists (idx, cosine, score: 24 * Q * m bytes per rank) among the R ranks
             of a query slot + merge kernel; the C slots all-gather their finished slices
  range search (`sharded_search_range`)
          8. all-gather of the per-shard hit counts (8 bytes per query), then of the ragged hits (16 bytes each) among the R
             ranks of a query slot + merge kernel; the C slots all-gather their counts and finished slices

The summation tree of the Gram is fixed (segments -> slices), so every world size produces
bit-identical graphs, lambdas and result lists.

`sharded_build` / `sharded_search` take an *engine* (the calls into the C ABI) so that the
orchestration can be exercised on CPU with gloo in tests; the product engine is `CudaEngine`.
"""
import ctypes as C

import numpy as np

from . import _lib


def _dist():
    import torch.distributed as dist
    return dist


def shard_rows(n_total, world, rank):
    r0, r1 = C.c_int64(), C.c_int64()
    _lib.check(_lib.load().asp_shard_rows(int(n_total), int(world), int(rank), C.byref(r0), C.byref(r1)))
    return r0.value, r1.value


def pack_allowed(allowed, row0, n_local):
    """A rank's slice [row0, row0 + n_local) of the global bool mask `allowed`, packed LSB-first as the library takes it
    (ceil(n_local / 8) bytes: bit i % 8 of byte i / 8 is local row i)."""
    return np.packbits(np.ascontiguousarray(allowed[row0:row0 + n_local], dtype=np.bool_), bitorder="little")


class CudaEngine:
    """The product engine: every method is one call into libarrowspace_b200.so."""

    def __init__(self, device=None):
        import torch
        self.torch = torch
        self.lib = _lib.load()
        self.ctx = _lib.context(device)
        self.device = torch.device("cuda", self.lib.asp_ctx_device(self.ctx))

    def _ptr(self, x):
        return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data

    def space_create(self, shard, n_total, world, rank):
        """Copies the row shard into the library (host ndarray or device tensor, any strides; float64 only)."""
        if hasattr(shard, "data_ptr"):
            if shard.dtype != self.torch.float64 or shard.dim() != 2:
                raise TypeError("argument 'items': expected a 2-D float64 tensor")
            shard = shard.contiguous()
            if shard.is_cuda:
                self.torch.cuda.current_stream(shard.device).synchronize()      # the library runs on its own stream
        else:
            if shard.dtype != np.float64 or shard.ndim != 2:
                raise TypeError("argument 'items': expected 2-D numpy.ndarray of float64")
            shard = np.ascontiguousarray(shard)
        n_local, f = shard.shape
        h = C.c_void_p()
        _lib.check(self.lib.asp_space_create(self.ctx, self._ptr(shard), n_local, f, n_total, world, rank, C.byref(h)))
        return h

    def gram_partials(self, space, f):
        segs = self.torch.zeros((_lib.GRAM_SEGMENTS, f, f), dtype=self.torch.float64, device=self.device)
        self.torch.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_space_gram_partials(space, segs.data_ptr()))
        _lib.check(self.lib.asp_ctx_synchronize(self.ctx))
        return segs

    def graph_from_gram(self, segs, f, n_total, cgp, sw, pairs, sums):
        """-> (graph handle | None, need_pairs int32[m, 2])"""
        cap = 1 << 16
        n_exact = 0 if pairs is None else len(pairs)
        pp = pairs.ctypes.data if n_exact else None
        sp = sums.ctypes.data if n_exact else None
        while True:
            need = np.empty((cap, 2), dtype=np.int32)
            n_need = C.c_int64(0)
            hg = C.c_void_p()
            rc = self.lib.asp_graph_from_gram(self.ctx, segs.data_ptr(), f, n_total, C.byref(cgp), C.byref(sw), pp, sp,
                                              n_exact, need.ctypes.data, cap, C.byref(n_need), C.byref(hg))
            if rc == _lib.ASP_ERR_ARG and n_need.value > cap:       # more undecided pairs than the list holds: grow it
                cap = n_need.value
                continue
            break
        if rc == _lib.ASP_NEED_EXACT:
            return None, need[: n_need.value].copy()
        _lib.check(rc)
        return hg, need[:0]

    def exact_pairs(self, space, pairs, sums):
        _lib.check(self.lib.asp_space_exact_pairs(space, pairs.ctypes.data, len(pairs), sums.ctypes.data))
        return sums

    def compute_lambdas(self, space, graph):
        _lib.check(self.lib.asp_space_compute_lambdas(space, graph))

    # ---- pre-graph reduction (SURVEY.md 8(f)-1)
    def sampled_rows(self, shard, red, row0):
        """R1 for this rank's rows (global offset row0) -> the kept rows as a device tensor [m, f]."""
        t = self.torch
        n_local = shard.shape[0]
        rows = np.empty(max(n_local, 1), dtype=np.int32)
        cnt = C.c_int64(0)
        _lib.check(self.lib.asp_reduction_sample(C.byref(red), int(row0), int(n_local), rows.ctypes.data, C.byref(cnt)))
        sel = t.from_numpy(rows[:cnt.value].astype(np.int64))
        if hasattr(shard, "is_cuda"):
            return shard.to(self.device).index_select(0, sel.to(self.device)).contiguous()
        return t.from_numpy(np.ascontiguousarray(shard[sel.numpy()])).to(self.device)

    def reduce_rows(self, rows, red, n_total):
        """R2-R4 on the gathered sample (every rank runs the same deterministic kernels on the same rows) ->
        (space handle over the centroids, info dict)."""
        h, hc = C.c_void_p(), C.c_void_p()
        info = _lib.ReductionInfo()
        n, f = rows.shape
        self.torch.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_space_create(self.ctx, rows.data_ptr(), n, f, n, 1, 0, C.byref(h)))
        try:
            _lib.check(self.lib.asp_space_reduce(h, C.byref(red), int(n_total), C.byref(info), C.byref(hc)))
        finally:
            self.lib.asp_free_space(h)
        return hc, info.as_dict()

    def feature_graph(self, space, cgp, sw):
        hg = C.c_void_p()
        _lib.check(self.lib.asp_space_feature_graph(space, C.byref(cgp), C.byref(sw), C.byref(hg)))
        return hg

    # ---- regrouping (item_shards < world)
    def lambdas_norms(self, space, n_local):
        """-> (lambdas, norms) of the space's rows as device tensors."""
        t = self.torch
        lam = t.empty(n_local, dtype=t.float64, device=self.device)
        nrm = t.empty(n_local, dtype=t.float64, device=self.device)
        t.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_space_lambdas(space, lam.data_ptr()))
        _lib.check(self.lib.asp_space_norms(space, nrm.data_ptr()))
        _lib.check(self.lib.asp_ctx_synchronize(self.ctx))
        return lam, nrm

    def space_from_gathered(self, x, lam, nrm, n_total, shards, shard):
        """Space over the gathered rows of item shard `shard` of `shards` with imported lambdas / norms.  The library
        works on the tensor itself when it can (no second copy); the caller keeps `self.adopted` alive."""
        n_local, f = x.shape
        h = C.c_void_p()
        self.torch.cuda.current_stream(self.device).synchronize()
        if f % 4 == 0 and x.is_contiguous() and x.data_ptr() % 16 == 0:
            _lib.check(self.lib.asp_space_adopt_shard(self.ctx, x.data_ptr(), n_local, f, n_total, shards, shard, C.byref(h)))
            self.adopted = x
        else:
            _lib.check(self.lib.asp_space_create(self.ctx, x.data_ptr(), n_local, f, n_total, shards, shard, C.byref(h)))
            self.adopted = None
        _lib.check(self.lib.asp_space_import_lambdas(h, lam.contiguous().data_ptr(), nrm.contiguous().data_ptr()))
        return h

    def free_space(self, space):
        self.lib.asp_free_space(space)

    def device_rows(self, shard):
        """The caller's row shard as a contiguous device tensor (uploaded when it is host memory)."""
        t = self.torch
        if hasattr(shard, "data_ptr") and hasattr(shard, "is_cuda"):
            return shard.to(self.device).contiguous()
        return t.from_numpy(np.ascontiguousarray(shard, dtype=np.float64)).to(self.device)

    # ---- item graph
    def full_space(self, x_full):
        """world-1 space over all items (device tensor)."""
        n, f = x_full.shape
        h = C.c_void_p()
        self.torch.cuda.current_stream(self.device).synchronize()
        if f % 4 == 0 and x_full.is_contiguous() and x_full.data_ptr() % 16 == 0:
            # no second copy of the gathered matrix (C5: 54 GB per rank): the library works on the tensor itself,
            # which the ArrowSpace keeps alive (build_item_graph_sharded)
            _lib.check(self.lib.asp_space_adopt(self.ctx, x_full.data_ptr(), n, f, C.byref(h)))
            self.adopted = x_full
        else:
            _lib.check(self.lib.asp_space_create(self.ctx, x_full.data_ptr(), n, f, n, 1, 0, C.byref(h)))
            self.adopted = None
        return h

    def knn_rows(self, space, cgp, r0, r1, sw=None):
        """-> (idx int32[rows, kk], dist f64[rows, kk], cnt int32[rows]) device tensors."""
        t = self.torch
        rows = r1 - r0
        kmax = max(1, min(int(cgp.k), 30))
        idx = t.full((max(rows, 1), kmax), -1, dtype=t.int32, device=self.device)
        dist = t.zeros((max(rows, 1), kmax), dtype=t.float64, device=self.device)
        cnt = t.zeros((max(rows, 1),), dtype=t.int32, device=self.device)
        kk = C.c_int32(0)
        t.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_item_knn_rows(space, C.byref(cgp), C.byref(sw) if sw is not None else None, r0, r1,
                                              idx.data_ptr(), dist.data_ptr(), cnt.data_ptr(), C.byref(kk)))
        if kk.value != kmax:                       # k was capped at n - 1: the library wrote rows of kk entries
            idx = idx.reshape(-1)[: rows * kk.value].reshape(rows, kk.value)
            dist = dist.reshape(-1)[: rows * kk.value].reshape(rows, kk.value)
        return idx[:rows], dist[:rows], cnt[:rows]

    def graph_from_knn(self, n, idx, dist, cnt, cgp, sw):
        hg = C.c_void_p()
        idx, dist, cnt = idx.contiguous(), dist.contiguous(), cnt.contiguous()
        self.torch.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_graph_from_knn(self.ctx, n, idx.shape[1], idx.data_ptr(), dist.data_ptr(), cnt.data_ptr(),
                                               C.byref(cgp), C.byref(sw), C.byref(hg)))
        return hg

    # ---- hybrid search on row-sharded spaces
    def hybrid_pool(self, n_total, topk, pool):
        return self.lib.asp_hybrid_pool(int(n_total), int(topk), int(pool))

    def hybrid_shard(self, space, graph, q, tau, pool, idx, cos, score, lam, allowed=None, k=None):
        """asp_search_hybrid_shard of the host rows q into the device tensors idx / cos / score [rows, width] and lam [rows]
        (cos is None when the shortlist is the whole set).  allowed: the global item mask (this shard's rows are used).
        k: a per-call k in place of the graph's topk (asp_search_hybrid_shard_k)."""
        self.torch.cuda.current_stream(self.device).synchronize()      # the outputs were filled on torch's stream
        args = (space, graph, q.ctypes.data, q.shape[0], float(tau), int(pool), idx.data_ptr(),
                None if cos is None else cos.data_ptr(), score.data_ptr(), lam.data_ptr())
        if k is not None:
            bits = None
            if allowed is not None:
                n_local, row0 = C.c_int64(), C.c_int64()
                _lib.check(self.lib.asp_space_dims(space, C.byref(n_local), C.byref(C.c_int32()), C.byref(row0), C.byref(C.c_int64())))
                bits = pack_allowed(allowed, row0.value, n_local.value)
            _lib.check(self.lib.asp_search_hybrid_shard_k(*args[:6], int(k), *args[6:], None if bits is None else bits.ctypes.data))
        elif allowed is None:
            _lib.check(self.lib.asp_search_hybrid_shard(*args))
        else:
            n_local, row0 = C.c_int64(), C.c_int64()
            _lib.check(self.lib.asp_space_dims(space, C.byref(n_local), C.byref(C.c_int32()), C.byref(row0), C.byref(C.c_int64())))
            bits = pack_allowed(allowed, row0.value, n_local.value)
            _lib.check(self.lib.asp_search_hybrid_shard_filtered(*args, bits.ctypes.data))

    def hybrid_merge(self, idx, cos, score, m, topk):
        """[parts, nq, m] shortlists of the shards -> (idx, score) [nq, topk] device tensors (asp_hybrid_merge)."""
        t = self.torch
        parts, nq = idx.shape[0], idx.shape[1]
        out_idx = t.empty((nq, topk), dtype=t.int64, device=self.device)
        out_sc = t.empty((nq, topk), dtype=t.float64, device=self.device)
        idx, cos, score = idx.contiguous(), cos.contiguous(), score.contiguous()
        t.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_hybrid_merge(self.ctx, idx.data_ptr(), cos.data_ptr(), score.data_ptr(), parts, nq, m, topk,
                                             out_idx.data_ptr(), out_sc.data_ptr()))
        return out_idx, out_sc

    def topk_merge(self, idx, score):
        """[parts, nq, topk] lists -> (idx, score) [nq, topk] device tensors (asp_topk_merge)."""
        t = self.torch
        parts, nq, topk = idx.shape
        out_idx = t.empty((nq, topk), dtype=t.int64, device=self.device)
        out_sc = t.empty((nq, topk), dtype=t.float64, device=self.device)
        idx, score = idx.contiguous(), score.contiguous()
        t.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_topk_merge(self.ctx, idx.data_ptr(), score.data_ptr(), parts, nq, topk, out_idx.data_ptr(),
                                           out_sc.data_ptr()))
        return out_idx, out_sc

    # ---- range search
    def range_shard(self, space, graph, q, tau, min_score, allowed=None, max_hits=0):
        """asp_search_range_batch of the host rows q on this rank's item shard -> (idx, score) device tensors of the hits
        (GLOBAL indices, query-major, each query sorted), counts [rows] and lambda_q [rows] as host arrays."""
        t = self.torch
        nq = q.shape[0]
        counts = np.empty(nq, dtype=np.int64)
        lam = np.empty(nq, dtype=np.float64)
        bits = None
        if allowed is not None:
            n_local, row0 = C.c_int64(), C.c_int64()
            _lib.check(self.lib.asp_space_dims(space, C.byref(n_local), C.byref(C.c_int32()), C.byref(row0), C.byref(C.c_int64())))
            bits = pack_allowed(allowed, row0.value, n_local.value)
        h = C.c_void_p()
        _lib.check(self.lib.asp_search_range_batch(space, graph, q.ctypes.data, nq, float(tau), float(min_score),
                                                   None if bits is None else bits.ctypes.data, int(max_hits), counts.ctypes.data,
                                                   lam.ctypes.data, C.byref(h)))
        try:
            nnz = int(counts.sum())
            idx = t.empty(nnz, dtype=t.int64, device=self.device)
            score = t.empty(nnz, dtype=t.float64, device=self.device)
            _lib.check(self.lib.asp_range_result_fetch(h, idx.data_ptr(), score.data_ptr()))
        finally:
            self.lib.asp_range_result_free(h)
        return idx, score, counts, lam

    def range_merge(self, counts, idx, score):
        """counts [parts, nq] (host), the parts' hits concatenated (device tensors) -> the merged hits (asp_range_merge)."""
        t = self.torch
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        parts, nq = counts.shape
        total = int(counts.sum())
        out_idx = t.empty(total, dtype=t.int64, device=self.device)
        out_sc = t.empty(total, dtype=t.float64, device=self.device)
        idx, score = idx.contiguous(), score.contiguous()
        t.cuda.current_stream(self.device).synchronize()
        _lib.check(self.lib.asp_range_merge(self.ctx, parts, nq, counts.ctypes.data, idx.data_ptr(), score.data_ptr(),
                                            out_idx.data_ptr(), out_sc.data_ptr()))
        return out_idx, out_sc

    def to_comm(self, arr):
        return self.torch.from_numpy(arr).to(self.device)

    def from_comm(self, t):
        return t.cpu().numpy()

    def after_collective(self):
        """NCCL runs on torch's stream, the library on its own: order them before the next library call."""
        self.torch.cuda.current_stream(self.device).synchronize()


def _all_gather_blocks(t_local, world, group):
    """all-gather equal-size blocks; returns a tensor [world, *t_local.shape]."""
    dist = _dist()
    import torch
    out = torch.empty((world,) + tuple(t_local.shape), dtype=t_local.dtype, device=t_local.device)
    try:
        dist.all_gather_into_tensor(out, t_local.contiguous(), group=group)
    except (RuntimeError, NotImplementedError):
        parts = [torch.empty_like(t_local) for _ in range(world)]
        dist.all_gather(parts, t_local.contiguous(), group=group)
        out = torch.stack(parts)
    return out


def _gather_ragged_rows(t_local, world, group):
    """all-gather row blocks of different heights (same width), concatenated in rank order."""
    import torch
    if world == 1:
        return t_local
    cnt = torch.tensor([t_local.shape[0]], dtype=torch.int64, device=t_local.device)
    counts = [int(c) for c in _all_gather_blocks(cnt, world, group).reshape(-1).tolist()]
    if max(counts) == 0:
        return t_local
    return _all_gather_ragged(t_local, counts, group).contiguous()


def sharded_reduction(engine, shard, n_total, row0, cgp, sw, red, group=None):
    """SURVEY.md 8(f)-1 across ranks: every rank samples ITS rows (the hash runs on global row numbers), the kept rows
    are all-gathered (C4: 0.6 x 3.07 GB), and every rank runs the same deterministic two-NN / k-means / centroid-graph
    kernels on them -- replicas, no further collective; the result is the single-GPU one bit for bit.
    Returns (graph handle, centroid space handle, info dict)."""
    dist = _dist()
    world = dist.get_world_size(group)
    mine = engine.sampled_rows(shard, red, row0)
    rows = _gather_ragged_rows(mine, world, group)
    if rows.shape[0] == 0:                                   # an empty sample keeps every row
        import torch
        all_rows = shard if hasattr(shard, "is_cuda") else torch.from_numpy(np.ascontiguousarray(shard))
        rows = _gather_ragged_rows(all_rows.to(mine.device).contiguous(), world, group)
    if hasattr(engine, "after_collective"):
        engine.after_collective()
    whole = _lib.Reduction.from_buffer_copy(red)
    whole.sample_rate = 1.0                                  # `rows` IS the sample
    cspace, info = engine.reduce_rows(rows, whole, n_total)
    graph = engine.feature_graph(cspace, cgp, sw)
    return graph, cspace, info


def sharded_build(engine, shard, n_total, cgp, sw, group=None, reduction=None):
    """Steps 1-2 above + lambdas.  Returns (space handle, graph handle).  With `reduction` (an asp_reduction) the graph
    comes from the centroid matrix instead (sharded_reduction) and (space, graph, centroid space, info) is returned."""
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if _lib.GRAM_SEGMENTS % world != 0:
        raise ValueError("world size %d must divide %d" % (world, _lib.GRAM_SEGMENTS))
    f = shard.shape[1]
    space = engine.space_create(shard, n_total, world, rank)
    if reduction is not None:
        from . import api
        row0 = api.shard_rows(n_total, world, rank)[0]
        graph, cspace, info = sharded_reduction(engine, shard, n_total, row0, cgp, sw, reduction, group)
        engine.compute_lambdas(space, graph)
        return space, graph, cspace, info
    segs = engine.gram_partials(space, f)                        # [8, f, f], own blocks filled
    per = _lib.GRAM_SEGMENTS // world
    if world > 1:
        own = segs[rank * per:(rank + 1) * per]
        gathered = _all_gather_blocks(own, world, group)         # [world, per, f, f] == [8, f, f] in order
        segs = gathered.reshape(_lib.GRAM_SEGMENTS, f, f)
        if hasattr(engine, "after_collective"):
            engine.after_collective()
    pairs = np.empty((0, 2), dtype=np.int32)
    sums = np.empty((0, 3), dtype=np.float64)
    graph = None
    for _ in range(6):
        graph, need = engine.graph_from_gram(segs, f, n_total, cgp, sw, pairs if len(pairs) else None,
                                             sums if len(sums) else None)
        if graph is not None:
            break
        # left-to-right sums continue from rank to rank (every rank sees the same `need`)
        add = np.zeros((len(need), 3), dtype=np.float64)
        for r in range(world):
            if rank == r:
                add = engine.exact_pairs(space, np.ascontiguousarray(need), add)
            if world > 1:
                t = engine.to_comm(add)
                dist.broadcast(t, src=dist.get_global_rank(group, r) if group is not None else r, group=group)
                add = np.ascontiguousarray(engine.from_comm(t))
        pairs = np.ascontiguousarray(np.concatenate([pairs, need]))
        sums = np.ascontiguousarray(np.concatenate([sums, add]))
    if graph is None:
        raise RuntimeError("exact-pair resolution did not converge")
    engine.compute_lambdas(space, graph)
    return space, graph


_GRIDS = {}


def grid_layout(world, rank, item_shards):
    """R x C grid of the search: (R, C, item shard r, query slot c) of `rank`; ranks of one item shard are consecutive."""
    r_ = int(item_shards)
    if r_ < 1 or world % r_ != 0 or _lib.GRAM_SEGMENTS % r_ != 0:
        raise ValueError("item_shards = %d must divide the world size %d and %d" % (r_, world, _lib.GRAM_SEGMENTS))
    c_ = world // r_
    return r_, c_, rank // c_, rank % c_


def query_slice(nq, slots, slot):
    """Rows [a, b) of a batch of nq queries answered by query slot `slot` of `slots`; `per` = rows of a full slice."""
    per = (nq + slots - 1) // slots
    a = min(slot * per, nq)
    return a, min(a + per, nq), per


def grid_groups(world, item_shards):
    """Process groups of the grid, created collectively (every rank creates every group, in the same order) and cached:
    -> (item_groups[r] = the C ranks holding item shard r, merge_groups[c] = the R ranks answering query slot c)."""
    dist = _dist()
    key = (world, int(item_shards))
    if key not in _GRIDS:
        r_, c_, _, _ = grid_layout(world, 0, item_shards)
        item_groups = [dist.new_group([r * c_ + c for c in range(c_)]) if c_ > 1 else None for r in range(r_)]
        merge_groups = [dist.new_group([r * c_ + c for r in range(r_)]) if (r_ > 1 and c_ > 1) else None for c in range(c_)]
        _GRIDS[key] = (item_groups, merge_groups)
    return _GRIDS[key]


def auto_item_shards(world, n_total, f, free_bytes):
    """Fewest item shards whose share of the items (f64 rows + fp16 operands of both split terms + emission scratch)
    takes at most half of the free device memory: replicate when it fits, shard when it must."""
    for r_ in (1, 2, 4, 8):
        if r_ > world or world % r_:
            continue
        need = (n_total / r_) * (8.0 * f + 4.0 * (f + 64)) + 6e9
        if need <= 0.5 * free_bytes:
            return r_
    return world


def regroup(engine, space, rows_dev, n_total, item_shards, group=None):
    """Step 6 above.  `space` = this rank's build-time space (rows of asp_shard_rows(n_total, world, rank), lambdas computed),
    rows_dev = the same rows as a device tensor.  Returns (space over item shard r with imported lambdas, grid dict);
    the build-time space is freed."""
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    r_, c_, r, c = grid_layout(world, rank, item_shards)
    grid = dict(R=r_, C=c_, r=r, c=c, item_group=None, merge_group=None)
    if c_ == 1:
        grid["merge_group"] = group
        return space, grid
    if group is not None and group is not dist.group.WORLD:
        raise ValueError("item_shards < world needs the default process group")
    item_groups, merge_groups = grid_groups(world, r_)
    grid["item_group"], grid["merge_group"] = item_groups[r], merge_groups[c]
    lam, nrm = engine.lambdas_norms(space, rows_dev.shape[0])
    counts = [shard_rows(n_total, world, r * c_ + j) for j in range(c_)]
    counts = [b - a for a, b in counts]
    x = _all_gather_rows(rows_dev, counts, item_groups[r])
    lam = _all_gather_rows(lam, counts, item_groups[r])
    nrm = _all_gather_rows(nrm, counts, item_groups[r])
    if hasattr(engine, "after_collective"):
        engine.after_collective()
    new_space = engine.space_from_gathered(x, lam, nrm, n_total, r_, r)
    engine.free_space(space)
    return new_space, grid


def sharded_search_hybrid(engine, space, graph, queries, tau, pool, topk, n_total, grid, allowed=None, call_k=False):
    """Hybrid search (step 7) on an item-sharded grid (grid["R"] > 1), bit for bit the one-GPU search_hybrid_batch over all
    n_total items.  Called collectively with the same host batch `queries` [Q, F] on every rank.  Query slot c answers rows
    [a, b) of the batch: each of its R ranks computes its item shard's shortlist (engine.hybrid_shard), the R lists are
    all-gathered over the slot's merge group (R * m * 24 bytes per query) and merged on every one of them; the C slots then
    all-gather their finished slices, as the grid search does.  Returns (idx, score, lambda_q) host arrays of the whole
    batch on every rank.  A failure on any rank raises the same LibraryError (same code) on every rank.
    allowed: the global bool item mask, the same on every rank (each shard filters its own rows; the merges take the
    -1-padded lists as they are), or None.  call_k: topk is the caller's per-call k, not the graph's (engine.hybrid_shard
    gets k=topk, the merges take lists of that width)."""
    import torch
    from ._lib import LibraryError
    r_, c_ = grid["R"], grid["C"]
    nq = queries.shape[0]
    a, b, per = query_slice(nq, c_, grid["c"])
    m = engine.hybrid_pool(n_total, topk, pool)
    whole = m >= n_total                                     # no shortlist: the plain search's lists, merged as such
    width = topk if whole else m
    dev = engine.device
    nan = float("nan")
    idx = torch.full((per, width), -1, dtype=torch.int64, device=dev)
    cos = None if whole else torch.full((per, width), nan, dtype=torch.float64, device=dev)
    score = torch.full((per, width), nan, dtype=torch.float64, device=dev)
    lam = torch.full((per + 1,), nan, dtype=torch.float64, device=dev)
    lam[per] = 0.0                                           # the last element carries the status of this slot
    err = None
    if b > a:
        try:
            extra = {} if allowed is None else {"allowed": allowed}
            if call_k:
                extra["k"] = topk
            engine.hybrid_shard(space, graph, queries[a:b], tau, pool, idx[:b - a], None if whole else cos[:b - a],
                                score[:b - a], lam[:b - a], **extra)
        except LibraryError as e:
            err = e
    status = torch.tensor([float(err.code) if err is not None else 0.0], dtype=torch.float64, device=dev)
    status = _all_gather_blocks(status, r_, grid["merge_group"]).reshape(-1)
    g_idx = _all_gather_blocks(idx, r_, grid["merge_group"])
    g_sc = _all_gather_blocks(score, r_, grid["merge_group"])
    g_cos = None if whole else _all_gather_blocks(cos, r_, grid["merge_group"])
    if hasattr(engine, "after_collective"):
        engine.after_collective()
    bad = [float(s) for s in status.tolist() if s != 0.0]
    lam[per] = bad[0] if bad else 0.0
    out_idx = torch.full((per, topk), -1, dtype=torch.int64, device=dev)
    out_sc = torch.full((per, topk), nan, dtype=torch.float64, device=dev)
    if not bad and per > 0 and topk > 0:
        out_idx, out_sc = engine.topk_merge(g_idx, g_sc) if whole else engine.hybrid_merge(g_idx, g_cos, g_sc, m, topk)
    if c_ > 1:
        out_idx = _all_gather_blocks(out_idx, c_, grid["item_group"]).reshape(c_ * per, topk)
        out_sc = _all_gather_blocks(out_sc, c_, grid["item_group"]).reshape(c_ * per, topk)
        lam = _all_gather_blocks(lam, c_, grid["item_group"])
        if hasattr(engine, "after_collective"):
            engine.after_collective()
    lam = lam.reshape(c_, per + 1).cpu()
    codes = [int(cd) for cd in lam[:, per].tolist() if cd != 0]
    if codes:
        msg = err.message if err is not None and err.code == codes[0] else \
            "a rank of the query grid failed with error %d" % codes[0]
        raise LibraryError(codes[0], msg)
    return (out_idx[:nq].cpu().numpy(), out_sc[:nq].cpu().numpy(),
            np.ascontiguousarray(lam[:, :per].reshape(-1)[:nq].numpy()))


def _limit_message(total, query, max_hits):
    """The text of ASP_ERR_LIMIT, as asp_search_range_batch words it."""
    return "range search: %d hits reached at query %d, more than max_hits = %d" % (total, query, max_hits)


def sharded_search_range(engine, space, graph, queries, tau, min_score, n_total, grid, allowed=None, max_hits=1 << 26):
    """Range search (step 8) on the search grid of build_sharded, bit for bit the one-GPU search_range_batch over all n_total
    items.  Called collectively with the same host batch `queries` [Q, F] on every rank.  Query slot c answers rows [a, b):
    each of its R ranks runs its item shard (engine.range_shard); the slot's merge group all-gathers the per-query counts,
    then the ragged hits, and engine.range_merge orders them; the C slots all-gather their counts and finished slices.
    Every rank returns (indptr, idx, score, lambda_q) host arrays of the whole batch.  A failure on any rank -- the result
    cap (max_hits > 0: ASP_ERR_LIMIT, checked on every rank against the merged counts) and the panics included -- raises
    the same LibraryError code on every rank.  allowed: the global bool item mask, the same on every rank, or None."""
    import torch
    from ._lib import ASP_ERR_LIMIT, LibraryError
    r_, c_ = grid["R"], grid["C"]
    nq = queries.shape[0]
    a, b, per = query_slice(nq, c_, grid["c"])
    dev = engine.device
    counts = torch.zeros(per + 1, dtype=torch.int64)       # the last element carries this rank's status
    lam = torch.full((per,), float("nan"), dtype=torch.float64)
    idx = torch.empty(0, dtype=torch.int64, device=dev)
    score = torch.empty(0, dtype=torch.float64, device=dev)
    err = None
    if b > a:
        try:
            idx, score, cnt, lq = engine.range_shard(space, graph, queries[a:b], tau, min_score, allowed, max_hits)
            counts[:b - a] = torch.from_numpy(np.asarray(cnt, dtype=np.int64))
            lam[:b - a] = torch.from_numpy(np.asarray(lq, dtype=np.float64))
        except LibraryError as e:
            err = e
            counts[per] = e.code
    # counts and statuses first: every rank learns every failure and every count before any hit moves
    shard_counts = counts.to(dev)
    if r_ > 1:
        shard_counts = _all_gather_blocks(shard_counts, r_, grid["merge_group"])
    else:
        shard_counts = shard_counts.reshape(1, per + 1)
    if hasattr(engine, "after_collective"):
        engine.after_collective()
    shard_counts = shard_counts.cpu()
    slot = torch.zeros(per + 1, dtype=torch.float64)
    slot[:per] = shard_counts[:, :per].sum(dim=0).to(torch.float64)
    bad = [int(v) for v in shard_counts[:, per].tolist() if v != 0]
    slot[per] = bad[0] if bad else 0
    slot_lam = torch.cat([slot, lam])                       # [per + 1 counts / status | per lambda_q]
    if c_ > 1:
        all_slots = _all_gather_blocks(slot_lam.to(dev), c_, grid["item_group"])
        if hasattr(engine, "after_collective"):
            engine.after_collective()
        all_slots = all_slots.cpu()
    else:
        all_slots = slot_lam.reshape(1, -1)
    codes = [int(v) for v in all_slots[:, per].tolist() if v != 0]
    if codes:
        code = codes[0]
        if err is not None and err.code == code:
            raise LibraryError(code, err.message)
        msg = ("range search: more than max_hits = %d hits" % max_hits) if code == ASP_ERR_LIMIT else \
            "a rank of the query grid failed with error %d" % code
        raise LibraryError(code, msg)
    q_counts = all_slots[:, :per].reshape(-1)[:nq].to(torch.int64).numpy()
    lam_all = np.ascontiguousarray(all_slots[:, per + 1:].reshape(-1)[:nq].numpy())
    indptr = np.zeros(nq + 1, dtype=np.int64)
    np.cumsum(q_counts, out=indptr[1:])
    if max_hits > 0 and indptr[-1] > max_hits:                # the merged total: the same decision on every rank
        qi = int(np.searchsorted(indptr[1:], max_hits, side="right"))
        raise LibraryError(ASP_ERR_LIMIT, _limit_message(int(indptr[qi + 1]), qi, max_hits))
    # the slot's hits: ragged all-gather over its R ranks, merged into the one-GPU order
    if r_ > 1:
        per_rank = [int(v) for v in shard_counts[:, :per].sum(dim=1).tolist()]
        if sum(per_rank) > 0:
            g_idx = _all_gather_ragged(idx, per_rank, grid["merge_group"])
            g_sc = _all_gather_ragged(score, per_rank, grid["merge_group"])
            if hasattr(engine, "after_collective"):
                engine.after_collective()
            idx, score = engine.range_merge(shard_counts[:, :per].numpy(), g_idx, g_sc)
    # the C slots' finished slices
    if c_ > 1:
        per_slot = [int(v) for v in all_slots[:, :per].sum(dim=1).tolist()]
        if sum(per_slot) > 0:
            idx = _all_gather_ragged(idx, per_slot, grid["item_group"])
            score = _all_gather_ragged(score, per_slot, grid["item_group"])
            if hasattr(engine, "after_collective"):
                engine.after_collective()
    return indptr, idx.cpu().numpy(), score.cpu().numpy(), lam_all


def _all_gather_ragged(t_local, counts, group):
    """all-gather row blocks of different lengths (counts[r] rows on rank r) -> [sum(counts), ...]."""
    import torch
    world = len(counts)
    per = max(counts)
    pad = torch.zeros((per,) + tuple(t_local.shape[1:]), dtype=t_local.dtype, device=t_local.device)
    if t_local.shape[0]:
        pad[: t_local.shape[0]] = t_local
    g = _all_gather_blocks(pad, world, group)
    return torch.cat([g[r, : counts[r]] for r in range(world)], dim=0)


def _all_gather_rows(t_local, counts, group):
    """Row blocks of rank order -> [sum(counts), ...].  Equal blocks are gathered straight into the result (no padded
    staging, no concatenation: the gathered item matrix of C5 is 54 GB); ragged blocks take the padded route."""
    import torch
    if len(set(counts)) == 1 and t_local.is_contiguous():
        out = torch.empty((sum(counts),) + tuple(t_local.shape[1:]), dtype=t_local.dtype, device=t_local.device)
        try:
            _dist().all_gather_into_tensor(out, t_local, group=group)
            return out
        except (RuntimeError, NotImplementedError):
            del out
    return _all_gather_ragged(t_local, counts, group)


def sharded_item_graph(engine, shard, n_total, row0, cgp, sw, group=None):
    """Steps 4-5 above.  `shard` = rows [row0, row0 + len(shard)) of the item matrix as a tensor on the engine's
    device.  Returns (world-1 space handle over ALL items, graph handle over n_total nodes) -- identical on every rank."""
    dist = _dist()
    import torch
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    mine = torch.tensor([shard.shape[0], row0], dtype=torch.int64, device=shard.device)
    meta = _all_gather_blocks(mine, world, group).cpu().tolist()
    counts = [int(m[0]) for m in meta]
    starts = [int(m[1]) for m in meta]
    if sum(counts) != n_total or starts != [sum(counts[:r]) for r in range(world)]:
        raise ValueError("item shards must be contiguous row blocks in rank order (got starts %s, counts %s)" % (starts, counts))
    x_full = _all_gather_rows(shard, counts, group) if world > 1 else shard
    if hasattr(engine, "after_collective"):
        engine.after_collective()
    space = engine.full_space(x_full)
    idx, dst, cnt = engine.knn_rows(space, cgp, row0, row0 + counts[rank], sw)
    if world > 1:
        idx = _all_gather_rows(idx.contiguous(), counts, group)
        dst = _all_gather_rows(dst.contiguous(), counts, group)
        cnt = _all_gather_rows(cnt.contiguous(), counts, group)
        if hasattr(engine, "after_collective"):
            engine.after_collective()
    graph = engine.graph_from_knn(n_total, idx, dst, cnt, cgp, sw)
    return space, graph


def build_item_graph_sharded(graph_params, items_shard, n_total, row0, group=None, **extras):
    """Multi-GPU item graph: every rank passes its contiguous row block; returns (ArrowSpace over all items, GraphLaplacian
    over n_total nodes), the same on every rank."""
    from . import api
    import torch
    gp = api.parse_graph_params(graph_params) or dict(api.DEFAULT_GRAPH_PARAMS)
    cgp = _lib.make_params(gp["eps"], gp["k"], gp["topk"], gp["p"], gp["sigma"])
    sw = _lib.switches_from(extras)
    engine = CudaEngine(extras.get("device"))
    if not (hasattr(items_shard, "data_ptr") and items_shard.is_cuda):
        items_shard = torch.from_numpy(np.ascontiguousarray(items_shard, dtype=np.float64)).to(engine.device)
    dist = _dist()
    if group is None:
        group = dist.group.WORLD
    space, graph = sharded_item_graph(engine, items_shard.contiguous(), int(n_total), int(row0), cgp, sw, group)
    aspace = api.ArrowSpace._wrap(space, engine.ctx)
    aspace._keepalive = getattr(engine, "adopted", None)       # the adopted item matrix outlives the space handle
    return aspace, api.GraphLaplacian._wrap(graph)


def build_sharded(graph_params, items_shard, n_total, group=None, item_shards=None, **extras):
    """One process per GPU; every rank passes ITS rows (api.shard_rows).  The build is row-partitioned over all ranks.
    item_shards = R (a divisor of the world size; None = the fewest shards that fit the device memory) chooses the layout
    of the search: R item shards x world / R query slots (see `regroup`)."""
    from . import api
    import torch
    gp = api.parse_graph_params(graph_params) or dict(api.DEFAULT_GRAPH_PARAMS)
    cgp = _lib.make_params(gp["eps"], gp["k"], gp["topk"], gp["p"], gp["sigma"])
    sw = _lib.switches_from(extras)
    engine = CudaEngine(extras.get("device"))
    if not (hasattr(items_shard, "data_ptr") and items_shard.is_cuda):
        items_shard = np.ascontiguousarray(items_shard, dtype=np.float64)
    dist = _dist()
    if group is None:
        group = dist.group.WORLD
    world = dist.get_world_size(group)
    if item_shards is None:
        free_bytes, _ = torch.cuda.mem_get_info(engine.device)
        t = torch.tensor([float(free_bytes)], dtype=torch.float64, device=engine.device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)          # every rank must take the same decision
        item_shards = auto_item_shards(world, int(n_total), items_shard.shape[1], float(t.item()))
    grid_layout(world, 0, item_shards)                                  # validates
    rows_dev = engine.device_rows(items_shard) if item_shards < world else None
    reduction = extras.get("reduction")
    src = items_shard if rows_dev is None else rows_dev
    if reduction:
        space, graph, cspace, info = sharded_build(engine, src, int(n_total), cgp, sw, group, _lib.make_reduction(reduction))
    else:
        space, graph = sharded_build(engine, src, int(n_total), cgp, sw, group)
    space, grid = regroup(engine, space, rows_dev, int(n_total), item_shards, group)
    aspace = api.ArrowSpace._wrap(space, engine.ctx, grid["merge_group"] if grid["R"] > 1 else None, grid)
    aspace._keepalive = getattr(engine, "adopted", None)              # the adopted item matrix outlives the space handle
    gl = api.GraphLaplacian._wrap(graph)
    if reduction:
        gl.reduction = info
        gl._centroids = api.ArrowSpace._wrap(cspace, engine.ctx)
    return aspace, gl
