"""Host-side mirror of the reference's Python surface, over the C ABI.

Mirrors /root/reference/src/lib.rs (pyo3 module ``arrowspace``): same class names, method
names, argument order / keyword names, return shapes and error behaviour.

    ArrowSpaceBuilder.build(graph_params, items) -> (ArrowSpace, GraphLaplacian)   src/lib.rs:270-300
    ArrowSpace.search(item, gl, tau) -> [(index, score)]                           src/lib.rs:132-174
    ArrowSpace.nitems / nfeatures / get_item(idx) / lambdas()                      src/lib.rs:78-124
    GraphLaplacian.nnodes / shape() / graph_params                                 src/lib.rs:40-61
    set_debug(enabled)                                                             src/helpers.rs:12-21

Extensions (not in the reference): ``ArrowSpace.search_batch``, ``ArrowSpace.search_range`` /
``search_range_batch`` (every item at or above a score threshold), ``ArrowSpaceBuilder.build_sharded``
and device-tensor inputs (anything exposing ``data_ptr()``), used by bench.py.

Every numeric step runs in libarrowspace_b200.so (hand-written sm_100a CUDA).  There is no CPU
path: without the library or without a GPU the calls raise.
"""
import ctypes as C
import os
import sys

import numpy as np

from . import _lib
from ._lib import LibraryError

_DEBUG = False

# crate defaults when graph_params is None (GRAPH_VARIABLES.md:15: eps~1e-3, k~6, p=2, sigma=eps).
# topk has no documented default; 3 is the binding's doc-comment default (src/lib.rs:131).  [UNPINNED]
DEFAULT_GRAPH_PARAMS = {"eps": 1e-3, "k": 6, "topk": 3, "p": 2.0, "sigma": 1e-3}


LAST_CALL_TRACE = {}       # host-side wall times of the last search call (diagnostics: tools/latency.py)


class PanicException(BaseException):
    """Stand-in for pyo3_runtime.PanicException: the reference `.unwrap()`s / `assert_ne!`s inside
    build and search (src/lib.rs:156-159,277,279), which surfaces as a BaseException subclass."""


def set_debug(enabled):
    """Process-global debug flag; messages go to stderr with the reference's prefix (src/helpers.rs:12-21)."""
    global _DEBUG
    _DEBUG = bool(enabled)


def dbg_println(msg):
    if _DEBUG:
        sys.stderr.write("[pyarrowspace] %s\n" % msg)
        sys.stderr.flush()


def _is_device_tensor(x):
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda") and bool(x.is_cuda)


def _unwrap(exc):
    """What `Result::unwrap()` on a PyErr looks like from Python."""
    return PanicException(
        "called `Result::unwrap()` on an `Err` value: PyErr { type: <class '%s'>, value: %s(%r), traceback: None }"
        % (type(exc).__name__, type(exc).__name__, str(exc)))


def _check_allowed(allowed, nitems):
    """The `allowed=` argument of the searches: None, or a 1-D host numpy bool array of one entry per item."""
    if allowed is None:
        return None
    if not isinstance(allowed, np.ndarray) or allowed.dtype != np.bool_:
        raise TypeError("allowed must be a numpy.ndarray of bool (got %s)" % (
            "ndarray of %s" % allowed.dtype if isinstance(allowed, np.ndarray) else type(allowed).__name__))
    if allowed.ndim != 1 or allowed.shape[0] != nitems:
        raise ValueError("allowed must be 1-D with one entry per item (%d), got shape %s" % (nitems, allowed.shape))
    return allowed


# Longest per-call k: the list length the batched exact scan keeps per query (asp_xs::TOPK_MAX, asp_search_batch_k).
K_MAX = 1024


def _check_k(k):
    """The `k=` argument of the searches: None (the graph's topk, today's call), or an integer 1 <= k <= K_MAX."""
    if k is None:
        return None
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or k < 1:
        raise ValueError("k must be a positive integer (the number of results per query)")
    if k > K_MAX:
        raise LibraryError(_lib.ASP_ERR_UNSUPPORTED, "k = %d is beyond the %d results the exact scan keeps per query" % (k, K_MAX))
    return int(k)


def _check_taus(taus):
    """The `taus` argument of search_batch_taus: a non-empty list, tuple or 1-D numpy array of finite real numbers, in the
    caller's order (duplicates kept).  Returns a C-contiguous float64 array."""
    if isinstance(taus, np.ndarray):
        if taus.ndim != 1:
            raise ValueError("taus must be 1-D (got shape %s)" % (taus.shape,))
        if taus.dtype == np.bool_ or not (np.issubdtype(taus.dtype, np.integer) or np.issubdtype(taus.dtype, np.floating)):
            raise TypeError("taus must hold real numbers (got ndarray of %s)" % taus.dtype)
        vals = taus.astype(np.float64)
    elif isinstance(taus, (list, tuple)):
        for t in taus:
            if isinstance(t, (bool, np.bool_)) or not isinstance(t, (int, float, np.integer, np.floating)):
                raise TypeError("taus must hold real numbers (got %s)" % type(t).__name__)
        vals = np.array([float(t) for t in taus], dtype=np.float64)
    else:
        raise TypeError("taus must be a list, tuple or 1-D numpy.ndarray of real numbers (got %s)" % type(taus).__name__)
    if vals.size == 0:
        raise ValueError("taus must not be empty")
    if not np.isfinite(vals).all():
        raise ValueError("taus must be finite (got %s)" % vals.tolist())
    return np.ascontiguousarray(vals)


# Default cap of a range search: 2**26 hits, 1 GiB of results (int64 index + f64 score) -- a threshold far below the
# scores of a data set would otherwise ask for every item of every query.  max_results= raises or lowers it.
DEFAULT_MAX_RESULTS = 1 << 26


def _check_min_score(min_score):
    """min_score of a range search: a real number (inclusive, compared in f64; -inf = every item); NaN is refused."""
    if isinstance(min_score, bool) or not isinstance(min_score, (int, float, np.integer, np.floating)):
        raise TypeError("min_score must be a real number (got %s)" % type(min_score).__name__)
    v = float(min_score)
    if v != v:
        raise ValueError("min_score must not be NaN")
    return v


def _check_max_results(max_results):
    if max_results is None:
        return DEFAULT_MAX_RESULTS
    if isinstance(max_results, bool) or not isinstance(max_results, (int, np.integer)):
        raise TypeError("max_results must be an integer (got %s)" % type(max_results).__name__)
    if max_results < 1:
        raise ValueError("max_results must be at least 1 (got %d)" % max_results)
    return int(max_results)


def _range_error(e):
    """What a failed range search raises: the search's panics, ValueError for the result cap, else the LibraryError."""
    if e.code == _lib.ASP_ERR_LAMBDA_ZERO:
        return PanicException("assertion `left != right` failed: The lambdas are zero, check the magnitude of items and eps.\n"
                              "  left: 0.0\n right: 0.0")
    if e.code == _lib.ASP_ERR_ZERO_VECTOR:
        return PanicException(e.message)
    if e.code == _lib.ASP_ERR_LIMIT:
        return ValueError(e.message)
    return e


def parse_graph_params(graph_params):
    """src/helpers.rs:48-77: eps, k, topk, p required; sigma missing/None -> eps * 0.5."""
    if graph_params is None:
        return None
    if not isinstance(graph_params, dict):
        raise TypeError("argument 'graph_params': 'dict' object expected")
    out = {}
    for key, conv in (("eps", float), ("k", int), ("topk", int), ("p", float)):
        if key not in graph_params:
            raise ValueError("graph_params['%s'] is required" % key)
        v = graph_params[key]
        if conv is int:
            if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
                raise TypeError("'%s' object cannot be interpreted as an integer" % type(v).__name__)
            if v < 0:
                raise OverflowError("can't convert negative int to unsigned")
            out[key] = int(v)
        else:
            if not isinstance(v, (int, float, np.integer, np.floating)) or isinstance(v, bool):
                raise TypeError("argument '%s': must be real number, not %s" % (key, type(v).__name__))
            out[key] = float(v)
    sigma = graph_params.get("sigma")
    out["sigma"] = out["eps"] * 0.5 if sigma is None else float(sigma)
    return out


# EnergyParams::default() as documented by the binding (src/lib.rs:311-322); the struct itself is in the crate.
DEFAULT_ENERGY_PARAMS = {"optical_tokens": None, "trim_quantile": 0.1, "eta": 0.1, "steps": 4, "split_quantile": 0.9,
                         "neighbor_k": 8, "split_tau": 0.15, "w_lambda": 1.0, "w_disp": 0.5, "w_dirichlet": 0.25,
                         "candidate_m": 32}
_ENERGY_INT_KEYS = ("steps", "neighbor_k", "candidate_m")


def _extract_usize(v):
    """pyo3 `extract::<usize>()`: ints only (bool is an int subclass and is accepted by pyo3), negative -> OverflowError."""
    if not isinstance(v, (int, np.integer)):
        raise TypeError("'%s' object cannot be interpreted as an integer" % type(v).__name__)
    if v < 0:
        raise OverflowError("can't convert negative int to unsigned")
    return int(v)


def _extract_f64(v):
    """pyo3 `extract::<f64>()`: anything float() accepts through __float__ / __index__ (so ints and bools too)."""
    if isinstance(v, (str, bytes)) or not (hasattr(v, "__float__") or hasattr(v, "__index__")):
        raise TypeError("must be real number, not %s" % type(v).__name__)
    return float(v)


def parse_energy_params(energy_params):
    """src/energyparams.rs:6-45: start from EnergyParams::default(), overwrite the keys present in the dict (absent keys
    keep their default, unknown keys are ignored); optical_tokens is Option<usize> (None allowed), steps / neighbor_k /
    candidate_m are usize, the rest f64.  Extraction errors surface as the Python exceptions pyo3 raises."""
    out = dict(DEFAULT_ENERGY_PARAMS)
    if energy_params is None:
        return out
    if not isinstance(energy_params, dict):
        raise TypeError("argument 'energy_params': 'dict' object expected")
    for key in DEFAULT_ENERGY_PARAMS:
        if key not in energy_params:
            continue
        v = energy_params[key]
        if key == "optical_tokens":
            out[key] = None if v is None else _extract_usize(v)
        elif key in _ENERGY_INT_KEYS:
            out[key] = _extract_usize(v)
        else:
            out[key] = _extract_f64(v)
    return out


class GraphLaplacian:
    """Opaque handle of the feature-graph Laplacian (CSR on the device) + its parameters."""

    def __new__(cls, *a, **k):
        raise ValueError("GraphLaplacian cannot be constructed directly; use ArrowSpaceBuilder.build_with_graph")

    @classmethod
    def _wrap(cls, handle):
        self = object.__new__(cls)
        self._h = handle
        self.reduction = None            # extension: outcome of the pre-graph reduction (ArrowSpaceBuilder.build(reduction=))
        self._centroids = None
        return self

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and _lib is not None and getattr(_lib, "_lib", None) is not None:
            _lib._lib.asp_free_graph(h)
            self._h = None

    def centroids(self):
        """Extension: the n_clusters x nfeatures centroid matrix the graph was built on (None without reduction=)."""
        if self._centroids is None:
            return None
        return persist_items(self._centroids)

    def _info(self):
        n, nnz, gp = C.c_int64(), C.c_int64(), _lib.GraphParams()
        _lib.check(_lib.load().asp_graph_info(self._h, C.byref(n), C.byref(nnz), C.byref(gp)))
        return n.value, nnz.value, gp

    @property
    def nnodes(self):
        return self._info()[0]

    def shape(self):
        n = self._info()[0]
        return (n, n)

    @property
    def graph_params(self):
        gp = self._info()[2]
        return {"eps": gp.eps, "k": gp.k, "topk": gp.topk, "p": gp.p, "sigma": gp.sigma}

    # -- extension: parity export
    @property
    def nnz(self):
        return self._info()[1]

    def csr(self):
        """(indptr int64[nnodes+1], indices int32[nnz], data f64[nnz]) of L = D - W."""
        n, nnz, _ = self._info()
        indptr = np.empty(n + 1, dtype=np.int64)
        indices = np.empty(nnz, dtype=np.int32)
        data = np.empty(nnz, dtype=np.float64)
        _lib.check(_lib.load().asp_graph_csr(self._h, indptr.ctypes.data, indices.ctypes.data, data.ctypes.data))
        return indptr, indices, data

    def edges(self):
        """Sorted (a, b), a < b, W_ab > 0."""
        indptr, indices, data = self.csr()
        rows = np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr))
        keep = (indices > rows) & (data < 0.0)
        return np.stack([rows[keep], indices[keep].astype(np.int64)], axis=1)


class ArrowSpace:
    """Device-resident items (row shard) + per-item taumode lambdas."""

    def __new__(cls, *a, **k):
        raise ValueError("ArrowSpace cannot be constructed directly; use ArrowSpaceBuilder.build")

    @classmethod
    def _wrap(cls, handle, ctx, group=None, grid=None):
        self = object.__new__(cls)
        self._h = handle
        self._ctx = ctx
        self._group = group          # torch.distributed group the per-shard results are merged over (item shards > 1), else None
        self._grid = grid            # multi-GPU layout (distributed.regroup): R item shards x C query slots
        return self

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and _lib is not None and getattr(_lib, "_lib", None) is not None:
            _lib._lib.asp_free_space(h)
            self._h = None

    def _dims(self):
        n, f, r0, nt = C.c_int64(), C.c_int32(), C.c_int64(), C.c_int64()
        _lib.check(_lib.load().asp_space_dims(self._h, C.byref(n), C.byref(f), C.byref(r0), C.byref(nt)))
        return n.value, f.value, r0.value, nt.value

    @property
    def nitems(self):
        return self._dims()[3]

    @property
    def nfeatures(self):
        return self._dims()[1]

    @property
    def nitems_local(self):
        return self._dims()[0]

    @property
    def row_offset(self):
        return self._dims()[2]

    def get_item(self, idx):
        """(features ndarray[f64, F], lambda) -- src/lib.rs:100-120.  Sharded spaces: local rows only."""
        if isinstance(idx, bool) or not isinstance(idx, (int, np.integer)):
            raise TypeError("argument 'idx': '%s' object cannot be interpreted as an integer" % type(idx).__name__)
        if idx < 0:
            raise OverflowError("can't convert negative int to unsigned")
        n_local, f, row0, n_total = self._dims()
        if idx >= n_total:
            raise ValueError("index %d out of range [0, %d)" % (idx, n_total))
        local = idx - row0
        if local < 0 or local >= n_local:
            raise ValueError("index %d is not on this rank (rows [%d, %d))" % (idx, row0, row0 + n_local))
        feats = np.empty(f, dtype=np.float64)
        lam = C.c_double()
        _lib.check(_lib.load().asp_space_get_item(self._h, local, feats.ctypes.data, C.byref(lam)))
        return feats, lam.value

    def lambdas(self):
        """New ndarray[f64] of the per-item lambdas (src/lib.rs:122-124); sharded: this rank's rows."""
        out = np.empty(self._dims()[0], dtype=np.float64)
        _lib.check(_lib.load().asp_space_lambdas(self._h, out.ctypes.data))
        return out

    def norms(self):
        out = np.empty(self._dims()[0], dtype=np.float64)
        _lib.check(_lib.load().asp_space_norms(self._h, out.ctypes.data))
        return out

    # ------------------------------------------------------------------ search
    def search(self, item, gl, tau):
        """list[(index, score)], best first, length min(topk, nitems) -- src/lib.rs:132-174.  (The reference's signature;
        a filtered single query is search_batch(item.reshape(1, -1), gl, tau, allowed=mask).)"""
        if not isinstance(gl, GraphLaplacian):
            raise TypeError("argument 'gl': 'GraphLaplacian' object expected")
        if not isinstance(item, np.ndarray) or item.dtype != np.float64 or item.ndim != 1:
            raise TypeError("argument 'item': expected 1-D numpy.ndarray of float64")
        if not item.flags.c_contiguous:
            raise ValueError("The given array is not contiguous")           # as_slice()? src/lib.rs:139
        if item.shape[0] != self.nfeatures:
            raise ValueError("query length %d must match nfeatures %d" % (item.shape[0], self.nfeatures))
        tau = float(tau)
        idx, score, lam_q = self._search_batch(item.reshape(1, -1), gl, tau, want_lambda=True)
        dbg_println("search: qlen=%d, lambda_q=%.6f" % (item.shape[0], lam_q[0]))
        return [(int(i), float(s)) for i, s in zip(idx[0], score[0]) if i >= 0]

    def search_batch(self, queries, gl, tau, out=None, *, allowed=None, k=None):
        """Extension: (idx int64[Q, topk], score f64[Q, topk]); rows padded with -1 / NaN.
        out = (idx, score) host arrays to fill (C-contiguous, right shapes / dtypes; e.g. pinned memory that the caller
        reuses from call to call: the device -> host read then runs at the PCIe rate instead of the page-fault rate of
        freshly allocated memory).  Host query batches only.
        allowed = numpy bool[nitems] (keyword only): per query the best topk among the allowed items, padded with -1 / NaN
        when fewer are allowed; the same mask for every query.  Collective calls: every rank passes the same mask.
        k = int (keyword only, 1 .. 1024): k results per query instead of gl.graph_params["topk"] (no rebuild; the answer is
        the one a graph of topk = k gives, bit for bit); out shapes are then (Q, k).  k = None is the graph's topk."""
        allowed = _check_allowed(allowed, self.nitems)
        k = _check_k(k)
        if out is not None:
            topk = gl.graph_params["topk"] if k is None else k
            nq = queries.shape[0]
            oi, os_ = out
            if not (isinstance(oi, np.ndarray) and isinstance(os_, np.ndarray) and oi.dtype == np.int64 and os_.dtype == np.float64
                    and oi.shape == (nq, topk) and os_.shape == (nq, topk) and oi.flags.c_contiguous and os_.flags.c_contiguous):
                raise ValueError("out must be (int64[%d, %d], float64[%d, %d]) C-contiguous host arrays" % (nq, topk, nq, topk))
            if _is_device_tensor(queries):
                raise ValueError("out= is for host query batches (device batches return device tensors)")
        idx, score, _ = self._search_batch(queries, gl, float(tau), want_lambda=False, out=out, allowed=allowed, k=k)
        return idx, score

    def search_batch_taus(self, queries, gl, taus, *, allowed=None, k=None):
        """Extension: the same queries at several taus.  Returns (idx int64[T, Q, k], score f64[T, Q, k]) where T = len(taus)
        and k is the call's k or gl.graph_params["topk"]; idx[t], score[t] are, bit for bit, search_batch(queries, gl,
        taus[t], allowed=allowed, k=k), -1 / NaN padding included.  taus: a list, tuple or 1-D ndarray of finite real
        numbers (duplicates allowed).  lambda_q is computed once, with search_batch's panics.  On one GPU the taus that take
        the tensor-core candidate pass with k <= 16 share one pass per group of up to 3; on multi-GPU layouts the call loops
        over the collective search_batch.  Host batches return numpy arrays, device float64 batches device tensors."""
        taus = _check_taus(taus)
        allowed = _check_allowed(allowed, self.nitems)
        k = _check_k(k)
        if self._group is not None or (self._grid is not None and self._grid["C"] > 1):
            outs = [self.search_batch(queries, gl, float(t), allowed=allowed, k=k) for t in taus]
            if _is_device_tensor(outs[0][0]):
                import torch
                return torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs])
            return np.stack([o[0] for o in outs]), np.stack([o[1] for o in outs])
        lib = _lib.load()
        f = self.nfeatures
        topk = gl.graph_params["topk"] if k is None else k
        ntau = taus.shape[0]
        if _is_device_tensor(queries):
            if queries.dim() != 2 or queries.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (queries.shape[-1], f))
            import torch
            q = queries.contiguous()
            if q.dtype != torch.float64:
                raise TypeError("queries must be float64")
            nq = q.shape[0]
            idx = torch.empty((ntau, nq, topk), dtype=torch.int64, device=q.device)
            score = torch.empty((ntau, nq, topk), dtype=torch.float64, device=q.device)
            qp, ip, sp = q.data_ptr(), idx.data_ptr(), score.data_ptr()
            torch.cuda.current_stream(q.device).synchronize()      # the library runs on its own stream
        else:
            q = np.ascontiguousarray(queries, dtype=np.float64)
            if q.ndim != 2 or q.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (q.shape[-1], f))
            nq = q.shape[0]
            idx = np.empty((ntau, nq, topk), dtype=np.int64)
            score = np.empty((ntau, nq, topk), dtype=np.float64)
            qp, ip, sp = q.ctypes.data, idx.ctypes.data, score.ctypes.data
        bits = self._allowed_bits(allowed)
        try:
            _lib.check(lib.asp_search_batch_taus(self._h, gl._h, qp, nq, taus.ctypes.data, ntau, topk, ip, sp, None,
                                                 None if bits is None else bits.ctypes.data))
        except LibraryError as e:
            if e.code == _lib.ASP_ERR_LAMBDA_ZERO:                          # src/lib.rs:156-159
                raise PanicException("assertion `left != right` failed: %s\n  left: 0.0\n right: 0.0" % e.message)
            if e.code == _lib.ASP_ERR_ZERO_VECTOR:
                raise PanicException(e.message)
            raise
        return idx, score

    def _allowed_bits(self, allowed):
        """This rank's slice of the mask, packed for the library (None: no filter)."""
        if allowed is None:
            return None
        from .distributed import pack_allowed
        n_local, _, row0, _ = self._dims()
        return pack_allowed(allowed, row0, n_local)

    def _search_batch(self, queries, gl, tau, want_lambda, out=None, allowed=None, k=None):
        import time
        if self._grid is not None and self._grid["C"] > 1:
            return self._search_batch_grid(queries, gl, tau, out, allowed, k)
        t_a = time.perf_counter()
        lib = _lib.load()
        f = self.nfeatures
        topk = gl.graph_params["topk"] if k is None else k
        host_in = not _is_device_tensor(queries)
        host_out, toucher = None, None
        if host_in and self._group is not None:
            # sharded space, host queries: every rank uploads 1/world of the batch over its own PCIe link and the
            # shards are all-gathered over NVLink (each rank scores ALL queries against its item shard)
            q_np = np.ascontiguousarray(queries, dtype=np.float64)
            if q_np.ndim != 2 or q_np.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (q_np.shape[-1], f))
            queries = _upload_queries_sharded(self, q_np)
            if out is not None:
                host_out = (out[0], out[1], np.empty(q_np.shape[0], dtype=np.float64))
            elif q_np.shape[0] * max(topk, 1) >= 65536:
                # result arrays for the caller: freshly allocated pageable memory page-faults on first touch (~3 GB/s, 3 ms
                # for 64k x 10 results).  A helper thread touches them while this thread sits in the library (ctypes drops
                # the GIL), so the final D2H copy lands in resident pages.
                import threading
                host_out = (np.empty((q_np.shape[0], topk), dtype=np.int64), np.empty((q_np.shape[0], topk), dtype=np.float64),
                            np.empty(q_np.shape[0], dtype=np.float64))
                toucher = threading.Thread(target=lambda: [a.fill(0) for a in host_out])
                toucher.start()
        if _is_device_tensor(queries):
            if queries.dim() != 2 or queries.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (queries.shape[-1], f))
            import torch
            q = queries.contiguous()
            if q.dtype != torch.float64:
                raise TypeError("queries must be float64")
            nq = q.shape[0]
            idx = torch.empty((nq, topk), dtype=torch.int64, device=q.device)
            score = torch.empty((nq, topk), dtype=torch.float64, device=q.device)
            lam = torch.empty(nq, dtype=torch.float64, device=q.device)
            qp, ip, sp, lp = q.data_ptr(), idx.data_ptr(), score.data_ptr(), lam.data_ptr()
            torch.cuda.current_stream(q.device).synchronize()      # the library runs on its own stream
        else:
            q = np.ascontiguousarray(queries, dtype=np.float64)
            if q.ndim != 2 or q.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (q.shape[-1], f))
            nq = q.shape[0]
            idx = out[0] if out is not None else np.empty((nq, topk), dtype=np.int64)
            score = out[1] if out is not None else np.empty((nq, topk), dtype=np.float64)
            lam = np.empty(nq, dtype=np.float64)
            qp, ip, sp, lp = q.ctypes.data, idx.ctypes.data, score.ctypes.data, lam.ctypes.data
        bits = self._allowed_bits(allowed)
        t_b = time.perf_counter()
        try:
            if k is not None:
                _lib.check(lib.asp_search_batch_k(self._h, gl._h, qp, nq, tau, k, ip, sp, lp, None if bits is None else bits.ctypes.data))
            elif bits is None:
                _lib.check(lib.asp_search_batch(self._h, gl._h, qp, nq, tau, ip, sp, lp))
            else:
                _lib.check(lib.asp_search_batch_filtered(self._h, gl._h, qp, nq, tau, ip, sp, lp, bits.ctypes.data))
            LAST_CALL_TRACE["prepare_ms"] = (t_b - t_a) * 1e3
            LAST_CALL_TRACE["library_ms"] = (time.perf_counter() - t_b) * 1e3
        except LibraryError as e:
            if e.code == _lib.ASP_ERR_LAMBDA_ZERO:                          # src/lib.rs:156-159
                raise PanicException("assertion `left != right` failed: %s\n  left: 0.0\n right: 0.0" % e.message)
            if e.code == _lib.ASP_ERR_ZERO_VECTOR:
                raise PanicException(e.message)
            raise
        if self._group is not None:
            idx, score = _merge_across_ranks(self, idx, score, nq, topk)
        if toucher is not None:
            toucher.join()                                              # before anything is written into host_out
        if host_in and _is_device_tensor(idx):
            idx, score, lam = _to_host(idx, host_out and host_out[0]), _to_host(score, host_out and host_out[1]), \
                _to_host(lam, host_out and host_out[2])
        return idx, score, lam

    def _search_batch_grid(self, queries, gl, tau, out=None, allowed=None, k=None):
        """R item shards x C query slots (distributed.regroup): this rank answers rows [a, b) of the batch against its item
        shard; R > 1: the R ranks of the slot merge their lists (K5); the C slots all-gather the finished slices, so every
        rank returns the whole batch.  Host batches: this rank uploads only ITS slice (over its own PCIe link)."""
        import threading
        import torch
        import torch.distributed as dist
        from .distributed import query_slice
        lib = _lib.load()
        g = self._grid
        f = self.nfeatures
        topk = gl.graph_params["topk"] if k is None else k
        dev = torch.device("cuda", lib.asp_ctx_device(self._ctx))
        host_in = not _is_device_tensor(queries)
        if host_in:
            q = np.ascontiguousarray(queries, dtype=np.float64)
            if q.ndim != 2 or q.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (q.shape[-1], f))
        else:
            if queries.dim() != 2 or queries.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (queries.shape[-1], f))
            q = queries.contiguous()
            if q.dtype != torch.float64:
                raise TypeError("queries must be float64")
        nq = q.shape[0]
        a, b, per = query_slice(nq, g["C"], g["c"])
        host_out, toucher = None, None
        if host_in and out is not None:
            host_out = (out[0], out[1], np.empty(nq, dtype=np.float64))
        elif host_in and nq * max(topk, 1) >= 65536:    # first touch of the caller's result pages while the kernels run
            host_out = (np.empty((nq, topk), dtype=np.int64), np.empty((nq, topk), dtype=np.float64), np.empty(nq, dtype=np.float64))
            toucher = threading.Thread(target=lambda: [arr.fill(0) for arr in host_out])
            toucher.start()
        # this slot's slice, padded to `per` rows; lam carries one extra element: this rank's status, so that every rank
        # raises the same error
        idx_p = torch.full((per, topk), -1, dtype=torch.int64, device=dev)
        sc_p = torch.full((per, topk), float("nan"), dtype=torch.float64, device=dev)
        lam_p = torch.full((per + 1,), float("nan"), dtype=torch.float64, device=dev)
        lam_p[per] = 0.0
        err = None
        if b > a:
            qp = q[a:b].ctypes.data if host_in else q[a:b].data_ptr()
            torch.cuda.current_stream(dev).synchronize()                 # the library runs on its own stream
            bits = self._allowed_bits(allowed)
            if k is not None:
                rc = lib.asp_search_batch_k(self._h, gl._h, qp, b - a, tau, k, idx_p.data_ptr(), sc_p.data_ptr(), lam_p.data_ptr(),
                                            None if bits is None else bits.ctypes.data)
            elif bits is None:
                rc = lib.asp_search_batch(self._h, gl._h, qp, b - a, tau, idx_p.data_ptr(), sc_p.data_ptr(), lam_p.data_ptr())
            else:
                rc = lib.asp_search_batch_filtered(self._h, gl._h, qp, b - a, tau, idx_p.data_ptr(), sc_p.data_ptr(),
                                                   lam_p.data_ptr(), bits.ctypes.data)
            if rc != _lib.ASP_OK:
                msg = lib.asp_last_error()
                err = LibraryError(rc, msg.decode("utf-8", "replace") if msg else "unknown error")
                lam_p[per] = float(rc)
        if g["R"] > 1:
            idx_p, sc_p = _merge_across_ranks(self, idx_p, sc_p, per, topk)
        idx = torch.empty((g["C"] * per, topk), dtype=torch.int64, device=dev)
        score = torch.empty((g["C"] * per, topk), dtype=torch.float64, device=dev)
        lam = torch.empty((g["C"] * (per + 1),), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(idx, idx_p, group=g["item_group"])
        dist.all_gather_into_tensor(score, sc_p, group=g["item_group"])
        dist.all_gather_into_tensor(lam, lam_p, group=g["item_group"])
        lam = lam.view(g["C"], per + 1)
        codes = lam[:, per].cpu().tolist()
        if toucher is not None:
            toucher.join()
        bad = [int(cd) for cd in codes if cd != 0]
        if bad:
            code = bad[0]
            message = err.message if err is not None else ("a rank of the query grid failed with error %d" % code)
            if code == _lib.ASP_ERR_LAMBDA_ZERO:
                raise PanicException("assertion `left != right` failed: The lambdas are zero, check the magnitude of items and eps.\n  left: 0.0\n right: 0.0")
            if code == _lib.ASP_ERR_ZERO_VECTOR:
                raise PanicException(message)
            raise LibraryError(code, message)
        idx, score, lam = idx[:nq], score[:nq], lam[:, :per].reshape(-1)[:nq]
        if host_in:
            return (_to_host(idx, host_out and host_out[0]), _to_host(score, host_out and host_out[1]),
                    _to_host(lam.contiguous(), host_out and host_out[2]))
        return idx, score, lam.contiguous()

    # ------------------------------------------------------------------ range search (extension)
    def search_range(self, item, gl, tau, min_score):
        """list[(index, score)] of EVERY item with score >= min_score, best first (score desc, index asc).  Same argument
        checks, lambda_q and panics as `search`; a filtered single query is search_range_batch(item.reshape(1, -1), ...)."""
        if not isinstance(gl, GraphLaplacian):
            raise TypeError("argument 'gl': 'GraphLaplacian' object expected")
        if not isinstance(item, np.ndarray) or item.dtype != np.float64 or item.ndim != 1:
            raise TypeError("argument 'item': expected 1-D numpy.ndarray of float64")
        if not item.flags.c_contiguous:
            raise ValueError("The given array is not contiguous")
        if item.shape[0] != self.nfeatures:
            raise ValueError("query length %d must match nfeatures %d" % (item.shape[0], self.nfeatures))
        indptr, idx, score = self.search_range_batch(item.reshape(1, -1), gl, tau, min_score)
        return [(int(i), float(s)) for i, s in zip(idx, score)]

    def search_range_batch(self, queries, gl, tau, min_score, *, allowed=None, max_results=None):
        """Range search: per query every item whose score (the search's, evaluated in the reference order) is >= min_score,
        ordered by (score desc, index asc).  Returns CSR (indptr int64[Q + 1], idx int64[nnz], score f64[nnz]): the hits of
        query q are idx[indptr[q]:indptr[q + 1]].  Host batches return numpy arrays, device batches device tensors.
        min_score: inclusive, compared in f64; -inf returns every item, > 1 empty rows, NaN raises ValueError.
        allowed = numpy bool[nitems]: only allowed items are hits (collective calls: the same mask on every rank).
        max_results: the cap on the total number of hits of the call (default DEFAULT_MAX_RESULTS = 2**26, 1 GiB of
        results); more raises ValueError stating the count.  lambda_q == 0 and zero vectors panic as in `search`.
        Row-sharded spaces (build_sharded) are called collectively and every rank returns the whole batch."""
        if not isinstance(gl, GraphLaplacian):
            raise TypeError("argument 'gl': 'GraphLaplacian' object expected")
        min_score = _check_min_score(min_score)
        max_hits = _check_max_results(max_results)
        tau = float(tau)
        n_local, f, _, n_total = self._dims()
        allowed = _check_allowed(allowed, n_total)
        device_in = _is_device_tensor(queries)
        if device_in:
            import torch
            if queries.dim() != 2 or queries.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (queries.shape[-1], f))
            if queries.dtype != torch.float64:
                raise TypeError("queries must be float64")
        else:
            queries = np.ascontiguousarray(queries, dtype=np.float64)
            if queries.ndim != 2 or queries.shape[1] != f:
                raise ValueError("query length %d must match nfeatures %d" % (queries.shape[-1], f))
        if self._grid is not None:
            from .distributed import CudaEngine, sharded_search_range
            engine = CudaEngine(_lib.load().asp_ctx_device(self._ctx))
            q_host = queries.cpu().numpy() if device_in else queries
            try:
                indptr, idx, score, _ = sharded_search_range(engine, self._h, gl._h, q_host, tau, min_score, n_total, self._grid,
                                                             allowed=allowed, max_hits=max_hits)
            except LibraryError as e:
                raise _range_error(e)
            if device_in:
                import torch
                return tuple(torch.from_numpy(a).to(queries.device) for a in (indptr, idx, score))
            return indptr, idx, score
        if n_local != n_total:
            raise NotImplementedError("search_range on a row shard needs the search grid of build_sharded")
        return self._search_range_local(queries, gl, tau, min_score, allowed, max_hits, device_in)

    def _search_range_local(self, queries, gl, tau, min_score, allowed, max_hits, device_in):
        lib = _lib.load()
        nq = queries.shape[0]
        counts = np.empty(nq, dtype=np.int64)
        lam = np.empty(nq, dtype=np.float64)
        if device_in:
            import torch
            q = queries.contiguous()
            qp = q.data_ptr()
            torch.cuda.current_stream(q.device).synchronize()      # the library runs on its own stream
        else:
            qp = queries.ctypes.data
        bits = self._allowed_bits(allowed)
        h = C.c_void_p()
        try:
            _lib.check(lib.asp_search_range_batch(self._h, gl._h, qp, nq, tau, min_score, None if bits is None else bits.ctypes.data,
                                                  max_hits, counts.ctypes.data, lam.ctypes.data, C.byref(h)))
        except LibraryError as e:
            raise _range_error(e)
        try:
            indptr = np.zeros(nq + 1, dtype=np.int64)
            np.cumsum(counts, out=indptr[1:])
            nnz = int(indptr[-1])
            if device_in:
                import torch
                idx = torch.empty(nnz, dtype=torch.int64, device=q.device)
                score = torch.empty(nnz, dtype=torch.float64, device=q.device)
                _lib.check(lib.asp_range_result_fetch(h, idx.data_ptr(), score.data_ptr()))
                return torch.from_numpy(indptr).to(q.device), idx, score
            idx = np.empty(nnz, dtype=np.int64)
            score = np.empty(nnz, dtype=np.float64)
            _lib.check(lib.asp_range_result_fetch(h, idx.ctypes.data, score.ctypes.data))
            return indptr, idx, score
        finally:
            lib.asp_range_result_free(h)

    # ------------------------------------------------------------------ persistence (extension, SURVEY.md 8(f)-4)
    def save(self, path, gl, items=None):
        """Write this space and its graph to `path` (.npz); ArrowSpaceBuilder.load restores the pair without rebuilding."""
        from . import persist
        return persist.save(path, self, gl, items)

    # ------------------------------------------------------------------ hybrid search (SURVEY.md 8(f)-2)
    def search_hybrid(self, item, gl, tau, *, pool=None, allowed=None, k=None):
        """list[(index, score)], best first -- src/lib.rs:182-219: same argument checks and lambda_q as `search`, no
        lambda_q != 0 assertion, k = gl.graph_params.topk, then the crate's search_lambda_aware_hybrid.  That function is not
        in the reference (PARITY UNPINNED): restated as a cosine shortlist of `pool` items (keyword-only extra, default
        min(2 * topk, 31)) re-ranked by the lambda-aware score (include/arrowspace_b200.h, asp_search_hybrid_batch).
        allowed (keyword only, numpy bool[nitems]): the shortlist is the `pool` ALLOWED items of largest cosine.
        k (keyword only): k results instead of gl.graph_params["topk"], as in search_hybrid_batch."""
        if not isinstance(gl, GraphLaplacian):
            raise TypeError("argument 'gl': 'GraphLaplacian' object expected")
        if not isinstance(item, np.ndarray) or item.dtype != np.float64 or item.ndim != 1:
            raise TypeError("argument 'item': expected 1-D numpy.ndarray of float64")
        if not item.flags.c_contiguous:
            raise ValueError("The given array is not contiguous")           # as_slice()? src/lib.rs:189
        if item.shape[0] != self.nfeatures:
            raise ValueError("query length %d must match nfeatures %d" % (item.shape[0], self.nfeatures))   # src/lib.rs:190-196
        idx, score, lam_q = self.search_hybrid_batch(item.reshape(1, -1), gl, float(tau), pool=pool, want_lambda=True,
                                                     allowed=allowed, k=k)
        dbg_println("search: qlen=%d, lambda_q=%.6f" % (item.shape[0], lam_q[0]))     # src/lib.rs:207-211 (same text as search)
        return [(int(i), float(s)) for i, s in zip(idx[0], score[0]) if i >= 0]

    def search_hybrid_batch(self, queries, gl, tau, *, pool=None, want_lambda=False, allowed=None, k=None):
        """Extension: search_hybrid for a host batch; (idx int64[Q, topk], score f64[Q, topk]) padded with -1 / NaN
        (+ lambda_q with want_lambda).  On one GPU, and on the replicated layout of build_sharded (item_shards = 1), each
        rank answers on its own.  On an item-sharded space (item_shards > 1) it is called collectively, like `search`, and
        every rank returns the whole batch: the one-GPU answer, bit for bit (distributed.sharded_search_hybrid).
        allowed = numpy bool[nitems]: H2's shortlist is taken from the allowed items only (the pool length is unchanged);
        collective calls pass the same mask on every rank.
        k = int (1 .. 1024): k replaces gl.graph_params["topk"] in H2 and H3 (default pool min(2k, 31) raised to k), outputs
        (Q, k); the answer of a graph built with topk = k where topk does not prune."""
        if not isinstance(gl, GraphLaplacian):
            raise TypeError("argument 'gl': 'GraphLaplacian' object expected")
        n_local, f, _, n_total = self._dims()
        if n_local != n_total and self._grid is None:
            raise NotImplementedError("search_hybrid on a row shard needs the search grid of build_sharded (this rank holds "
                                      "%d of %d rows)" % (n_local, n_total))
        q = np.ascontiguousarray(queries, dtype=np.float64)
        if q.ndim != 2 or q.shape[1] != f:
            raise ValueError("query length %d must match nfeatures %d" % (q.shape[-1], f))
        if pool is not None and (isinstance(pool, bool) or not isinstance(pool, (int, np.integer)) or pool < 1):
            raise ValueError("pool must be a positive integer (the shortlist length; default min(2 * topk, 31))")
        allowed = _check_allowed(allowed, n_total)
        k = _check_k(k)
        topk = gl.graph_params["topk"] if k is None else k
        nq = q.shape[0]
        try:
            if n_local != n_total:
                from .distributed import CudaEngine, sharded_search_hybrid
                engine = CudaEngine(_lib.load().asp_ctx_device(self._ctx))
                idx, score, lam = sharded_search_hybrid(engine, self._h, gl._h, q, float(tau), int(pool or 0), topk, n_total,
                                                        self._grid, allowed=allowed, call_k=k is not None)
                return (idx, score, lam) if want_lambda else (idx, score)
            idx = np.empty((nq, topk), dtype=np.int64)
            score = np.empty((nq, topk), dtype=np.float64)
            lam = np.empty(nq, dtype=np.float64)
            bits = self._allowed_bits(allowed)
            if k is not None:
                _lib.check(_lib.load().asp_search_hybrid_batch_k(self._h, gl._h, q.ctypes.data, nq, float(tau), int(pool or 0), k,
                                                                 idx.ctypes.data, score.ctypes.data, lam.ctypes.data,
                                                                 None if bits is None else bits.ctypes.data))
            elif bits is None:
                _lib.check(_lib.load().asp_search_hybrid_batch(self._h, gl._h, q.ctypes.data, nq, float(tau), int(pool or 0),
                                                               idx.ctypes.data, score.ctypes.data, lam.ctypes.data))
            else:
                _lib.check(_lib.load().asp_search_hybrid_batch_filtered(self._h, gl._h, q.ctypes.data, nq, float(tau),
                                                                        int(pool or 0), idx.ctypes.data, score.ctypes.data,
                                                                        lam.ctypes.data, bits.ctypes.data))
        except LibraryError as e:
            if e.code == _lib.ASP_ERR_ZERO_VECTOR:
                raise PanicException(e.message)
            raise
        return (idx, score, lam) if want_lambda else (idx, score)

    # ------------------------------------------------------------------ out of scope (SURVEY.md 8(f))

    def search_energy(self, item, gl, k, w_lambda=None, w_dirichlet=None):
        """src/lib.rs:232-262.  The binding's own part is here -- argument types, the query-length check (lib.rs:241-247),
        the defaults w_lambda = 1.0 / w_dirichlet = 0.5 (lib.rs:252-253) and the debug line (lib.rs:255-258).  The scoring
        is the crate's ArrowSpace::search_energy (lib.rs:260), whose arithmetic (lambda proximity + "Rayleigh-Dirichlet
        term") exists nowhere under /root/reference -- no formula, no test, no golden output, only retrieval metrics on an
        absent dataset (tests/output/1761234699_v0_18_energymaps_8_sweep) -- so the call ends in NotImplementedError
        rather than in numbers nothing can check (DESIGN.md section 6)."""
        if not isinstance(gl, GraphLaplacian):
            raise TypeError("argument 'gl': 'GraphLaplacian' object expected")
        if not isinstance(item, np.ndarray) or item.dtype != np.float64 or item.ndim != 1:
            raise TypeError("argument 'item': expected 1-D numpy.ndarray of float64")
        if not item.flags.c_contiguous:
            raise ValueError("The given array is not contiguous")
        if item.shape[0] != self.nfeatures:
            raise ValueError("query length %d must match nfeatures %d" % (item.shape[0], self.nfeatures))
        k = _extract_usize(k)
        w_l = 1.0 if w_lambda is None else _extract_f64(w_lambda)
        w_d = 0.5 if w_dirichlet is None else _extract_f64(w_dirichlet)
        dbg_println("search_energy: qlen=%d, k=%d, w_λ=%.2f, w_D=%.2f" % (item.shape[0], k, w_l, w_d))
        raise NotImplementedError("search_energy: the energy score is defined only inside the crate arrowspace 0.18.0 "
                                  "(src/lib.rs:260); there is no specification to build it against")


def persist_items(space):
    """The stored rows of a space as a host array (asp_space_items)."""
    n, f = space.nitems_local, space.nfeatures
    out = np.empty((n, f), dtype=np.float64)
    _lib.check(_lib.load().asp_space_items(space._h, out.ctypes.data))
    return out


def _to_host(t, out=None):
    """Device tensor -> numpy; into `out` (already resident pages, or the caller's pinned buffer) when given."""
    if out is None:
        return t.cpu().numpy()
    import torch
    torch.from_numpy(out).copy_(t)
    return out


def _upload_queries_sharded(space, q_np):
    """Host batch [Q, F] -> device tensor [Q, F] on every rank of the space's group: rank r copies rows
    [r*per, (r+1)*per) from (pinned) host memory, all_gather_into_tensor over NCCL assembles the batch."""
    import torch
    import torch.distributed as dist
    group = space._group
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = torch.device("cuda", _lib.load().asp_ctx_device(space._ctx))
    nq, f = q_np.shape
    per = (nq + world - 1) // world
    r0, r1 = min(rank * per, nq), min((rank + 1) * per, nq)
    part = torch.zeros((per, f), dtype=torch.float64, device=dev)
    if r1 > r0:
        part[: r1 - r0].copy_(torch.from_numpy(q_np[r0:r1]), non_blocking=True)
    full = torch.empty((world * per, f), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(full, part, group=group)
    return full[:nq]


def _peer_exchange(space, world, nq, topk, dev):
    """Exchange buffer of the peer-memory merge (csrc/peer.cu): one symmetric allocation per space, mapped by every rank
    of the group (torch.distributed._symmetric_memory is the plumbing; the kernels that use the peer pointers are ours)."""
    import torch
    import torch.distributed as dist
    import torch.distributed._symmetric_memory as symm_mem
    st = getattr(space, "_peer", None)
    if st is None or st["cap"] < nq or st["topk"] != topk:
        lib = _lib.load()
        cap = max(int(nq), 65536)
        nbytes = lib.asp_peer_exchange_bytes(world, cap, topk)
        if nbytes == 0:
            raise ValueError("peer merge supports at most %d ranks" % 8)
        buf = symm_mem.empty(nbytes, dtype=torch.uint8, device=dev)
        group = space._group if space._group is not None else dist.group.WORLD
        hdl = symm_mem.rendezvous(buf, group)
        buf.zero_()
        torch.cuda.current_stream(dev).synchronize()
        dist.barrier(group)                                   # every rank's flags are zero before anyone publishes
        ptrs = (C.c_uint64 * world)(*[int(p) for p in hdl.buffer_ptrs])
        st = dict(buf=buf, hdl=hdl, ptrs=ptrs, cap=cap, topk=topk, epoch=0)
        space._peer = st
    return st


def _merge_across_ranks(space, idx, score, nq, topk):
    """K5 host side: all-gather the per-shard (idx, score) lists, merge on the device.  ASP_PEER_MERGE=1: the lists travel
    as P2P stores into every rank's exchange buffer and the merge kernel waits on flags instead (csrc/peer.cu; bitwise
    equal to this route on 2 GPUs, opt-in until it has been run on 8 and timed)."""
    import torch
    import torch.distributed as dist
    lib = _lib.load()
    group = space._group
    world = dist.get_world_size(group)
    dev = torch.device("cuda", _lib.load().asp_ctx_device(space._ctx))
    was_numpy = isinstance(idx, np.ndarray)
    t_idx = torch.from_numpy(idx).to(dev) if was_numpy else idx
    t_sc = torch.from_numpy(score).to(dev) if was_numpy else score
    if os.environ.get("ASP_PEER_MERGE", "0") == "1" and topk > 0 and nq > 0:
        st = _peer_exchange(space, world, nq, topk, dev)
        st["epoch"] += 1
        out_idx = torch.empty((nq, topk), dtype=torch.int64, device=dev)
        out_sc = torch.empty((nq, topk), dtype=torch.float64, device=dev)
        t_idx, t_sc = t_idx.contiguous(), t_sc.contiguous()
        torch.cuda.current_stream(dev).synchronize()
        try:
            _lib.check(lib.asp_peer_merge(space._ctx, world, dist.get_rank(group), st["ptrs"], st["cap"], st["epoch"],
                                          t_idx.data_ptr(), t_sc.data_ptr(), nq, topk, out_idx.data_ptr(), out_sc.data_ptr()))
        except LibraryError:
            space._peer = None          # flags / epochs are out of step now: the next call re-rendezvouses (zeroed flags + barrier)
            raise
        if was_numpy:
            return out_idx.cpu().numpy(), out_sc.cpu().numpy()
        return out_idx, out_sc
    all_idx = torch.empty((world, nq, topk), dtype=torch.int64, device=dev)
    all_sc = torch.empty((world, nq, topk), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(all_idx, t_idx.contiguous(), group=group)
    dist.all_gather_into_tensor(all_sc, t_sc.contiguous(), group=group)
    out_idx = torch.empty((nq, topk), dtype=torch.int64, device=dev)
    out_sc = torch.empty((nq, topk), dtype=torch.float64, device=dev)
    torch.cuda.current_stream(dev).synchronize()
    _lib.check(lib.asp_topk_merge(space._ctx, all_idx.data_ptr(), all_sc.data_ptr(), world, nq, topk,
                                  out_idx.data_ptr(), out_sc.data_ptr()))
    _lib.check(lib.asp_ctx_synchronize(space._ctx))
    if was_numpy:
        return out_idx.cpu().numpy(), out_sc.cpu().numpy()
    return out_idx, out_sc


class ArrowSpaceBuilder:
    @staticmethod
    def build(graph_params, items, **extras):
        """Feature graph + Laplacian + per-item lambdas.  src/lib.rs:270-300.

        keyword-only extras (never positional, SURVEY.md section 5): device=int and the switches of the choices the
        reference's tests cannot pin (include/arrowspace_b200.h asp_switches): kernel=, tau_mode=, tau_fixed=,
        lambda_form=, symmetrise=, laplacian=, k_counts_self=, topk_prunes=, distance=, or a named set profile="kat12".

        reduction=True | {"sample_rate": 0.6, "seed": 42, "n_clusters": 0, "max_iters": 10, "probes": 2048} runs the
        pre-graph reduction the crate runs inside this call (src/lib.rs:282-283; SURVEY.md 8(f)-1): rows sampled, two-NN
        intrinsic dimension, k-means; the graph is built on the centroid matrix, lambdas for every item.  The outcome is
        on `gl.reduction` (dict) and the centroids on `gl.centroids()`.  Default: off (the documented recipe on all rows).
        """
        lib = _lib.load()
        dbg_println("Convert pyarray2 and Vec<Vec>")
        device_in = _is_device_tensor(items)
        if device_in:
            import torch
            if items.dtype != torch.float64 or items.dim() != 2:
                raise TypeError("argument 'items': expected a 2-D float64 tensor")
            x = items.contiguous()
            n, f = x.shape
            ptr = x.data_ptr()
            torch.cuda.current_stream(x.device).synchronize()      # the library runs on its own stream
        else:
            if not isinstance(items, np.ndarray) or items.dtype != np.float64 or items.ndim != 2:
                raise TypeError("argument 'items': expected 2-D numpy.ndarray of float64")
            n, f = items.shape
            x = np.ascontiguousarray(items)          # any strides accepted (as_array()), src/helpers.rs:25
            ptr = x.ctypes.data
        if n == 0 or f == 0:
            raise _unwrap(ValueError("items must be non-empty 2D array"))        # src/helpers.rs:27-29 + .unwrap()
        dbg_println("items shape: (%d, %d)" % (n, f))
        if _DEBUG and not device_in:
            dbg_println("items[0][:5]: %s" % list(x[0, :5]))
            dbg_println("NaNs: %d, Infs: %d" % (int(np.isnan(x).sum()), int(np.isinf(x).sum())))
        try:
            gp = parse_graph_params(graph_params)
        except (ValueError, TypeError, OverflowError) as e:
            raise _unwrap(e)                                                     # src/lib.rs:279 .unwrap()
        if gp is None:
            gp = dict(DEFAULT_GRAPH_PARAMS)
        cgp = _lib.make_params(gp["eps"], gp["k"], gp["topk"], gp["p"], gp["sigma"])
        sw = _lib.switches_from(extras)
        ctx = _lib.context(extras.get("device"))
        dbg_println("Building from rows")
        hs, hg, hc = C.c_void_p(), C.c_void_p(), C.c_void_p()
        reduction = extras.get("reduction")
        info = _lib.ReductionInfo()
        try:
            if reduction:
                red = _lib.make_reduction(reduction)
                _lib.check(lib.asp_build_reduced(ctx, ptr, n, f, C.byref(cgp), C.byref(sw), C.byref(red), C.byref(hs),
                                                 C.byref(hg), C.byref(info), C.byref(hc)))
            else:
                _lib.check(lib.asp_build(ctx, ptr, n, f, C.byref(cgp), C.byref(sw), C.byref(hs), C.byref(hg)))
        except LibraryError as e:
            if e.code in (_lib.ASP_ERR_ZERO_VECTOR, _lib.ASP_ERR_EMPTY):
                raise PanicException(e.message)
            raise
        aspace, gl = ArrowSpace._wrap(hs, ctx), GraphLaplacian._wrap(hg)
        if reduction:
            gl.reduction = info.as_dict()
            gl._centroids = ArrowSpace._wrap(hc, ctx)
        dbg_println("built ArrowSpace: nitems=%d, nfeatures=%d, lambdas_len=%d" % (n, f, n))
        return aspace, gl

    @staticmethod
    def build_sharded(graph_params, items_shard, n_total, group=None, **extras):
        """Extension: one process per GPU, each passing ITS rows (see shard_rows).  Collectives:
        all-gather of the Gram segment partials (8 x F x F f64), rank-ordered continuation of the
        exact column sums (rare), nothing else.  Returns (ArrowSpace shard, GraphLaplacian replica)."""
        from . import distributed
        return distributed.build_sharded(graph_params, items_shard, n_total, group, **extras)

    @staticmethod
    def build_item_graph(graph_params, items, **extras):
        """Extension (SURVEY.md Appendix A2, `nodes = items`): the eps / k-NN graph whose nodes are the ITEMS
        (the graph-build workload of BASELINE.json configs C4/C5).  Returns (ArrowSpace without lambdas,
        GraphLaplacian over nitems nodes).  Single GPU."""
        lib = _lib.load()
        if _is_device_tensor(items):
            import torch
            x = items.contiguous()
            ptr = x.data_ptr()
            torch.cuda.current_stream(x.device).synchronize()
        else:
            if not isinstance(items, np.ndarray) or items.dtype != np.float64 or items.ndim != 2:
                raise TypeError("argument 'items': expected 2-D numpy.ndarray of float64")
            x = np.ascontiguousarray(items)
            ptr = x.ctypes.data
        n, f = x.shape
        gp = parse_graph_params(graph_params) or dict(DEFAULT_GRAPH_PARAMS)
        cgp = _lib.make_params(gp["eps"], gp["k"], gp["topk"], gp["p"], gp["sigma"])
        sw = _lib.switches_from(extras)
        ctx = _lib.context(extras.get("device"))
        hs, hg = C.c_void_p(), C.c_void_p()
        _lib.check(lib.asp_space_create(ctx, ptr, n, f, n, 1, 0, C.byref(hs)))
        aspace = ArrowSpace._wrap(hs, ctx)
        _lib.check(lib.asp_item_graph(hs, C.byref(cgp), C.byref(sw), C.byref(hg)))
        return aspace, GraphLaplacian._wrap(hg)

    @staticmethod
    def build_item_graph_sharded(graph_params, items_shard, n_total, row0, group=None, **extras):
        """Extension: the item graph across the GPUs of one box (one process per GPU): all-gather of the item shards
        (halo rows), every rank resolves its rows on the tensor cores, all-gather of the neighbour lists."""
        from .distributed import build_item_graph_sharded
        return build_item_graph_sharded(graph_params, items_shard, n_total, row0, group=group, **extras)

    @staticmethod
    def load(path, **extras):
        """Extension: (ArrowSpace, GraphLaplacian) from a file written by ArrowSpace.save -- no build kernel runs."""
        from . import persist
        return persist.load(path, extras.get("device"))

    @staticmethod
    def build_energy(items, energy_params=None, graph_params=None):
        """src/lib.rs:333-376.  The binding's own part is here: the marshalling check (`pyarray2_to_vecvec(items)?`,
        lib.rs:341 -- a ValueError, not a panic, because this entry point propagates with `?`), parse_energy_params
        (src/energyparams.rs:6-45) and parse_graph_params, the debug lines.  The pipeline itself (optical compression,
        diffusion, sub-centroid splitting, energy-distance graph: RustBuilder::build_energy, lib.rs:362) is documented only
        by its parameter names (lib.rs:309-322); nothing under /root/reference states its arithmetic or holds an output
        that could check a restatement, so the call ends in NotImplementedError (DESIGN.md section 6)."""
        dbg_println("build_energy: Converting pyarray2 to Vec<Vec>")
        if _is_device_tensor(items):
            n, f = (items.shape + (0, 0))[:2] if items.dim() == 2 else (0, 0)
        else:
            if not isinstance(items, np.ndarray) or items.dtype != np.float64 or items.ndim != 2:
                raise TypeError("argument 'items': expected 2-D numpy.ndarray of float64")
            n, f = items.shape
        if n == 0 or f == 0:
            raise ValueError("items must be non-empty 2D array")                 # src/helpers.rs:27-29 through `?`
        e = parse_energy_params(energy_params)
        dbg_println("build_energy: optical_tokens=%s, w_λ=%.2f, w_G=%.2f, w_D=%.2f"
                    % ("None" if e["optical_tokens"] is None else "Some(%d)" % e["optical_tokens"], e["w_lambda"], e["w_disp"],
                       e["w_dirichlet"]))
        parse_graph_params(graph_params)                                          # lib.rs:351 `?`: errors propagate as they are
        dbg_println("build_energy: Starting energy pipeline")
        raise NotImplementedError("build_energy: the energy pipeline is defined only inside the crate arrowspace 0.18.0 "
                                  "(src/lib.rs:362); there is no specification to build it against")


def shard_rows(n_total, world, rank):
    """Rows [row0, row1) of `rank`: whole Gram segments (see ASP_GRAM_SEGMENTS)."""
    r0, r1 = C.c_int64(), C.c_int64()
    _lib.check(_lib.load().asp_shard_rows(int(n_total), int(world), int(rank), C.byref(r0), C.byref(r1)))
    return r0.value, r1.value


def stat(key, device=None):
    return _lib.load().asp_ctx_stat(_lib.context(device), key.encode())


def launch_count(device=None):
    return _lib.load().asp_ctx_launch_count(_lib.context(device))
