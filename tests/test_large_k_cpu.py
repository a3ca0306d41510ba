"""Search with a per-call k (k= on search_batch, search_hybrid and search_hybrid_batch) without a GPU.

- The argument checks of k= and which C entry point a call reaches (k=None: exactly the graph-topk call of before), on a
  library stand-in that records the calls.
- The new C entry points refuse NULL handles before any CUDA call.
- The wide stage 2's selection (csrc/large_k.cuh: the cut, the survivors, the band, the final order) walked on the CPU
  against a numpy restatement, on inputs with heavy exact ties across the k-th place."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------- the Python surface on a stand-in library

class _RecordingLib:
    """Enough of the library for the search calls of one GPU: records (entry point, args), answers ASP_OK."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("asp_search"):
            raise AttributeError(name)

        def fn(*args):
            self.calls.append((name, args))
            return 0
        return fn


@pytest.fixture
def fake(monkeypatch):
    from pyarrowspace_b200 import _lib, api
    lib = _RecordingLib()
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(api.ArrowSpace, "_dims", lambda self: (50, 4, 0, 50))
    monkeypatch.setattr(api.GraphLaplacian, "graph_params", property(lambda self: {"topk": 6}))
    space = api.ArrowSpace._wrap(None, None)
    gl = api.GraphLaplacian._wrap(None)
    return lib, space, gl


def test_k_none_calls_the_graph_topk_entry_points(fake):
    lib, space, gl = fake
    q = np.ones((3, 4))
    idx, sc = space.search_batch(q, gl, 0.5)
    assert idx.shape == (3, 6) and [c[0] for c in lib.calls] == ["asp_search_batch"]
    space.search_batch(q, gl, 0.5, allowed=np.ones(50, dtype=bool))
    idx, sc = space.search_hybrid_batch(q, gl, 0.5)
    assert idx.shape == (3, 6)
    space.search_hybrid_batch(q, gl, 0.5, allowed=np.ones(50, dtype=bool))
    assert [c[0] for c in lib.calls] == ["asp_search_batch", "asp_search_batch_filtered", "asp_search_hybrid_batch",
                                        "asp_search_hybrid_batch_filtered"]


def test_k_calls_the_k_entry_points_with_k_wide_outputs(fake):
    lib, space, gl = fake
    q = np.ones((3, 4))
    idx, sc = space.search_batch(q, gl, 0.5, k=40)
    assert idx.shape == sc.shape == (3, 40) and idx.dtype == np.int64 and sc.dtype == np.float64
    name, args = lib.calls[-1]
    assert name == "asp_search_batch_k" and args[5] == 40 and args[-1] is None         # no mask: NULL
    space.search_batch(q, gl, 0.5, k=np.int64(7), allowed=np.ones(50, dtype=bool))
    name, args = lib.calls[-1]
    assert name == "asp_search_batch_k" and args[5] == 7 and args[-1] is not None
    idx, sc = space.search_hybrid_batch(q, gl, 0.5, k=100, pool=3)
    name, args = lib.calls[-1]
    assert idx.shape == (3, 100) and name == "asp_search_hybrid_batch_k" and args[5:7] == (3, 100) and args[-1] is None
    res = space.search_hybrid(q[0].copy(), gl, 0.5, k=2)
    assert lib.calls[-1][0] == "asp_search_hybrid_batch_k" and lib.calls[-1][1][6] == 2 and isinstance(res, list)


def test_k_argument_checks(fake):
    from pyarrowspace_b200 import _lib
    lib, space, gl = fake
    q = np.ones((2, 4))
    for bad in (0, -3, True, False, 2.0, "5", np.float64(3.0)):
        for call in (lambda: space.search_batch(q, gl, 0.5, k=bad), lambda: space.search_hybrid_batch(q, gl, 0.5, k=bad),
                     lambda: space.search_hybrid(q[0].copy(), gl, 0.5, k=bad)):
            with pytest.raises(ValueError):
                call()
    for call in (lambda: space.search_batch(q, gl, 0.5, k=1025), lambda: space.search_hybrid_batch(q, gl, 0.5, k=5000)):
        with pytest.raises(_lib.LibraryError) as e:
            call()
        assert e.value.code == _lib.ASP_ERR_UNSUPPORTED
    assert lib.calls == []
    space.search_batch(q, gl, 0.5, k=1024)
    assert lib.calls[-1][0] == "asp_search_batch_k"
    with pytest.raises(TypeError):
        space.search_batch(q, gl, 0.5, None, None, 5)                                     # keyword only


def test_out_shapes_follow_k(fake):
    lib, space, gl = fake
    q = np.ones((3, 4))
    good = (np.empty((3, 33), dtype=np.int64), np.empty((3, 33)))
    idx, sc = space.search_batch(q, gl, 0.5, good, k=33)
    assert idx is good[0] and sc is good[1] and lib.calls[-1][0] == "asp_search_batch_k"
    with pytest.raises(ValueError):
        space.search_batch(q, gl, 0.5, (np.empty((3, 6), dtype=np.int64), np.empty((3, 6))), k=33)   # the graph's topk shape
    with pytest.raises(ValueError):
        space.search_batch(q, gl, 0.5, good)                                               # k=None: (Q, topk)


def test_k_entry_points_reject_null_handles_without_a_gpu():
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    q = np.ones((1, 4))
    idx, sc, cs, lam = np.zeros((1, 40), dtype=np.int64), np.zeros((1, 40)), np.zeros((1, 40)), np.zeros(1)
    for call in (lambda: lib.asp_search_batch_k(None, None, q.ctypes.data, 1, 0.5, 40, idx.ctypes.data, sc.ctypes.data,
                                                lam.ctypes.data, None),
                 lambda: lib.asp_search_hybrid_batch_k(None, None, q.ctypes.data, 1, 0.5, 0, 40, idx.ctypes.data, sc.ctypes.data,
                                                       lam.ctypes.data, None),
                 lambda: lib.asp_search_hybrid_shard_k(None, None, q.ctypes.data, 1, 0.5, 0, 40, idx.ctypes.data, cs.ctypes.data,
                                                       sc.ctypes.data, lam.ctypes.data, None)):
        assert call() == _lib.ASP_ERR_ARG
        assert b"NULL argument" in lib.asp_last_error()


# ----------------------------------------------------------------------------- the selection header on the CPU

@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("lk") / "liblk_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "host_emul", "large_k_host.cpp")])
    lib = C.CDLL(out)
    vp, i64, ci = C.c_void_p, C.c_int64, C.c_int
    lib.lk_emulate.argtypes = [ci, ci, i64, ci, ci, vp, vp, vp, vp, C.c_double, vp, vp, i64, vp, vp, vp, vp, vp]
    lib.lk_emulate.restype = None
    return lib


SURV_CAP = 4096


def _numpy_select(k, n_local, cnt, esc, eix, delta, eps, fast, exact, row0, capb):
    """The restatement: (idx, score, route) per query."""
    nq = cnt.shape[0]
    kk = min(k, n_local)
    idx = np.full((nq, k), -1, dtype=np.int64)
    sc = np.full((nq, k), np.nan)
    route = np.zeros(nq, dtype=np.int32)
    for q in range(nq):
        if (cnt[q] > capb).any():
            route[q] = 1
            continue
        s = np.concatenate([esc[q, c, :cnt[q, c]] for c in range(cnt.shape[1])])
        ix = np.concatenate([eix[q, c, :cnt[q, c]] for c in range(cnt.shape[1])])
        if len(s) < kk:
            route[q] = 1
            continue
        kth = np.sort(s)[::-1][kk - 1]
        cutoff = np.float32(kth) - np.float32(2.0) * np.float32(delta[q])
        surv = ix[s >= cutoff]
        if len(surv) > SURV_CAP or len(surv) < kk:
            route[q] = 1
            continue
        fs = fast[q, surv]
        order = np.lexsort((surv, -fs))
        kth_f = fs[order[kk - 1]]
        band = surv[fs >= kth_f - 2.0 * eps]
        ex = exact[q, band]
        fin = np.lexsort((band, -ex))[:kk]
        idx[q, :kk] = row0 + band[fin]
        sc[q, :kk] = ex[fin]
    return idx, sc, route


def _walk(emul, k, n_local, cnt, esc, eix, delta, eps, fast, exact, row0, capb):
    nq, ns = cnt.shape
    out_i = np.full((nq, k), 77, dtype=np.int64)
    out_s = np.full((nq, k), 77.0)
    route, nsurv, nband = (np.zeros(nq, dtype=np.int32) for _ in range(3))
    emul.lk_emulate(nq, k, n_local, ns, capb, cnt.ctypes.data, esc.ctypes.data, eix.ctypes.data, delta.ctypes.data, eps,
                    fast.ctypes.data, exact.ctypes.data, row0, out_i.ctypes.data, out_s.ctypes.data, route.ctypes.data,
                    nsurv.ctypes.data, nband.ctypes.data)
    return out_i, out_s, route, nsurv, nband


def _case(seed, nq, n_local, k, nstreams, capb, levels, emit_frac):
    """Emission lists of distinct items spread over the streams; approximate scores on a coarse grid (heavy exact ties), fast
    scores near the exact ones with ties of their own, exact scores on a grid too (ties broken by the index)."""
    rng = np.random.default_rng(seed)
    exact = np.round(rng.uniform(0, 1, (nq, n_local)) * levels) / levels
    fast = exact + np.round(rng.uniform(-1, 1, (nq, n_local)) * 2) * 1e-14
    approx = (np.round((exact + rng.uniform(-0.02, 0.02, (nq, n_local))) * levels) / levels).astype(np.float32)
    cnt = np.zeros((nq, nstreams), dtype=np.int32)
    esc = np.zeros((nq, nstreams, capb), dtype=np.float32)
    eix = np.zeros((nq, nstreams, capb), dtype=np.int32)
    for q in range(nq):
        items = rng.permutation(n_local)[:int(emit_frac * n_local)]
        for c in range(nstreams):
            mine = items[c::nstreams][:capb + 1]                                  # one stream may overflow by one
            n = min(len(mine), capb)
            cnt[q, c] = len(mine) if rng.random() < 0.05 else n
            esc[q, c, :n] = approx[q, mine[:n]]
            eix[q, c, :n] = mine[:n]
    delta = rng.uniform(0, 0.01, nq).astype(np.float32)
    return cnt, esc, eix, delta, fast, exact


@pytest.mark.parametrize("k,n_local,levels,emit_frac", [(32, 600, 20, 0.5), (64, 900, 8, 0.7), (33, 200, 3, 1.0), (64, 50, 5, 1.0),
                                                        (40, 3000, 50, 0.3), (48, 60, 10, 0.5)])
def test_selection_walk_equals_numpy(emul, k, n_local, levels, emit_frac):
    """Coarse score grids put long runs of exact ties across the kk-th place at every stage: the cut, the band and the final
    order (score desc, index asc).  k > n_local and fewer emitted than kk take the exact scan."""
    eps = 3e-14
    cnt, esc, eix, delta, fast, exact = _case(k + n_local, 12, n_local, k, 3, 700, levels, emit_frac)
    gi, gs, gr, nsurv, nband = _walk(emul, k, n_local, cnt, esc, eix, delta, eps, fast, exact, 1000, 700)
    wi, ws, wr = _numpy_select(k, n_local, cnt, esc, eix, delta, eps, fast, exact, 1000, 700)
    assert np.array_equal(gr, wr)
    done = gr == 0
    assert np.array_equal(gi[done], wi[done])
    ok = wi >= 0
    assert np.array_equal(gs[done & ok.any(1)][ok[done & ok.any(1)]], ws[done & ok.any(1)][ok[done & ok.any(1)]])
    assert np.isnan(gs[done][~ok[done]]).all()
    assert (nband[done] >= min(k, n_local)).all() and (nsurv[done] >= nband[done]).all()


@settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])
@given(st.integers(0, 2 ** 31 - 1), st.integers(32, 64), st.integers(1, 400), st.integers(1, 6), st.sampled_from([2, 4, 30]))
def test_selection_walk_random(emul, seed, k, n_local, nstreams, levels):
    eps = 1e-13
    cnt, esc, eix, delta, fast, exact = _case(seed, 4, n_local, k, nstreams, 128, levels, 0.8)
    gi, gs, gr, _, _ = _walk(emul, k, n_local, cnt, esc, eix, delta, eps, fast, exact, 0, 128)
    wi, ws, wr = _numpy_select(k, n_local, cnt, esc, eix, delta, eps, fast, exact, 0, 128)
    assert np.array_equal(gr, wr)
    done = gr == 0
    assert np.array_equal(gi[done], wi[done])
    both = done[:, None] & (wi >= 0)
    assert np.array_equal(gs[both], ws[both])


def test_survivor_cap_sends_the_query_to_the_exact_scan(emul):
    """More than SURV_CAP candidates at or above the cut (one long run of ties) cannot be kept: exact scan."""
    n_local, k = 6000, 40
    cnt = np.array([[5000]], dtype=np.int32)
    esc = np.full((1, 1, 5000), 0.5, dtype=np.float32)
    eix = np.arange(5000, dtype=np.int32).reshape(1, 1, -1)
    z = np.zeros((1, n_local))
    gi, gs, gr, nsurv, _ = _walk(emul, k, n_local, cnt, esc, eix, np.zeros(1, dtype=np.float32), 1e-13, z, z, 0, 5000)
    assert gr[0] == 1 and nsurv[0] == 5000
    esc[0, 0, 4000:] = 0.25                                                       # now 4000 survive: finished here
    gi, gs, gr, nsurv, nband = _walk(emul, k, n_local, cnt, esc, eix, np.zeros(1, dtype=np.float32), 1e-13, z, z, 0, 5000)
    assert gr[0] == 0 and nsurv[0] == 4000 and nband[0] == 4000 and list(gi[0]) == list(range(k))
