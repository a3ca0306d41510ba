"""The tau sweep (search_batch_taus) without a GPU.

- The argument checks of taus= (_check_taus) and what the Python layer hands the C entry point, on a library stand-in
  that records the calls; the loop over search_batch on multi-GPU layouts.
- The new C entry point refuses NULL handles before any CUDA call.
- csrc/sweep_bound.cuh compiled with g++: every column whose f32 score reaches some tau's emission threshold passes the
  combined raw-accumulator threshold of the common path, and each per-tau score is the single-tau epilogue's expression,
  bit for bit."""
import ctypes as C
import os
import subprocess
import tempfile

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


def test_check_taus_accepts_real_sequences_and_keeps_duplicates():
    from pyarrowspace_b200.api import _check_taus
    for taus in ([1.0, 0.8, 0.62], (0.62, 0.62), np.array([1, 0], dtype=np.int32), np.array([0.5, 0.5, 0.1], dtype=np.float32),
                 [np.float64(0.3), 2, np.int64(0)], [-0.2, 1.5]):
        got = _check_taus(taus)
        assert got.dtype == np.float64 and got.ndim == 1 and got.flags.c_contiguous
        assert got.tolist() == [float(t) for t in taus]


def test_check_taus_refusals():
    from pyarrowspace_b200.api import _check_taus
    for bad in ([True, 0.5], [0.5, np.bool_(False)], np.array([True, False]), ["0.5"], [None], [[0.5]], [1 + 2j],
                np.array([1 + 0j]), 0.5, "0.5", {0.5}, None):
        with pytest.raises(TypeError):
            _check_taus(bad)
    for bad in ([], np.array([]), [float("nan")], [0.5, float("inf")], np.array([-np.inf]), np.ones((2, 2))):
        with pytest.raises(ValueError):
            _check_taus(bad)


def test_search_batch_taus_calls_the_taus_entry_point(fake):
    lib, space, gl = fake
    q = np.ones((3, 4))
    idx, sc = space.search_batch_taus(q, gl, [1.0, 0.8, 0.62])
    assert idx.shape == sc.shape == (3, 3, 6) and idx.dtype == np.int64 and sc.dtype == np.float64
    name, args = lib.calls[-1]
    assert name == "asp_search_batch_taus" and args[3] == 3 and args[5] == 3 and args[6] == 6 and args[-1] is None
    taus = np.frombuffer(C.string_at(args[4], 3 * 8), dtype=np.float64)
    assert taus.tolist() == [1.0, 0.8, 0.62]
    idx, sc = space.search_batch_taus(q, gl, (0.5,), k=17, allowed=np.ones(50, dtype=bool))
    name, args = lib.calls[-1]
    assert idx.shape == (1, 3, 17) and args[5] == 1 and args[6] == 17 and args[-1] is not None
    assert [c[0] for c in lib.calls] == ["asp_search_batch_taus"] * 2


def test_search_batch_taus_argument_checks_before_the_library(fake):
    from pyarrowspace_b200 import _lib
    lib, space, gl = fake
    q = np.ones((2, 4))
    with pytest.raises(ValueError):
        space.search_batch_taus(q, gl, [])
    with pytest.raises(TypeError):
        space.search_batch_taus(q, gl, [False])
    with pytest.raises(ValueError):
        space.search_batch_taus(q, gl, [0.5], k=0)
    with pytest.raises(_lib.LibraryError):
        space.search_batch_taus(q, gl, [0.5], k=1025)
    with pytest.raises(ValueError):
        space.search_batch_taus(q, gl, [0.5], allowed=np.ones(49, dtype=bool))
    with pytest.raises(ValueError):
        space.search_batch_taus(np.ones((2, 5)), gl, [0.5])
    with pytest.raises(TypeError):
        space.search_batch_taus(q, gl, [0.5], None)                                       # keyword only
    assert lib.calls == []


def test_multi_gpu_layouts_loop_over_search_batch(fake, monkeypatch):
    from pyarrowspace_b200 import api
    lib, space, gl = fake
    seen = []

    def one(self, queries, gl_, tau, out=None, *, allowed=None, k=None):
        seen.append((tau, allowed is not None, k))
        nq = queries.shape[0]
        return np.full((nq, k or 6), int(tau * 10), dtype=np.int64), np.full((nq, k or 6), tau)
    monkeypatch.setattr(api.ArrowSpace, "search_batch", one)
    space._group = object()
    idx, sc = space.search_batch_taus(np.ones((2, 4)), gl, [0.5, 0.2, 0.5], k=3, allowed=np.ones(50, dtype=bool))
    assert seen == [(0.5, True, 3), (0.2, True, 3), (0.5, True, 3)]
    assert idx.shape == (3, 2, 3) and idx[1, 0, 0] == 2 and sc[2, 1, 2] == 0.5
    assert lib.calls == []


def test_taus_entry_point_refusals_without_a_gpu():
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    q = np.ones((1, 4))
    idx, sc, lam = np.zeros((2, 1, 4), dtype=np.int64), np.zeros((2, 1, 4)), np.zeros(1)
    taus = np.array([0.5, 0.8])
    assert lib.asp_search_batch_taus(None, None, q.ctypes.data, 1, taus.ctypes.data, 2, 4, idx.ctypes.data, sc.ctypes.data,
                                     lam.ctypes.data, None) == _lib.ASP_ERR_ARG
    assert b"NULL argument" in lib.asp_last_error()


# ----------------------------------------------------------------------------- the bound header on the CPU

@pytest.fixture(scope="module")
def bound():
    out = os.path.join(tempfile.mkdtemp(prefix="swb"), "libsweep_bound_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "host_emul", "sweep_bound_host.cpp")])
    lib = C.CDLL(out)
    f = C.c_float
    lib.sw_nt_max.restype = C.c_int
    lib.sw_prox.argtypes, lib.sw_prox.restype = [f, f], f
    lib.sw_score.argtypes, lib.sw_score.restype = [f] * 4, f
    lib.sw_single_tau_score.argtypes, lib.sw_single_tau_score.restype = [f] * 5, f
    lib.sw_prox_bound.argtypes, lib.sw_prox_bound.restype = [f] * 3, f
    fp = C.POINTER(f)
    lib.sw_combined.argtypes, lib.sw_combined.restype = [fp, fp, fp, f, C.c_int], f
    return lib


def _f32(v):
    return float(np.float32(v))


def _arr(vals):
    return (C.c_float * len(vals))(*vals)


PROP = settings(max_examples=300, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])


def test_nt_max_is_what_the_documents_say(bound):
    assert bound.sw_nt_max() == 3


@PROP
@given(st.integers(1, 4), st.lists(st.floats(0.0011, 1.0), min_size=4, max_size=4), st.sampled_from([0, 1, 2]),
       st.floats(0.0, 50.0), st.floats(-2e-3, 2e-3), st.floats(0.0, 5e-3), st.lists(st.booleans(), min_size=4, max_size=4),
       st.integers(0, 2 ** 31 - 1))
def test_combined_threshold_drops_no_column_some_tau_emits(bound, nt, taus, special, lq, off, width, finite, seed):
    """Taus in (0.001, 1] with 1.0 and values near 0.001 among them; lambda_q inside, below and above the tile's interval
    (2.5e-7 slack of f32 roundings); theta_emit -inf for some taus and finite around the tile's scores for others; columns
    at the interval ends and inside; accumulators at, just below and just above the value where a score reaches its
    threshold.  Whenever a score reaches its tau's theta_emit, the accumulator is >= the combined threshold, and each
    score is the single-tau expression bit for bit."""
    rng = np.random.default_rng(seed)
    taus = [_f32(t) for t in taus[:nt]]
    if special == 1:
        taus[0] = 1.0
    elif special == 2:
        taus[-1] = _f32(0.001 + 1e-6 * rng.uniform())
    betas = [_f32(1.0 - float(np.float64(t))) for t in taus]
    inv = [_f32(np.float32(1.0) / np.float32(t)) for t in taus]
    lq = _f32(lq)
    tl = _f32(lq + off)
    th = _f32(tl + width)
    lams = {tl, th, _f32(tl + (th - tl) * rng.uniform()), _f32(np.nextafter(np.float32(th), np.float32(-np.inf))),
            _f32(tl - 1e-7), _f32(th + 1e-7)}
    lams = [v for v in lams if tl - 2e-7 <= v <= th + 2e-7]          # a tile's f32 lambdas lie in [tl, th] (rounded outwards)
    pb = bound.sw_prox_bound(lq, tl, th)
    cos0 = rng.uniform(-0.2, 1.0)
    theta = []
    for t, b in zip(taus, betas):
        px = 1.0 / (1.0 + abs(lq - tl))
        theta.append(_f32(t * cos0 + b * px + rng.uniform(-1e-3, 1e-3)))
    for u in range(nt):
        if not finite[u]:
            theta[u] = -np.inf
    if all(not finite[u] for u in range(nt)):
        theta[0] = _f32(cos0)
    thr = bound.sw_combined(_arr(theta), _arr(betas), _arr(inv), pb, nt)
    for lam in lams:
        px = bound.sw_prox(lq, lam)
        accs = {float(np.float32(v)) for v in rng.uniform(-1.0, 1.0, 6) * 16384.0}
        for t, b, th_ in zip(taus, betas, theta):
            if np.isfinite(th_):
                a0 = np.float32((th_ - b * px) / t * 16384.0)
                a = a0
                for _ in range(3):
                    accs.add(float(a))
                    a = np.nextafter(a, np.float32(-np.inf))
                accs.add(float(np.nextafter(a0, np.float32(np.inf))))
        accs.add(float(np.float32(thr)) if np.isfinite(thr) else 0.0)
        for a in accs:
            reach = False
            for t, b, th_ in zip(taus, betas, theta):
                sc = bound.sw_score(t, b, px, a)
                assert sc == bound.sw_single_tau_score(t, b, lq, lam, a), (t, b, lq, lam, a)
                reach |= sc >= th_
            if reach:
                assert a >= thr, (taus, theta, lq, tl, th, lam, a, thr)


def test_combined_threshold_is_the_smallest_and_ignores_unused_slots(bound):
    inf = float("inf")
    betas = [0.0, 0.5]
    inv = [1.0, 2.0]
    one = bound.sw_combined(_arr([0.9]), _arr(betas[:1]), _arr(inv[:1]), 1.0, 1)
    two = bound.sw_combined(_arr([0.9, 0.9]), _arr(betas), _arr(inv), 1.0, 2)
    assert two == min(one, bound.sw_combined(_arr([0.9]), _arr(betas[1:]), _arr(inv[1:]), 1.0, 1))
    assert bound.sw_combined(_arr([0.9, inf]), _arr(betas), _arr(inv), 1.0, 2) == one          # unused slot: +inf
    assert bound.sw_combined(_arr([-inf, 0.9]), _arr(betas), _arr(inv), 1.0, 2) == -inf        # a tau without a threshold
