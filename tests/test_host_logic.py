"""Host side of the drop-in boundary, no GPU needed: the C-ABI library loads and exports every symbol
include/arrowspace_b200.h declares, the Python surface mirrors src/lib.rs / src/helpers.rs, the product
never touches oracle/, and compute calls fail loudly without a device."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "arrowspace_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(asp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    declared = _header_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), "libarrowspace_b200.so lacks %s" % name
    assert sorted(_lib.SYMBOLS) == declared, "ctypes table and header disagree"
    assert lib.asp_abi_version() == 2
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (asp_[a-z0-9_]+)", out))
    assert set(declared) <= exported


def test_entry_points_reject_null_handles_without_a_gpu():
    """Argument checks come before any CUDA call: the typed ctypes signatures reach the library and NULL handles are refused
    with ASP_ERR_ARG (no compute, no device needed)."""
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    q = np.ones((1, 4))
    idx, sc, lam = np.zeros((1, 3), dtype=np.int64), np.zeros((1, 3)), np.zeros(1)
    for call in (lambda: lib.asp_search_batch(None, None, q.ctypes.data, 1, 0.5, idx.ctypes.data, sc.ctypes.data, lam.ctypes.data),
                 lambda: lib.asp_search_hybrid_batch(None, None, q.ctypes.data, 1, 0.5, 0, idx.ctypes.data, sc.ctypes.data,
                                                     lam.ctypes.data)):
        assert call() == _lib.ASP_ERR_ARG
        assert b"NULL argument" in lib.asp_last_error()


def test_header_is_plain_c_and_links_from_a_c_program(tmp_path):
    """The drop-in boundary is a C ABI: include/arrowspace_b200.h compiles as C99 and a C program linked against the library
    reaches it (entry points that need no device: ABI version, defaults, the row-shard arithmetic, argument checks)."""
    from pyarrowspace_b200 import _lib
    src = tmp_path / "abi.c"
    src.write_text(r"""
#include <stdio.h>
#include "arrowspace_b200.h"
int main(void)
{
    asp_switches sw; asp_reduction red; int64_t r0 = -1, r1 = -1;
    asp_default_switches(&sw); asp_default_reduction(&red);
    if (asp_abi_version() != ASP_ABI_VERSION) return 1;
    if (sw.kernel != ASP_KERNEL_INV_POWER || sw.symmetrise != ASP_SYM_MAX || red.seed != 42) return 2;
    if (asp_shard_rows(1000000, 8, 3, &r0, &r1) != ASP_OK || r0 >= r1) return 3;
    if (asp_search_hybrid_batch(NULL, NULL, NULL, 1, 0.5, 0, NULL, NULL, NULL) != ASP_ERR_ARG) return 4;
    printf("%lld %lld %s\n", (long long)r0, (long long)r1, asp_last_error());
    return 0;
}
""")
    exe = tmp_path / "abi"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", str(exe), "-L", libdir, "-larrowspace_b200", "-Wl,-rpath," + libdir])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    r0, r1 = (int(v) for v in r.stdout.split()[:2])
    from pyarrowspace_b200 import shard_rows
    assert (r0, r1) == shard_rows(1000000, 8, 3) and "NULL argument" in r.stdout


def test_library_is_built_for_sm_100a_only():
    from pyarrowspace_b200 import _lib
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_sass_has_dmma_and_tma():
    """FP64 tensor-core instructions and TMA tile loads are really in the binary."""
    from pyarrowspace_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert sass.count("DMMA.8x8x4") > 500
    assert "UTMALDG" in sass
    assert "UTCHMMA" in sass and "LDTM" in sass          # tcgen05.mma / tcgen05.ld of the candidate pass


def test_module_surface_matches_reference():
    import arrowspace
    assert set(arrowspace.__all__) == {"ArrowSpaceBuilder", "ArrowSpace", "GraphLaplacian", "set_debug"}
    from arrowspace import ArrowSpace, ArrowSpaceBuilder, GraphLaplacian
    with pytest.raises(ValueError, match="ArrowSpace cannot be constructed directly; use ArrowSpaceBuilder.build"):
        ArrowSpace()
    with pytest.raises(ValueError, match="use ArrowSpaceBuilder.build_with_graph"):
        GraphLaplacian()
    for name in ("nitems", "nfeatures", "get_item", "lambdas", "search", "search_hybrid", "search_energy"):
        assert hasattr(ArrowSpace, name)
    for name in ("nnodes", "shape", "graph_params"):
        assert hasattr(GraphLaplacian, name)
    assert isinstance(ArrowSpaceBuilder.__dict__["build"], staticmethod)
    assert isinstance(ArrowSpaceBuilder.__dict__["build_energy"], staticmethod)
    import inspect
    assert list(inspect.signature(ArrowSpace.search).parameters)[1:] == ["item", "gl", "tau"]
    assert list(inspect.signature(ArrowSpaceBuilder.build).parameters)[:2] == ["graph_params", "items"]


def test_parse_graph_params():
    from pyarrowspace_b200.api import parse_graph_params
    assert parse_graph_params(None) is None
    gp = parse_graph_params({"eps": 1, "k": 6, "topk": 3, "p": 2})
    assert gp == {"eps": 1.0, "k": 6, "topk": 3, "p": 2.0, "sigma": 0.5}          # helpers.rs:68-72
    assert parse_graph_params({"eps": 0.2, "k": 1, "topk": 1, "p": 2.0, "sigma": None})["sigma"] == 0.1
    assert parse_graph_params({"eps": 0.2, "k": 1, "topk": 1, "p": 2.0, "sigma": 0.7})["sigma"] == 0.7
    for key in ("eps", "k", "topk", "p"):
        d = {"eps": 1.0, "k": 6, "topk": 3, "p": 2.0}
        del d[key]
        with pytest.raises(ValueError, match=re.escape("graph_params['%s'] is required" % key)):
            parse_graph_params(d)
    with pytest.raises(OverflowError):
        parse_graph_params({"eps": 1.0, "k": -1, "topk": 3, "p": 2.0})
    with pytest.raises(TypeError):
        parse_graph_params({"eps": 1.0, "k": 2.5, "topk": 3, "p": 2.0})


def test_build_argument_errors_surface_as_panics():
    """.unwrap() in src/lib.rs:277,279 turns ValueErrors into PanicException (a BaseException)."""
    from arrowspace import ArrowSpaceBuilder, PanicException
    assert issubclass(PanicException, BaseException) and not issubclass(PanicException, Exception)
    with pytest.raises(PanicException, match="items must be non-empty 2D array"):
        ArrowSpaceBuilder.build({"eps": 1.0, "k": 1, "topk": 1, "p": 2.0}, np.zeros((0, 4)))
    with pytest.raises(PanicException, match=r"graph_params\[\\?'topk\\?'\] is required"):
        ArrowSpaceBuilder.build({"eps": 1.0, "k": 1, "p": 2.0}, np.ones((2, 4)))
    with pytest.raises(TypeError):
        ArrowSpaceBuilder.build({"eps": 1.0, "k": 1, "topk": 1, "p": 2.0}, np.ones((2, 4), dtype=np.float32))
    with pytest.raises(TypeError):
        ArrowSpaceBuilder.build({"eps": 1.0, "k": 1, "topk": 1, "p": 2.0}, np.ones(4))
    with pytest.raises(NotImplementedError):
        ArrowSpaceBuilder.build_energy(np.ones((2, 2)))


def test_parse_energy_params():
    """src/energyparams.rs:6-45: defaults (src/lib.rs:311-322), present keys overwrite, unknown keys ignored, pyo3's
    extraction errors."""
    from pyarrowspace_b200.api import DEFAULT_ENERGY_PARAMS, parse_energy_params
    assert parse_energy_params(None) == DEFAULT_ENERGY_PARAMS
    assert parse_energy_params({}) == DEFAULT_ENERGY_PARAMS
    assert DEFAULT_ENERGY_PARAMS == {"optical_tokens": None, "trim_quantile": 0.1, "eta": 0.1, "steps": 4, "split_quantile": 0.9,
                                     "neighbor_k": 8, "split_tau": 0.15, "w_lambda": 1.0, "w_disp": 0.5, "w_dirichlet": 0.25,
                                     "candidate_m": 32}
    # the dict of tests/test_8_CVE_db_sweep.py:164-176
    got = parse_energy_params({"optical_tokens": 40, "trim_quantile": 0.1, "eta": 0.05, "steps": 2, "split_quantile": 0.9,
                               "neighbor_k": 8, "split_tau": 0.15, "w_lambda": 1.0, "w_disp": 0.5, "w_dirichlet": 0.25,
                               "candidate_m": 32, "not_a_key": "ignored"})
    assert got["optical_tokens"] == 40 and got["eta"] == 0.05 and got["steps"] == 2 and "not_a_key" not in got
    assert parse_energy_params({"optical_tokens": None})["optical_tokens"] is None
    assert parse_energy_params({"eta": 1})["eta"] == 1.0 and isinstance(parse_energy_params({"eta": 1})["eta"], float)
    assert parse_energy_params({"steps": np.int64(6)})["steps"] == 6
    with pytest.raises(TypeError, match="cannot be interpreted as an integer"):
        parse_energy_params({"steps": 2.5})
    with pytest.raises(OverflowError):
        parse_energy_params({"neighbor_k": -1})
    with pytest.raises(TypeError, match="must be real number, not str"):
        parse_energy_params({"eta": "0.1"})
    with pytest.raises(TypeError):
        parse_energy_params({"eta": None})                                 # f64, not Option<f64>
    with pytest.raises(TypeError):
        parse_energy_params([("eta", 0.1)])


def test_energy_entry_points_do_the_bindings_part_then_stop(capsys):
    """build_energy / search_energy (src/lib.rs:232-262,333-376): argument handling and debug lines of the binding are
    reproduced; the crate-internal arithmetic has no specification under /root/reference, so they stop with
    NotImplementedError instead of returning numbers nothing can check."""
    from arrowspace import ArrowSpaceBuilder, set_debug
    with pytest.raises(ValueError, match="items must be non-empty 2D array"):     # `?`, not .unwrap(): a plain ValueError
        ArrowSpaceBuilder.build_energy(np.zeros((0, 4)))
    with pytest.raises(TypeError):
        ArrowSpaceBuilder.build_energy(np.ones((2, 2), dtype=np.float32))
    with pytest.raises(TypeError, match="must be real number"):
        ArrowSpaceBuilder.build_energy(np.ones((2, 2)), {"eta": "x"})
    with pytest.raises(ValueError, match=r"graph_params\['k'\] is required"):
        ArrowSpaceBuilder.build_energy(np.ones((2, 2)), None, {"eps": 1.0, "topk": 1, "p": 2.0})
    set_debug(True)
    try:
        with pytest.raises(NotImplementedError, match="src/lib.rs:362"):
            ArrowSpaceBuilder.build_energy(np.ones((2, 2)), {"optical_tokens": 40})
    finally:
        set_debug(False)
    err = capsys.readouterr().err
    assert "[pyarrowspace] build_energy: optical_tokens=Some(40), w_λ=1.00, w_G=0.50, w_D=0.25" in err   # src/lib.rs:344-347
    assert "[pyarrowspace] build_energy: Starting energy pipeline" in err


def test_search_hybrid_signature():
    """src/lib.rs:182-188: (item, gl, tau) positionally; the shortlist length is a keyword-only extra."""
    import inspect
    from arrowspace import ArrowSpace
    params = inspect.signature(ArrowSpace.search_hybrid).parameters
    assert list(params)[1:4] == ["item", "gl", "tau"]
    assert params["pool"].kind is inspect.Parameter.KEYWORD_ONLY and params["pool"].default is None
    assert list(inspect.signature(ArrowSpace.search_energy).parameters)[1:] == ["item", "gl", "k", "w_lambda", "w_dirichlet"]


def test_set_debug_prefix(capsys):
    from pyarrowspace_b200 import api
    api.set_debug(True)
    api.dbg_println("items shape: (3, 3)")
    api.set_debug(False)
    api.dbg_println("silent")
    err = capsys.readouterr().err
    assert err == "[pyarrowspace] items shape: (3, 3)\n"


def test_shard_rows_cover_and_align():
    from pyarrowspace_b200 import shard_rows
    for n in (1, 5, 31, 32, 33, 255, 256, 257, 1000, 99_999, 1_000_000, 8_800_000):
        for world in (1, 2, 4, 8):
            prev = 0
            for r in range(world):
                r0, r1 = shard_rows(n, world, r)
                assert r0 == prev and r0 <= r1 <= n
                assert r0 % 32 == 0 or r0 == n
                prev = r1
            assert prev == n
        # world sizes nest: a rank of world 2 is the union of two ranks of world 4
        a0, a1 = shard_rows(n, 2, 1)
        assert a0 == shard_rows(n, 4, 2)[0] and a1 == shard_rows(n, 4, 3)[1]
    with pytest.raises(Exception):
        shard_rows(100, 3, 0)


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_without_gpu():
    """The product path must fail loudly when there is no device -- never compute on the CPU."""
    from arrowspace import ArrowSpaceBuilder
    from pyarrowspace_b200._lib import LibraryError
    with pytest.raises(LibraryError, match="no CUDA device"):
        ArrowSpaceBuilder.build({"eps": 1.0, "k": 6, "topk": 3, "p": 2.0, "sigma": 1.0},
                                np.array([[0.1, 0.2, 0.3], [0.0, 0.5, 0.1], [0.9, 0.1, 0.0]]))


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under pyarrowspace_b200/ or arrowspace/ may reference it."""
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|liboracle|oracle_np|orc_[a-z_]+\(", re.M)
    for pkg in ("pyarrowspace_b200", "arrowspace"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, pkg)):
            if "_obj" in dirpath:
                continue
            for fn in files:
                if fn.endswith((".py", ".cu", ".cuh", ".h")):
                    text = open(os.path.join(dirpath, fn)).read()
                    assert not pat.search(text), "%s references the oracle" % os.path.join(dirpath, fn)
    code = ("import sys; import arrowspace, pyarrowspace_b200, pyarrowspace_b200.distributed; "
            "assert not [m for m in sys.modules if m == 'oracle' or m.startswith('oracle.')]")
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the oracle port on the host cores) prints exactly ONE JSON line on stdout carrying the
    keys the driver reads; run here on a reduced item count so that it takes seconds."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-queries", "4", "--items", "20000"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bench_dump_outputs_reference_arm(tmp_path, oracle_mod):
    """`bench.py --dump-outputs DIR` writes the last timed step's results as float64 .npy files; on the reference arm they
    equal the oracle's search of the same seeded queries."""
    from pyarrowspace_b200 import synth
    n, nq = 20000, 4
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--ref-queries", str(nq), "--items", str(n), "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {p.stem: np.load(p) for p in (tmp_path / "out").iterdir()}
    assert sorted(got) == ["query_rows", "search_idx", "search_scores"]
    assert all(a.dtype == np.float64 for a in got.values())
    cfg = synth.config("C4")
    x = synth.make_items(n, cfg["f"], cfg["seed"], cfg["scale"])
    q, _ = synth.make_queries(x, nq, cfg["seed"], cfg["scale"])
    s, g = oracle_mod.build(cfg["graph_params"], x)
    oidx, osc, _ = s.search_batch(q, g, cfg["tau"])
    np.testing.assert_array_equal(got["query_rows"], np.arange(nq))
    np.testing.assert_array_equal(got["search_idx"], oidx)
    np.testing.assert_array_equal(got["search_scores"], osc)


def test_bench_dump_outputs_sample_large_results(tmp_path, monkeypatch):
    """Results above the dump budget are written as a fixed, seeded, sorted sample of the queries, within the budget."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 100 * (8 + 16 * 10))
    idx = np.arange(1000 * 10, dtype=np.int64).reshape(1000, 10)
    sc = idx / 7.0
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), idx, sc)
    rows = np.load(tmp_path / "a" / "query_rows.npy")
    assert len(rows) == 100 and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "search_idx.npy"), idx[rows.astype(np.int64)])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "search_scores.npy"), sc[rows.astype(np.int64)])
    for name in ("query_rows", "search_idx", "search_scores"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy")))
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES


def test_peer_exchange_buffer_size():
    """asp_peer_exchange_bytes (pure host arithmetic, no GPU): 4 KB of flags + two parities of `world` slots of
    cap x topk (int64 index, f64 score) pairs; unsupported shapes give 0."""
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    assert lib.asp_peer_exchange_bytes(8, 65536, 10) == 4096 + 2 * 8 * 65536 * 10 * 16
    assert lib.asp_peer_exchange_bytes(2, 1000, 3) == 4096 + 2 * 2 * 1000 * 3 * 16
    assert lib.asp_peer_exchange_bytes(9, 10, 10) == 0 and lib.asp_peer_exchange_bytes(0, 10, 10) == 0
    assert lib.asp_peer_exchange_bytes(2, 0, 10) == 0 and lib.asp_peer_exchange_bytes(2, 10, 0) == 0


def test_reduction_sampler_is_the_oracles(oracle_mod):
    """R1 of the pre-graph reduction is a host function of the C ABI (counter-based hash): same rows as the oracle's for any
    shard offset, keep rate close to the one asked, and shards concatenate to the unsharded sample."""
    import ctypes as C
    from pyarrowspace_b200 import _lib
    lib = _lib.load()
    for rate, seed in ((0.6, 42), (0.25, 7), (1.0, 1)):
        red = _lib.make_reduction({"sample_rate": rate, "seed": seed})
        n = 50000
        rows = np.empty(n, dtype=np.int32)
        cnt = C.c_int64()
        assert lib.asp_reduction_sample(C.byref(red), 0, n, rows.ctypes.data, C.byref(cnt)) == 0
        want = oracle_mod.reduction_sample(n, {"sample_rate": rate, "seed": seed})
        assert np.array_equal(rows[:cnt.value], want)
        assert abs(cnt.value / n - rate) < 0.01
        parts = []
        for r0, r1 in ((0, 12345), (12345, 30000), (30000, n)):
            assert lib.asp_reduction_sample(C.byref(red), r0, r1 - r0, rows.ctypes.data, C.byref(cnt)) == 0
            parts.append(rows[:cnt.value].astype(np.int64) + r0)
        assert np.array_equal(np.concatenate(parts), want)
