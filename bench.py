#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

metric   : search queries/s (top-10) on the BEIR/MS MARCO-shaped synthetic 1M x 384 f64 workload (C4, configs[3]: the
           configuration the metric is quoted on), with the build (feature graph + Laplacian + lambda) timed beside it.
step     : one pass of the search hot path over one batch of Q = 65536 synthetic queries (SURVEY.md 8(d): C4 is batched 64k
           per call) against all N items.  N > 1 (torchrun, one rank per GPU): the build is row-partitioned over all ranks;
           the search runs on an R x C grid (R item shards x C query slots, --item-shards, default: replicate the items when
           they fit, i.e. R = 1 for C4) and every rank ends with the whole result; strong scaling (fixed N and Q).
value    : whole-job queries/s with items and queries resident in HBM.
e2e      : the same through the public API (ArrowSpace.search_batch(q, gl, tau, out=...)) with HOST buffers: pinned host ->
           device copy of the batch and device -> host read of (idx, score) into the caller's pinned result buffers, every
           step, inside the timed region.
roofline : dominant kernel = tc_gemm_kernel (tcgen05.mma kind::f16 candidate pass): ALGORITHMIC 2*Q*N_local*F FLOP per
           launch (SURVEY.md 8(d) K4) / its CUDA-event duration, against MEASURED_PEAKS.json's dense 16-bit tensor figure;
           the executed FLOP (K padded to 16, extra split terms) are reported next to it.  The build's kernels are reported
           under "build" (K1 Gram: FP64 tensor, K3 lambda: HBM + the shared-memory gather floor).
parity_check : UNTIMED, after the timed loops: the CPU oracle builds the same 1M x 384 matrix and full-scans a sample of
           the last step's queries; indices must be identical and scores within 1e-9 for both the device-resident and the
           end-to-end results (at N > 1: the merged / gathered result), plus the feature graph and this rank's lambdas.
regimes  : the same search on MEAN-ZERO embeddings (no positive shift, tau_mode = median_abs) with queries that are fresh
           draws from the clusters, not perturbed copies of items: the regime in which the candidate pass needs the
           two-term fp16 split; throughput, mode, survivors per query and its own parity_check.
hybrid   : N = 1 only, in a separate process (tools/hybrid_leg.py): ArrowSpace.search_hybrid_batch (SURVEY.md 8(f)-2, restated
           semantics) on the same items, wall clock of the public call with host buffers, and its own oracle check.
cpu_baseline / --impl reference : the CPU oracle (oracle/, a restatement: the reference's Rust engine is not
           vendored and cannot be built here) timed on this box's host cores.

Launch: python bench.py --gpus N --steps K --warmup W   (N > 1 under torchrun, one rank per GPU).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLAGSHIP = "C4"


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner on the
    first communicator), so file descriptor 1 is pointed at stderr for the whole run and the line goes to the saved one."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--items", type=int, default=None, help="override N (default: the C4 shape, 1,000,000)")
    ap.add_argument("--features", type=int, default=None)
    ap.add_argument("--queries", type=int, default=65536, help="queries per step (SURVEY.md 8(d): C4 is batched 64k per call)")
    ap.add_argument("--build-reps", type=int, default=3)
    ap.add_argument("--cpu-sample-items", type=int, default=100_000)
    ap.add_argument("--cpu-sample-queries", type=int, default=64)
    ap.add_argument("--ref-queries", type=int, default=256, help="--impl reference: queries per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-item-graph", action="store_true", help="skip the item-graph (nodes = items) build of the C4 matrix")
    ap.add_argument("--item-shards", type=int, default=None, help="N > 1: item shards R of the search grid (default: fewest that fit; N: fully sharded)")
    ap.add_argument("--parity-queries", type=int, default=64, help="queries of the last step checked against the oracle's full scan (0: skip)")
    ap.add_argument("--no-regimes", action="store_true", help="skip the mean-zero regime")
    ap.add_argument("--no-reduction", action="store_true", help="skip the build with the pre-graph reduction (SURVEY.md 8(f)-1)")
    ap.add_argument("--no-hybrid", action="store_true", help="skip the hybrid-search leg (SURVEY.md 8(f)-2; N = 1 only, separate process)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's search results (top-k indices and scores) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, idx, score):
    """--dump-outputs: the result arrays of the last timed step, so that two builds run with the same arguments (same seeded
    inputs) can be compared output for output.  float64 holds the int64 indices exactly (-1 = no hit).  A batch whose results
    exceed 64 MB is written as a fixed, seeded sample of its queries; query_rows.npy names the rows written."""
    rows = np.arange(idx.shape[0])
    keep = (DUMP_BYTES - 4096) // (8 + 16 * idx.shape[1])              # bytes per query: its row number + topk (index, score)
    if len(rows) > keep:
        rows = np.sort(np.random.default_rng(0).choice(len(rows), keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("query_rows", rows), ("search_idx", idx[rows]), ("search_scores", score[rows])):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        # median over the samples taken under load (>= 60 % of the highest draw seen)
        load = [s for s, p in zip(sm, pw) if pw and p >= 0.6 * max(pw)] or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU oracle legs
def cpu_oracle_run(cfg, n_items, nq, reps, label):
    """Oracle build on n_items rows of the workload + `reps` search batches of nq queries, all host threads."""
    import oracle
    from pyarrowspace_b200 import synth
    # all the host threads this process may use: torchrun exports OMP_NUM_THREADS=1 to every rank, which would turn the
    # CPU arm into a single-thread run at N > 1 (rank 0 is the only rank that works here; the others exit)
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)
    x = synth.make_items(cfg["n"], cfg["f"], cfg["seed"], cfg["scale"], rows=(0, n_items))
    q, _ = synth.make_queries(x, nq, cfg["seed"], cfg["scale"])
    t0 = time.perf_counter()
    s, g = oracle.build(cfg["graph_params"], x)
    t_build = time.perf_counter() - t0
    s.search_batch(q[: max(1, nq // 8)], g, cfg["tau"])              # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        idx, sc, _ = s.search_batch(q, g, cfg["tau"])
        ts.append(time.perf_counter() - t0)
    return {"build_s": t_build, "search_s": ts, "threads": oracle.num_threads(), "n_items": n_items, "nq": nq,
            "idx": idx, "sc": sc}


def run_reference(args, cfg):
    """--impl reference: the CPU implementation of the path (the oracle port) on the host cores, same config/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.items or cfg["n"]
    cfg = dict(cfg, n=n)
    nq = args.ref_queries
    r = cpu_oracle_run(cfg, n, nq, args.warmup + args.steps, "reference")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["idx"], r["sc"])
    ts = r["search_s"][args.warmup:]
    total = sum(ts)
    val = nq * len(ts) / total
    line = {
        "impl": "reference", "metric": "search queries/s (top-10, 1M x 384 f64)", "value": val, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(ts),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C4 BEIR/MS MARCO-shaped synthetic %d x %d f64, top-%d, tau %.2f" % (n, cfg["f"], cfg["graph_params"]["topk"], cfg["tau"]),
                   "queries_per_step": nq, "graph_params": cfg["graph_params"]},
        "cpu_baseline": {"value": val, "unit": "queries/s", "cores": r["threads"], "kind": "port",
                         "sample": "oracle (C + OpenMP) search of %d queries per step against all %d items; build %.1f s (%.0f items/s) untimed"
                                   % (nq, n, r["build_s"], n / r["build_s"])},
        "build": {"items_per_s": n / r["build_s"], "seconds": r["build_s"]},
        "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def gram_roofline(n_local, f, ms, peak):
    """K1: 2*N*F^2 algorithmic FLOP; the kernel executes only the upper-triangular 128x128 output tiles
    (symmetry), so `frac` is EXECUTED FLOP / peak and the symmetry gain is reported separately."""
    nt = (f + 3) // 4 * 4
    nt = (nt + 127) // 128
    executed = 2.0 * n_local * (nt * (nt + 1) // 2) * 128 * 128
    algorithmic = 2.0 * n_local * f * f
    return {"ms": ms, "bound": "tensor", "algorithmic_flop": algorithmic, "executed_flop": executed,
            "achieved_tflops": executed / (ms * 1e-3) / 1e12, "frac": executed / (ms * 1e-3) / 1e12 / peak,
            "symmetry_speedup_vs_algorithmic": algorithmic / executed,
            "note": "ms is the stage time (slice kernel + reduces + scratch allocation), not the kernel alone"}


def hybrid_leg(args, n, local):
    """search_hybrid on the same workload (SURVEY.md 8(f)-2), in a separate process with a timeout: the path was written after
    the round's GPU budget was spent, so whatever happens in it must not cost this run its JSON line."""
    cmd = [sys.executable, os.path.join(ROOT, "tools", "hybrid_leg.py"), "--items", str(n), "--device", str(local)]
    if args.parity_queries <= 0:
        cmd += ["--parity-queries", "0"]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=180)
        for ln in reversed(r.stdout.splitlines()):
            if ln.startswith("HYBRID_LEG "):
                def finite(v):                                         # the bench line must stay strict JSON: no NaN / Infinity
                    if isinstance(v, dict):
                        return {k: finite(x) for k, x in v.items()}
                    if isinstance(v, float) and not np.isfinite(v):
                        return None
                    return v
                return finite(json.loads(ln[len("HYBRID_LEG "):]))
        return {"error": "exit code %d: %s" % (r.returncode, (r.stderr or r.stdout).strip()[-400:])}
    except subprocess.TimeoutExpired:
        return {"error": "timed out after 180 s"}
    except Exception as e:                                             # noqa: BLE001 -- a diagnostic leg never fails the bench
        return {"error": "%s: %s" % (type(e).__name__, e)}


# --------------------------------------------------------------------------- GPU arm
def oracle_parity(gp, tau, x_full, q_sample, got, lam_local, lam_rows, edges, switches, rtol=1e-9):
    """The CPU oracle on the SAME bytes: feature graph, lambdas of this rank's rows, full scan of the sample queries.
    `got` = {name: (idx, score)} result sets to compare (device-resident and end-to-end).  Untimed."""
    import oracle
    t0 = time.perf_counter()
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)
    s, g = oracle.build(gp, x_full, **switches)
    oidx, osc, _ = s.search_batch(q_sample, g, tau)
    out = {"queries": int(q_sample.shape[0]), "items": int(x_full.shape[0]), "rtol": rtol}
    ok = True
    for name, (idx, sc) in got.items():
        same = bool(np.array_equal(idx, oidx))
        m = oidx >= 0
        rel = float(np.max(np.abs(sc[m] - osc[m]) / np.abs(osc[m]))) if m.any() else 0.0
        out[name] = {"idx_equal": same, "score_max_rel_err": rel}
        ok = ok and same and rel <= rtol
    olam = s.lambdas()[lam_rows[0]:lam_rows[1]]
    lam_rel = float(np.max(np.abs(lam_local - olam) / np.abs(olam))) if len(olam) else 0.0
    out["lambda_max_rel_err"] = lam_rel
    out["lambda_rows_checked"] = int(len(olam))
    out["graph_edges_equal"] = bool(np.array_equal(edges, g.edges()))
    out["ok"] = bool(ok and lam_rel <= rtol and out["graph_edges_equal"])
    out["seconds"] = time.perf_counter() - t0
    out["oracle_threads"] = oracle.num_threads()
    return out


def main():
    args = parse_args()
    quiet_stdout()
    from pyarrowspace_b200 import synth
    cfg = synth.config(FLAGSHIP)
    if args.features:
        cfg["f"] = args.features
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch
    import torch.distributed as dist
    from pyarrowspace_b200 import _lib, api
    from pyarrowspace_b200.api import ArrowSpaceBuilder, shard_rows

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.items or cfg["n"]
    f, gp, tau, Q = cfg["f"], cfg["graph_params"], cfg["tau"], args.queries
    topk = gp["topk"]
    lib = _lib.load()
    ctx = _lib.context(local)
    stream = torch.cuda.Stream(device=dev)
    _lib.check(lib.asp_ctx_set_stream(ctx, stream.cuda_stream))       # the library's kernels go on this stream

    def barrier_sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- FP64 tensor peak on this GPU (cuBLAS DGEMM), the roofline denominator for the DMMA kernels
    with torch.cuda.stream(stream):
        a = torch.randn(4096, 4096, dtype=torch.float64, device=dev)
        b = torch.randn(4096, 4096, dtype=torch.float64, device=dev)
        best = 1e9
        for i in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); torch.matmul(a, b); e1.record(stream); e1.synchronize()
            if i:
                best = min(best, e0.elapsed_time(e1))
        fp64_peak_tflops = 2 * 4096 ** 3 / best / 1e9
        del a, b

    def build(items, switches):
        if world == 1:
            return ArrowSpaceBuilder.build(gp, items, device=local, **switches)
        return ArrowSpaceBuilder.build_sharded(gp, items, n, device=local, item_shards=args.item_shards, **switches)

    def search_regime(aspace, gl, q_dev, q_host, steps, warmup):
        """W warm-up steps, exactly `steps` timed steps with device-resident queries, then the same from pinned host
        memory (end to end).  Returns timings, the library's stage statistics and the LAST step's results of both."""
        nb = len(q_dev)
        clocks = ClockSampler(local)
        with torch.cuda.stream(stream):
            for w in range(warmup):
                aspace.search_batch(q_dev[w % nb], gl, tau)
            barrier_sync()
            if rank == 0:
                clocks.start()
            l0 = lib.asp_ctx_launch_count(ctx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            stage1 = []
            e0.record(stream)
            for k in range(steps):
                idx, sc = aspace.search_batch(q_dev[k % nb], gl, tau)
                stage1.append(api.stat("search_stage1_ms", local))
            e1.record(stream)
            barrier_sync()
            step_ms = max_over_ranks(e0.elapsed_time(e1)) / steps
            launches = lib.asp_ctx_launch_count(ctx) - l0
            st = {k: api.stat(k, local) for k in ("search_slow_queries", "search_stage1_is_tc", "search_rescored_per_query", "search_terms",
                                                 "search_stage2_ms", "search_a_resident", "search_delta_cos_max", "search_rho_q_max",
                                                 "search_rho_x_max", "search_exact_per_query", "search_retry_queries")}
            # the caller's result buffers: pinned host memory reused from step to step (search_batch(out=...))
            out_h = (torch.empty((q_host[0].shape[0], topk), dtype=torch.int64).pin_memory().numpy(),
                     torch.empty((q_host[0].shape[0], topk), dtype=torch.float64).pin_memory().numpy())
            for w in range(2 if warmup else 0):
                aspace.search_batch(q_host[w % nb].numpy(), gl, tau, out=out_h)
            barrier_sync()
            e0.record(stream)
            for k in range(steps):
                idx_h, sc_h = aspace.search_batch(q_host[k % nb].numpy(), gl, tau, out=out_h)
            e1.record(stream)
            barrier_sync()
            e2e_ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        clk = clocks.stop() if rank == 0 else None
        return {"step_ms": step_ms, "e2e_ms": e2e_ms, "launches": int(launches), "stage1_ms": max_over_ranks(float(np.mean(stage1))),
                "stats": st, "clocks": clk, "last_batch": (steps - 1) % nb,
                "idx": idx.cpu().numpy(), "sc": sc.cpu().numpy(), "idx_h": np.array(idx_h), "sc_h": np.array(sc_h)}

    # ---- synthetic inputs: this rank's row shard (identical bytes to what the oracle sees)
    r0, r1 = shard_rows(n, world, rank)
    x_host = torch.from_numpy(synth.make_items(n, f, cfg["seed"], cfg["scale"], rows=(r0, r1))).pin_memory()
    nbatch = 2
    qrng_src = synth.make_items(n, f, cfg["seed"], cfg["scale"], rows=(0, min(n, 65536)))
    q_host = [torch.from_numpy(synth.make_queries(qrng_src, Q, cfg["seed"] + b_, cfg["scale"])[0]).pin_memory()
              for b_ in range(nbatch)]
    with torch.cuda.stream(stream):
        x_dev = x_host.to(dev, non_blocking=True)
        q_dev = [q.to(dev, non_blocking=True) for q in q_host]
    stream.synchronize()

    # ---- build: items resident in HBM (value) and from pinned host memory (e2e)
    launches0 = lib.asp_ctx_launch_count(ctx)
    build_ms, build_e2e_ms, stages = [], [], {}
    with torch.cuda.stream(stream):
        for rep in range(1 + args.build_reps):
            barrier_sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            aspace, gl = build(x_dev, {})
            e1.record(stream)
            barrier_sync()
            if rep:
                build_ms.append(max_over_ranks(e0.elapsed_time(e1)))
                for k in ("gram_ms", "graph_ms", "lambda_ms"):
                    stages.setdefault(k, []).append(api.stat(k, local))
            del aspace, gl
        for rep in range(2):
            barrier_sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            aspace, gl = build(x_host.numpy(), {})
            e1.record(stream)
            barrier_sync()
            build_e2e_ms.append(max_over_ranks(e0.elapsed_time(e1)))
            if rep == 0:
                del aspace, gl
    build_launches = (lib.asp_ctx_launch_count(ctx) - launches0) // (3 + args.build_reps)
    feature_graph_nnz = int(gl.nnz)
    grid = getattr(aspace, "_grid", None) or {"R": 1, "C": 1}
    n_shard = aspace.nitems_local                                     # items every query of this rank is scored against
    q_rank = -(-Q // grid["C"])                                       # queries this rank answers per step

    # ---- search: W warm-up steps, then exactly K timed steps (+ the end-to-end loop)
    main_run = search_regime(aspace, gl, q_dev, q_host, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:                               # N > 1: every rank holds the whole merged result
        dump_outputs(args.dump_outputs, main_run["idx"], main_run["sc"])
    step_ms, e2e_ms, launches, stage1_ms, sstat, clk = (main_run[k] for k in ("step_ms", "e2e_ms", "launches", "stage1_ms", "stats", "clocks"))
    slow = sstat["search_slow_queries"]
    stage1_is_tc = sstat["search_stage1_is_tc"] == 1.0
    rescored = sstat["search_rescored_per_query"] if stage1_is_tc else None
    lam_local = aspace.lambdas()
    lam_rows = (aspace.row_offset, aspace.row_offset + aspace.nitems_local)
    edges = gl.edges()

    # ---- the reference's own call shape: ONE query per ArrowSpace.search call (src/lib.rs:132-174), host vector in,
    # Python list of (index, score) out; wall clock per call (includes the ctypes call, the upload and the read-back)
    single = None
    if world == 1:
        qs = q_host[0].numpy()
        for i in range(20):
            aspace.search(qs[i], gl, tau)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for i in range(200):
            hits = aspace.search(qs[20 + i], gl, tau)
        dt = (time.perf_counter() - t0) / 200
        single = {"ms_per_call": dt * 1e3, "queries_per_s": 1.0 / dt,
                  "f64_scan_equivalent_gbs": 8.0 * n * f / dt / 1e9,
                  "note": "candidate pass streams the fp16 operands (%.2f GB) instead of the f64 rows (%.2f GB); exact f64 stage 2"
                          % (2.0 * n * (((f + 3 + 63) // 64) * 64) / 1e9, 8.0 * n * f / 1e9)}
    del aspace, gl

    # ---- second regime: mean-zero embeddings, queries that are not near-duplicates of items (VERDICT r01 weak #8)
    regime = None
    mz_sw = {"tau_mode": "median_abs"}
    if not args.no_regimes:
        xz_host = torch.from_numpy(synth.make_items(n, f, cfg["seed"], cfg["scale"], rows=(r0, r1), shift=0.0)).pin_memory()
        qz_host = [torch.from_numpy(synth.make_fresh_queries(f, Q, cfg["seed"] + 100 + b_)[0]).pin_memory() for b_ in range(nbatch)]
        with torch.cuda.stream(stream):
            xz_dev = xz_host.to(dev, non_blocking=True)
            qz_dev = [q.to(dev, non_blocking=True) for q in qz_host]
            stream.synchronize()
            aspace, gl = build(xz_dev, mz_sw)
        # probe step (also builds the operand cache): a regime that fell onto the exact-scan path would take minutes --
        # then it is measured on ONE step and says so
        t0 = time.perf_counter()
        with torch.cuda.stream(stream):
            aspace.search_batch(qz_dev[0], gl, tau)
        torch.cuda.synchronize(dev)
        probe_s = max_over_ranks(time.perf_counter() - t0)
        mz_steps, mz_warm = (max(2, min(args.steps, 5)), 3) if probe_s < 2.0 else (1, 0)
        mz = search_regime(aspace, gl, qz_dev, qz_host, mz_steps, mz_warm)
        mz_lam, mz_rows, mz_edges = aspace.lambdas(), (aspace.row_offset, aspace.row_offset + aspace.nitems_local), gl.edges()
        regime = {"data": "unit rows x %g, no shift (entries of both signs); queries = fresh draws from the 256 clusters (no near-duplicate item)" % cfg["scale"],
                  "switches": mz_sw, "probe_step_s": probe_s, "value": Q / (mz["step_ms"] * 1e-3), "unit": "queries/s", "ms_per_step": mz["step_ms"], "steps": mz_steps,
                  "e2e": {"value": Q / (mz["e2e_ms"] * 1e-3), "unit": "queries/s", "ms_per_step": mz["e2e_ms"]},
                  "stage1_ms": mz["stage1_ms"], "stage2_ms": mz["stats"]["search_stage2_ms"], "mma_terms": int(mz["stats"]["search_terms"]),
                  "query_operand_resident": mz["stats"]["search_a_resident"] == 1.0,
                  "three_term_retry_queries_last_step": mz["stats"].get("search_retry_queries"),
                  "survivors_per_query": mz["stats"]["search_rescored_per_query"], "exact_rescan_queries_last_step": mz["stats"]["search_slow_queries"],
                  "band_cos_max": mz["stats"]["search_delta_cos_max"],
                  "residual_norms": {"rho_q_max": mz["stats"]["search_rho_q_max"], "rho_x_max": mz["stats"]["search_rho_x_max"]},
                  "algorithmic_tflops": 2.0 * q_rank * n_shard * f / (mz["stage1_ms"] * 1e-3) / 1e12}
        del aspace, gl, xz_dev, qz_dev

    # ---- item graph (nodes = items) of the same matrix: the graph-build workload of C4 (eps / k-NN lists of all 1M items
    # against all 1M items on the tensor cores, exact stage 2, Laplacian CSR); sharded over the ranks when N > 1
    item_graph = None
    if not args.no_item_graph:
        ig_ms = []
        with torch.cuda.stream(stream):
            for rep in range(2):
                barrier_sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                if world == 1:
                    a_ig, g_ig = ArrowSpaceBuilder.build_item_graph(gp, x_dev, device=local)
                else:
                    a_ig, g_ig = ArrowSpaceBuilder.build_item_graph_sharded(gp, x_dev, n, r0, device=local)
                e1.record(stream)
                barrier_sync()
                ig_ms.append(max_over_ranks(e0.elapsed_time(e1)))
                ig_nnz = g_ig.nnz
                ig_stats = {k: api.stat(k, local) for k in ("knn_stage1_ms", "knn_stage2_ms", "knn_slow_rows", "knn_rescored_per_row")}
                del a_ig, g_ig
        ig_exec = 2.0 * n * (r1 - r0) * 16.0 * ((f + 3 + 15) // 16)
        ig_alg = 2.0 * n * (r1 - r0) * f
        item_graph = {"ms": min(ig_ms), "items_per_s": n / (min(ig_ms) * 1e-3), "nnz": int(ig_nnz),
                      "rows_per_rank": r1 - r0, "stage1_ms": ig_stats["knn_stage1_ms"], "stage2_ms": ig_stats["knn_stage2_ms"],
                      "exact_scan_rows": ig_stats["knn_slow_rows"], "rescored_per_row": ig_stats["knn_rescored_per_row"],
                      "algorithmic_flop": ig_alg, "executed_fp16_flop": ig_exec,
                      "stage1_algorithmic_tflops": ig_alg / (ig_stats["knn_stage1_ms"] * 1e-3) / 1e12 if ig_stats["knn_stage1_ms"] > 0 else None,
                      "stage1_tflops": ig_exec / (ig_stats["knn_stage1_ms"] * 1e-3) / 1e12 if ig_stats["knn_stage1_ms"] > 0 else None,
                      "note": "rows of this rank against all %d items; N > 1: + all-gather of the item shards and of the lists" % n}

    # ---- build with the pre-graph reduction the crate runs inside build (SURVEY.md 8(f)-1): sample 60 %, two-NN intrinsic
    # dimension, k-means, graph on the centroid matrix, lambdas of every item.  N > 1: sampled rows all-gathered, replicas.
    reduced = None
    if not args.no_reduction:
        red_ms = []
        with torch.cuda.stream(stream):
            for rep in range(2):
                barrier_sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                if world == 1:
                    a_rd, g_rd = ArrowSpaceBuilder.build(gp, x_dev, device=local, reduction=True)
                else:
                    a_rd, g_rd = ArrowSpaceBuilder.build_sharded(gp, x_dev, n, device=local, item_shards=world, reduction=True)
                e1.record(stream)
                barrier_sync()
                red_ms.append(max_over_ranks(e0.elapsed_time(e1)))
                rd_info = g_rd.reduction
                rd_stats = {k: api.stat(k, local) for k in ("reduce_two_nn_ms", "reduce_kmeans_ms", "reduce_assign_ms", "reduce_assign_passes")}
                del a_rd, g_rd
        dp_ops = 3.0 * rd_info["n_sampled"] * rd_info["n_clusters"] * f * rd_stats["reduce_assign_passes"]
        reduced = {"ms": min(red_ms), "items_per_s": n / (min(red_ms) * 1e-3), "info": rd_info,
                   "two_nn_ms": rd_stats["reduce_two_nn_ms"], "kmeans_ms": rd_stats["reduce_kmeans_ms"],
                   "assign": {"kernel": "sqdist_min2_kernel (squared distances in the oracle's order: subtract, multiply, add -- no FMA "
                                        "contraction under the parity contract; two smallest per row)",
                              "ms": rd_stats["reduce_assign_ms"], "passes": rd_stats["reduce_assign_passes"], "bound": "fp64 issue",
                              "dp_instructions": dp_ops, "achieved_per_s": dp_ops / (rd_stats["reduce_assign_ms"] * 1e-3),
                              "peak_per_s_at_max_clock": 148 * 64 * 1.965e9,
                              "frac_at_max_clock": dp_ops / (rd_stats["reduce_assign_ms"] * 1e-3) / (148 * 64 * 1.965e9)},
                   "note": "centroids bit-identical to the oracle's at test sizes (tests/test_gpu_parity.py); the reference spends "
                           "its ~2-minute build floor here (SURVEY.md section 6)"}

    if rank != 0:
        if world > 1:
            dist.barrier()                                            # rank 0 runs the untimed oracle checks meanwhile
            dist.destroy_process_group()
        return

    # ---- UNTIMED parity gate on the benchmarked configuration (VERDICT r01 next #1): oracle full scan of a sample of the
    # last step's queries against ALL items, for the device-resident and the end-to-end result (N > 1: the merged result)
    parity = None
    if args.parity_queries > 0:
        pick = np.unique(np.linspace(0, Q - 1, args.parity_queries).astype(np.int64))
        x_full = x_host.numpy() if world == 1 else synth.make_items(n, f, cfg["seed"], cfg["scale"])
        lb = main_run["last_batch"]
        parity = oracle_parity(gp, tau, x_full, q_host[lb].numpy()[pick],
                               {"device_resident": (main_run["idx"][pick], main_run["sc"][pick]),
                                "end_to_end": (main_run["idx_h"][pick], main_run["sc_h"][pick])},
                               lam_local, lam_rows, edges, {})
        if regime is not None:
            del x_full
            xz_full = xz_host.numpy() if world == 1 else synth.make_items(n, f, cfg["seed"], cfg["scale"], shift=0.0)
            lbz = mz["last_batch"]
            regime["parity_check"] = oracle_parity(gp, tau, xz_full, qz_host[lbz].numpy()[pick],
                                                   {"device_resident": (mz["idx"][pick], mz["sc"][pick]),
                                                    "end_to_end": (mz["idx_h"][pick], mz["sc_h"][pick])},
                                                   mz_lam, mz_rows, mz_edges, mz_sw)
            del xz_full

    gemm_flop = 2.0 * q_rank * n_shard * f                  # algorithmic: one f64-accurate score per (query, item) of this rank
    gram_ms = float(np.mean(stages["gram_ms"]))
    lam_ms = float(np.mean(stages["lambda_ms"]))
    n_local = r1 - r0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    prof = {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "roofline.json")))
    except Exception:
        pass

    def profiled(kernel, key):
        e = prof.get(kernel)
        if isinstance(e, dict) and e.get("n_items") == n_shard and e.get("n_queries") == q_rank and e.get("n_features") == f:
            return e.get(key)
        return None

    def profiled_traffic(kernel):
        """dram__bytes_read + write of one launch from the committed `ncu --set full` capture -- only when that capture was
        taken at THIS launch shape (items per rank, queries per rank, features); otherwise null, never a stale constant."""
        e = prof.get(kernel)
        if isinstance(e, dict) and e.get("n_items") == n_shard and e.get("n_queries") == q_rank and e.get("n_features") == f:
            return e.get("dram_bytes_per_launch")
        return None

    if stage1_is_tc:
        terms = int(sstat["search_terms"])
        ksteps = (f + 3 + 15) // 16 + (2 * ((f + 15) // 16) if terms == 3 else 0)   # K=16 MMA steps per (query, item) tile pair
        executed = 2.0 * q_rank * n_shard * 16.0 * ksteps
        sustained = peaks.get("bf16_tflops_sustained", 1400.0)
        burst = peaks.get("bf16_tflops", sustained)
        achieved = gemm_flop / (stage1_ms * 1e-3) / 1e12
        executed_tflops = executed / (stage1_ms * 1e-3) / 1e12
        # the kernel is timed inside a long step: the sustained figure is the prescribed denominator.  The figure was
        # measured (cuBLAS bf16, 4 s back to back) at the clocks THAT workload reached under the power cap; this kernel draws
        # less power per FLOP and can clock higher, so its executed FLOP rate can exceed it -- the burst fraction is printed
        # next to it, and profiles/ holds the clock-independent figure (ncu sm__pipe_tensor_cycles_active)
        peak = sustained
        roofline = {"kernel": "tc_gemm_kernel (tcgen05.mma kind::f16, fp16 operands, f32 TMEM accumulators, TMA SWIZZLE_128B; items in "
                              "lambda order, rank-1 mean-direction term + %s of the residuals; single-compare epilogue, thresholds "
                              "shared across CTAs); exact f64 stage 2 follows"
                              % ("ONE fp16 term" if terms == 1 else "the two-term fp16 split (3 MMA terms)"),
                    "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "peak_nominal": 2250.0, "frac_of_nominal": achieved / 2250.0,     # dense 16-bit datasheet figure (SURVEY.md 8(d): report both)
                    "traffic": profiled_traffic("tc_gemm_kernel"),
                    "algorithmic": "ALGORITHMIC 2*Q_rank*N_shard*F = 2*%d*%d*%d = %.3e FLOP per launch (achieved / frac); the kernel EXECUTES "
                                   "2*Q_rank*N_shard*16*%d = %.3e fp16 tensor FLOP (K padded to 16%s)"
                                   % (q_rank, n_shard, f, gemm_flop, ksteps, executed, ", three split terms" if terms == 3 else ""),
                    "executed_tflops": executed_tflops, "executed_frac": executed_tflops / peak,
                    "peak_burst": burst, "frac_of_burst": achieved / burst, "executed_frac_of_burst": executed_tflops / burst,
                    # clock-independent evidence from the committed capture of this launch shape (profiles/ncu_full_r02.json)
                    "ncu_tensor_pipe_active_pct": profiled("tc_gemm_kernel", "tensor_pipe_active_pct"),
                    "fp64_tensor_peak_tflops": fp64_peak_tflops,
                    "kernel_ms": stage1_ms, "share_of_step": stage1_ms / step_ms,
                    "stage2_ms": sstat["search_stage2_ms"],
                    "mma_terms": terms, "query_operand_resident": sstat["search_a_resident"] == 1.0,
                    "band_cos_max": sstat["search_delta_cos_max"],
                    "residual_norms": {"rho_q_max": sstat["search_rho_q_max"], "rho_x_max": sstat["search_rho_x_max"]},
                    "rescored_candidates_per_query": rescored,
                    "reference_order_rescored_per_query": sstat["search_exact_per_query"],
                    "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
                                    + ("; executed FLOP rate above it: this kernel held higher clocks under the power cap than the "
                                       "cuBLAS run that set the figure -- see frac_of_burst and the ncu tensor-pipe activity in profiles/"
                                       if executed_tflops > sustained else ""))
                                   if "bf16_tflops_sustained" in peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"}
    else:
        achieved = gemm_flop / (stage1_ms * 1e-3) / 1e12
        roofline = {"kernel": "search_gemm_kernel (FP64 DMMA.8x8x4, TMA fed, fused score/top-k epilogue)",
                    "bound": "tensor", "achieved": achieved, "peak": fp64_peak_tflops, "unit": "TFLOP/s",
                    "frac": achieved / fp64_peak_tflops, "traffic": profiled_traffic("search_gemm_kernel"),
                    "algorithmic": "2*Q_rank*N_shard*F = %.3e FLOP per launch" % gemm_flop,
                    "kernel_ms": stage1_ms, "share_of_step": stage1_ms / step_ms,
                    "peak_source": "cuBLAS DGEMM 4096^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry)"}
    upper_nnz = (feature_graph_nnz - f) // 2
    sm_mhz = (clk or {}).get("sm_mhz") or 1900.0
    lam_bytes = 8.0 * n_local * f + 8.0 * n_local
    lam_flop = 2.0 * n_local * (2.0 * upper_nnz + f) + 4.0 * n_local * f          # SURVEY.md 8(d) K3: 2*N*nnz(L) + 4*N*F
    gather_floor_ms = 8.0 * n_local * upper_nnz / (148 * 128.0 * sm_mhz * 1e6) * 1e3
    line = {
        "metric": "search queries/s (top-10, 1M x 384 f64)",
        "value": Q / (step_ms * 1e-3), "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C4 BEIR/MS MARCO-shaped synthetic %d x %d f64 items (seed %d, x%g), %d queries per step, top-%d, tau %.2f"
                               % (n, f, cfg["seed"], cfg["scale"], Q, topk, tau),
                   "graph_params": gp, "queries_per_step": Q,
                   "sharding": "build: rows over %d rank(s); search: %d item shard(s) x %d query slot(s)" % (world, grid["R"], grid["C"]),
                   "l2": "inputs larger than L2 (item shard %.2f GB f64 + %.2f GB fp16 operands)" % (n_shard * f * 8 / 1e9, n_shard * (((f + 3 + 63) // 64) * 64) * 2 / 1e9),
                   "stage1": "tcgen05 fp16 candidates + exact f64 rescoring" if stage1_is_tc else "FP64 DMMA",
                   "exact_rescan_queries_last_step": slow},
        "e2e": {"value": Q / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": Q * f * 8, "d2h_bytes_per_step": Q * topk * 16 * world,
                "note": "per step, summed over ranks: every rank uploads its slice of the batch and reads back the whole result"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "parity_check": parity,
        "regimes": {"mean_zero": regime},
        "build": {"items_per_s": n / (float(np.mean(build_ms)) * 1e-3), "ms": float(np.mean(build_ms)),
                  "e2e_items_per_s": n / (min(build_e2e_ms) * 1e-3), "e2e_ms": min(build_e2e_ms),
                  "h2d_bytes": n_local * f * 8, "gpu_launches": int(build_launches),
                  "gram": gram_roofline(n_local, f, gram_ms, fp64_peak_tflops),
                  "graph_ms": float(np.mean(stages["graph_ms"])),
                  "lambda": {"kernel": "taumode_kernel (ONE pass over X: transposed tile + graph walk + median + norms)",
                             "ms": lam_ms, "bound": "hbm", "achieved_gbs": lam_bytes / (lam_ms * 1e-3) / 1e9,
                             "frac": lam_bytes / (lam_ms * 1e-3) / 1e9 / hbm_peak, "peak_gbs": hbm_peak,
                             # SURVEY.md 8(d): at nnz(L)/F > 16 the prescribed bound is FP64 FMA, not HBM
                             "fp64_fma": {"flop": lam_flop, "achieved_tflops": lam_flop / (lam_ms * 1e-3) / 1e12,
                                          "peak_tflops": fp64_peak_tflops, "frac": lam_flop / (lam_ms * 1e-3) / 1e12 / fp64_peak_tflops,
                                          "nnz_over_f": (feature_graph_nnz - f) / float(f)},
                             # the bound that actually binds at this graph density: one 8-byte shared-memory gather per
                             # strictly-upper non-zero of L per item (DESIGN.md section 4, K3), against 128 B/clk/SM
                             "gather": {"upper_nnz": upper_nnz, "smem_bytes": 8.0 * n_local * upper_nnz,
                                        "smem_floor_ms": gather_floor_ms, "frac_of_smem_floor": gather_floor_ms / lam_ms}}},
        "item_graph": item_graph,
        "reduced_build": reduced,
        "single_query": single,
        "clocks": clk,
    }
    if world == 1 and not args.no_hybrid:
        line["hybrid"] = hybrid_leg(args, n, local)
    if not args.no_cpu_baseline:
        ns = min(n, args.cpu_sample_items)
        r = cpu_oracle_run(dict(cfg, n=n), ns, args.cpu_sample_queries, 3, "sample")
        per_q = min(r["search_s"]) / r["nq"] * (n / ns)           # a scan is linear in the item count
        line["cpu_baseline"] = {
            "value": 1.0 / per_q, "unit": "queries/s", "cores": r["threads"], "kind": "port",
            "sample": "oracle (C + OpenMP) on the first %d items and %d queries of the workload; search time scaled x%.0f "
                      "to %d items (linear scan); oracle build of the sample %.2f s = %.0f items/s"
                      % (ns, r["nq"], n / ns, n, r["build_s"], ns / r["build_s"]),
            "build_items_per_s": ns / r["build_s"]}
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
