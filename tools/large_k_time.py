"""python tools/large_k_time.py [out.json] [--ks 10,32,64]

Search with a per-call k at C4 (1M x 384, tau = 0.62) on one GPU: search_batch(k=K) on the C4 graph (topk = 10) against
the same K through the graph-topk route (a graph built with topk = K, default switches: same graph and lambdas, same
answers), for K in {10, 32, 64, 100, 128} and 8192 / 65536 host queries per call.  The graph-topk route takes the batched
exact scan of every query for K >= 32, so its 65536-query calls at K >= 32 are timed once (REPS_SLOW), and so is every
call at K > 64, where search_batch(k=) takes the same exact scan.  Per case the
median of REPS timed calls after one warm-up call, each ending with the results on the host; the stats of the last call
(search_stage1_is_tc, search_slow_queries, search_retry_queries).  Parity, in the same run: the two routes give the same
bits on every query, and a sample of SAMPLE queries matches the oracle (indices identical, scores to 1e-9).  Prints one
JSON line per case with the GPU model and power limit read in the same run; the result goes to out.json when given, merged
with the cases of other K already there (--ks: a subset of K, so that the slow exact-scan cases can run separately).
The item matrix (3 GB) is larger than L2."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from pyarrowspace_b200 import synth  # noqa: E402
from pyarrowspace_b200.api import ArrowSpaceBuilder, stat  # noqa: E402

REPS, REPS_SLOW = 5, 1
KS = (10, 32, 64, 100, 128)
BATCHES = (8192, 65536)
SAMPLE = 16


def _time(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        res = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), res


def _oracle_ok(s, g, q, tau, k, idx, sc):
    """The sample against the oracle's scores of every item, ranked by (score desc, index asc) and cut to k."""
    from test_filtered_search_cpu import want_search
    lq = s.search_batch(q, g, tau)[2]
    wi, ws = want_search(s, q, lq, tau, np.ones(len(s.lambdas()), dtype=bool), k)
    ok = wi >= 0
    return bool(np.array_equal(idx, wi) and np.allclose(sc[ok], ws[ok], rtol=1e-9, atol=0))


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cfg = synth.config("C4")
    n, f, tau = cfg["n"], cfg["f"], cfg["tau"]
    x = synth.make_items(n, f, cfg["seed"], cfg["scale"])
    aspace, gl = ArrowSpaceBuilder.build(cfg["graph_params"], x, device=0)
    import oracle
    s_orc, g_orc = oracle.build(cfg["graph_params"], x)
    ks = KS
    if "--ks" in sys.argv:
        ks = tuple(int(v) for v in sys.argv[sys.argv.index("--ks") + 1].split(","))
    out = {"gpu": gpu, "n": n, "f": f, "graph_topk": cfg["graph_params"]["topk"], "tau": tau, "reps": REPS, "cases": []}
    q_all = synth.make_queries(x, max(BATCHES), cfg["seed"] + 7, cfg["scale"])[0]
    for k in ks:
        a2, g2 = (aspace, gl) if k == cfg["graph_params"]["topk"] else ArrowSpaceBuilder.build(dict(cfg["graph_params"], topk=k), x, device=0)
        for nq in BATCHES:
            q = np.ascontiguousarray(q_all[:nq])
            scan_k = k > 64                                    # search_batch(k=) beyond the tensor-core route: the exact scan
            t_k, (ik, sk) = _time(lambda: aspace.search_batch(q, gl, tau, k=k), REPS_SLOW if scan_k else REPS)
            st_k = {key: stat(key) for key in ("search_stage1_is_tc", "search_slow_queries", "search_retry_queries")}
            slow_old = k >= 32 and nq > 8192
            t_g, (ig, sg) = _time(lambda: a2.search_batch(q, g2, tau), REPS_SLOW if slow_old else REPS)
            st_g = {key: stat(key) for key in ("search_stage1_is_tc", "search_slow_queries")}
            same = bool(np.array_equal(ik, ig) and np.array_equal(sk, sg, equal_nan=True))
            pick = np.linspace(0, nq - 1, SAMPLE).astype(int)
            orc = _oracle_ok(s_orc, g_orc, np.ascontiguousarray(q[pick]), tau, k, ik[pick], sk[pick]) if nq == BATCHES[0] else None
            case = {"k": k, "queries": nq, "k_call_s": t_k, "k_call_qps": nq / t_k, "graph_topk_s": t_g, "graph_topk_qps": nq / t_g,
                    "speedup": t_g / t_k, "k_call_reps": REPS_SLOW if scan_k else REPS, "graph_topk_reps": REPS_SLOW if slow_old else REPS, "k_stats": st_k, "graph_topk_stats": st_g,
                    "same_bits": same, "oracle_sample_ok": orc, "gpu": gpu}
            print(json.dumps(case), flush=True)
            out["cases"].append(case)
        if a2 is not aspace:
            del a2, g2
    path = sys.argv[1] if len(sys.argv) > 1 and not sys.argv[1].startswith("--") else None
    if path and os.path.exists(path):
        with open(path) as fh:
            old = json.load(fh)
        out["cases"] = sorted([c for c in old["cases"] if c["k"] not in ks] + out["cases"], key=lambda c: (c["k"], c["queries"]))
    out["parity_ok"] = all(c["same_bits"] and c["oracle_sample_ok"] is not False for c in out["cases"])
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as fh:
            json.dump(out, fh, indent=1)
    print(json.dumps({"parity_ok": out["parity_ok"], "gpu": gpu}))


if __name__ == "__main__":
    main()
