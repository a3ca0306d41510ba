"""python tools/filtered_search_time.py [out.json]

Filtered search at C4 (1M x 384, topk = 10, tau = 0.62) on one GPU: search_batch with allowed=None and with masks of
density 1.0, 0.5, 0.1, 0.01 and 0.001, for 65536 device queries per call and for 16384 host queries per call.  The cases
are interleaved with unfiltered calls (one filtered call, one unfiltered call, ...), so both see the same clocks and
neighbours; per case the median and the spread of REPS timed calls after one warm-up call, each ending in a device
synchronise.  Per case also the stats of the last call: search_slow_queries (queries answered by the exact scan),
search_retry_queries (the three-term retry) and search_rescored_per_query (survivors per query).  The filtered answers
of the density-1.0 mask must be the bits of the unfiltered ones.  Prints one JSON line per case with the GPU model and
power limit read in the same run; the whole result is written to out.json only when a path is given.  The item matrix
(3 GB) is larger than L2."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from pyarrowspace_b200 import synth  # noqa: E402
from pyarrowspace_b200.api import ArrowSpaceBuilder, stat  # noqa: E402

REPS = 7
DENSITIES = (None, 1.0, 0.5, 0.1, 0.01, 0.001)
BATCHES = (("device", 65536), ("host", 16384))


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cfg = synth.config("C4")
    n, f, tau = cfg["n"], cfg["f"], cfg["tau"]
    x = synth.make_items(n, f, cfg["seed"], cfg["scale"])
    aspace, gl = ArrowSpaceBuilder.build(cfg["graph_params"], x, device=0)
    rng = np.random.default_rng(5)
    out = {"gpu": gpu, "n": n, "f": f, "topk": cfg["graph_params"]["topk"], "tau": tau, "reps": REPS, "cases": []}
    for where, nq in BATCHES:
        q, _ = synth.make_queries(x, nq, cfg["seed"], cfg["scale"])
        qd = torch.from_numpy(q).cuda() if where == "device" else q
        for d in DENSITIES:
            mask = None if d is None else (np.ones(n, dtype=bool) if d == 1.0 else rng.random(n) < d)
            aspace.search_batch(qd, gl, tau, allowed=mask)      # warm-up
            ts_f, ts_u = [], []
            for _ in range(REPS):                              # interleaved: filtered, unfiltered, filtered, ...
                t, res_f = timed_once(lambda: aspace.search_batch(qd, gl, tau, allowed=mask))
                ts_f.append(t)
                st = {k: stat(k) for k in ("search_slow_queries", "search_retry_queries", "search_rescored_per_query")}
                t, res_u = timed_once(lambda: aspace.search_batch(qd, gl, tau))
                ts_u.append(t)
            fi, fs = (r.cpu().numpy() if torch.is_tensor(r) else r for r in res_f)
            ui, us = (r.cpu().numpy() if torch.is_tensor(r) else r for r in res_u)
            case = {"batch": where, "queries_per_call": nq, "density": d,
                    "allowed_items": n if mask is None else int(mask.sum()),
                    "filtered_ms_median": 1e3 * float(np.median(ts_f)), "filtered_ms_min_max": [1e3 * min(ts_f), 1e3 * max(ts_f)],
                    "unfiltered_ms_median": 1e3 * float(np.median(ts_u)), "unfiltered_ms_min_max": [1e3 * min(ts_u), 1e3 * max(ts_u)],
                    "filtered_over_unfiltered": float(np.median(ts_f) / np.median(ts_u)),
                    "filtered_queries_per_s": nq / float(np.median(ts_f))}
            case.update(st)
            if d in (None, 1.0):
                case["bits_equal_unfiltered"] = bool(np.array_equal(fi, ui) and np.array_equal(fs, us, equal_nan=True))
            out["cases"].append(case)
            print(json.dumps(dict(case, gpu=gpu)), flush=True)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            json.dump(out, fh, indent=1)


def timed_once(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, res


if __name__ == "__main__":
    main()
