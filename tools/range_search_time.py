"""python tools/range_search_time.py [out.json]

Range search at C4 (1M x 384, tau = 0.62) on one GPU: search_range_batch for 65536 device queries per call and for 16384
host queries per call, at four thresholds chosen so that the mean number of hits per query is about 1, 10, 100 and 1000.
The thresholds come from a 256-query sample: lambda_q from search_batch, every item's score of the sample in torch f64 (a
matrix product, not the reference order: it only picks the thresholds), the median over the sample of the k-th best.
Each range call is interleaved with a search_batch call (topk = 10) over the same batch for scale, so both see the same
clocks and neighbours; per case the median and the spread of REPS timed calls after one warm-up call, each ending in a
device synchronise, queries/s, hits/query, and the stats of the last range call: search_slow_queries (queries answered by
the exact range scan) and the split between stage 1 (the tcgen05 candidate pass, device events) and stage 2 (everything
after it: exact scores, the scan, the host round trip for the counts, the fill and the sort).  Prints one JSON line per
case with the GPU model and power limit read in the same run; the whole result is written to out.json only when a path
is given.  The item matrix (3 GB) is larger than L2."""
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

REPS = 5
LEVELS = (1, 10, 100, 1000)
BATCHES = (("device", 65536), ("host", 16384))


def thresholds(aspace, gl, x, tau, q):
    """min_score per level: the median over the sample of its level-th best score (torch f64, all items)."""
    _, _, lam_q = aspace._search_batch(q, gl, tau, want_lambda=True)
    xd = torch.from_numpy(x).cuda()
    xn = xd / xd.norm(dim=1, keepdim=True)
    lam_x = torch.from_numpy(aspace.lambdas()).cuda()
    out = {}
    qd = torch.from_numpy(q).cuda()
    qn = qd / qd.norm(dim=1, keepdim=True)
    lq = torch.from_numpy(np.asarray(lam_q)).cuda()
    best = []
    for i in range(0, q.shape[0], 32):
        sc = tau * (qn[i:i + 32] @ xn.T) + (1 - tau) / (1 + (lq[i:i + 32, None] - lam_x[None, :]).abs())
        best.append(torch.topk(sc, max(LEVELS), dim=1).values.cpu())
    best = torch.cat(best).numpy()
    for k in LEVELS:
        out[k] = float(np.median(best[:, k - 1]))
    return out


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cfg = synth.config("C4")
    n, f, tau = cfg["n"], cfg["f"], cfg["tau"]
    x = synth.make_items(n, f, cfg["seed"], cfg["scale"])
    aspace, gl = ArrowSpaceBuilder.build(cfg["graph_params"], x, device=0)
    sample, _ = synth.make_queries(x, 256, cfg["seed"] + 7, cfg["scale"])
    thr = thresholds(aspace, gl, x, tau, sample)
    out = {"gpu": gpu, "n": n, "f": f, "tau": tau, "reps": REPS, "thresholds": {str(k): v for k, v in thr.items()}, "cases": []}
    for where, nq in BATCHES:
        q, _ = synth.make_queries(x, nq, cfg["seed"], cfg["scale"])
        qd = torch.from_numpy(q).cuda() if where == "device" else q
        aspace.search_batch(qd, gl, tau)                      # warm-up of the search used for scale
        for level in LEVELS:
            run = lambda: aspace.search_range_batch(qd, gl, tau, thr[level], max_results=1 << 28)   # noqa: E731
            run()                                              # warm-up
            ts_r, ts_s = [], []
            for _ in range(REPS):                              # interleaved: range, search, range, ...
                t, res = timed_once(run)
                ts_r.append(t)
                st = {k: stat(k) for k in ("search_slow_queries", "range_stage1_ms", "range_stage2_ms", "range_stage1_is_tc")}
                t, _ = timed_once(lambda: aspace.search_batch(qd, gl, tau))
                ts_s.append(t)
            hits = int(res[0][-1])
            case = {"batch": where, "queries_per_call": nq, "target_hits_per_query": level, "min_score": thr[level],
                    "hits_per_query": hits / nq,
                    "range_ms_median": 1e3 * float(np.median(ts_r)), "range_ms_min_max": [1e3 * min(ts_r), 1e3 * max(ts_r)],
                    "range_queries_per_s": nq / float(np.median(ts_r)),
                    "search_batch_topk10_ms_median": 1e3 * float(np.median(ts_s)),
                    "search_batch_topk10_ms_min_max": [1e3 * min(ts_s), 1e3 * max(ts_s)]}
            case.update(st)
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
