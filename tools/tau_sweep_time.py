"""python tools/tau_sweep_time.py [out.json]

A tau sweep at C4 (1M x 384, graph topk 10) on one GPU: search_batch_taus(q, gl, taus) against the loop of
search_batch(q, gl, tau) over the same taus, for taus (1.0, 0.8, 0.62), (0.62, 0.5) and (1.0, 0.8, 0.62, 0.5) (two shared
passes of two), k = 10 and 16, no mask and a 0.1-density mask, 65536 device queries and 16384 host queries per call.  The
two routes alternate in the same process; per case the median of REPS timed calls after one warm-up call of each, every
call ending with its results where the caller gets them (a device synchronise for device batches).  Recorded per case: the
sweep's stage-1 and stage-2 ms (shared passes), emitted candidates per query, search_slow_queries per tau, and the loop's
summed stage-1 + stage-2 ms.  Parity, in the same run: the two routes give the same bits on every query, and a sample of
SAMPLE queries per tau matches the oracle (indices identical, scores to 1e-9).  The GPU model and power limit are read in
the same run.  The item matrix (3 GB) is larger than L2."""
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

REPS = 7
TAUS = ((1.0, 0.8, 0.62), (0.62, 0.5), (1.0, 0.8, 0.62, 0.5))
KS = (10, 16)
BATCHES = ((65536, "device"), (16384, "host"))
SAMPLE = 8


def _sync(res):
    import torch
    if hasattr(res[0], "is_cuda"):
        torch.cuda.synchronize()
    return res


def _oracle_ok(s, g, q, tau, k, mask, idx, sc):
    from test_filtered_search_cpu import want_search
    lq = s.search_batch(q, g, tau)[2]
    wi, ws = want_search(s, q, lq, tau, np.ones(len(s.lambdas()), dtype=bool) if mask is None else mask, k)
    ok = wi >= 0
    return bool(np.array_equal(idx, wi) and np.allclose(sc[ok], ws[ok], rtol=1e-9, atol=0))


def main():
    import torch
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cfg = synth.config("C4")
    n, f = cfg["n"], cfg["f"]
    x = synth.make_items(n, f, cfg["seed"], cfg["scale"])
    aspace, gl = ArrowSpaceBuilder.build(cfg["graph_params"], x, device=0)
    import oracle
    s_orc, g_orc = oracle.build(cfg["graph_params"], x)
    q_all = synth.make_queries(x, max(b for b, _ in BATCHES), cfg["seed"] + 7, cfg["scale"])[0]
    masks = {"none": None, "0.1": np.random.default_rng(3).random(n) < 0.1}
    out = {"gpu": gpu, "n": n, "f": f, "graph_topk": cfg["graph_params"]["topk"], "reps": REPS, "cases": []}
    for nq, where in BATCHES:
        q = np.ascontiguousarray(q_all[:nq])
        qin = torch.from_numpy(q).cuda() if where == "device" else q
        for taus in TAUS:
            for k in KS:
                for mname, mask in masks.items():
                    def sweep():
                        return _sync(aspace.search_batch_taus(qin, gl, taus, allowed=mask, k=k))

                    def loop():
                        return _sync([aspace.search_batch(qin, gl, t, allowed=mask, k=k) for t in taus])
                    sweep()
                    loop()
                    ts, tl = [], []
                    for _ in range(REPS):                      # alternate the two routes
                        t0 = time.perf_counter()
                        rs = sweep()
                        ts.append(time.perf_counter() - t0)
                        st_s = {key: stat(key) for key in ("sweep_stage1_ms", "sweep_stage2_ms", "sweep_emitted_per_query",
                                                           "sweep_fused_taus", "sweep_stage1_passes", "search_slow_queries")}
                        st_s["slow_per_tau"] = [stat("sweep_slow_queries_%d" % t) for t in range(len(taus))]
                        loop_ms, loop_slow = 0.0, []
                        t0 = time.perf_counter()
                        for t in taus:                         # the loop, with each call's stats read after it
                            r1 = _sync(aspace.search_batch(qin, gl, t, allowed=mask, k=k))
                            loop_ms += stat("search_stage1_ms") + stat("search_stage2_ms")
                            loop_slow.append(stat("search_slow_queries"))
                        tl.append(time.perf_counter() - t0)
                    rl = loop()
                    idx, sc = (rs[0].cpu().numpy(), rs[1].cpu().numpy()) if where == "device" else rs
                    same = True
                    orc = True
                    pick = np.linspace(0, nq - 1, SAMPLE).astype(int)
                    for t, tau in enumerate(taus):
                        i1, s1 = (rl[t][0].cpu().numpy(), rl[t][1].cpu().numpy()) if where == "device" else rl[t]
                        same &= bool(np.array_equal(idx[t], i1) and np.array_equal(sc[t], s1, equal_nan=True))
                        if nq == 16384:
                            orc &= _oracle_ok(s_orc, g_orc, np.ascontiguousarray(q[pick]), tau, k, mask, idx[t][pick], sc[t][pick])
                    t_s, t_l = float(np.median(ts)), float(np.median(tl))
                    case = {"queries": nq, "where": where, "taus": list(taus), "k": k, "mask": mname, "sweep_s": t_s, "loop_s": t_l,
                            "speedup": t_l / t_s, "sweep_stats": st_s, "loop_stage_ms": loop_ms, "loop_slow_per_tau": loop_slow,
                            "same_bits": same, "oracle_sample_ok": orc if nq == 16384 else None, "gpu": gpu}
                    print(json.dumps(case), flush=True)
                    out["cases"].append(case)
    out["parity_ok"] = all(c["same_bits"] and c["oracle_sample_ok"] is not False for c in out["cases"])
    path = sys.argv[1] if len(sys.argv) > 1 else None
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as fh:
            json.dump(out, fh, indent=1)
    print(json.dumps({"parity_ok": out["parity_ok"], "gpu": gpu}))


if __name__ == "__main__":
    main()
