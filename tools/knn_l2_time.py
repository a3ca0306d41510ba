"""The Euclidean item graph at C4 (1M x 384, the synth C4 matrix, k = 25) on one GPU, beside the cosine one in the same
process.  eps for l2 = the 10th / 50th / 90th percentile of the 25th-neighbour distance of a 2,000-row sample (f64 brute
force on the GPU).  Per run: wall time, stage 1 / stage 2 ms, survivors per row, two-term rows, exact-scan rows, nnz, and a
check of SAMPLE rows against all columns: the row's neighbour list must be the f64 brute-force top-k (ties within 1e-9
relative are accepted in either order) with the same distances to 1e-9.

    python tools/knn_l2_time.py [n=1000000] [sample=1000] [out.json]
Every run is printed as one JSON line; the whole result is also written to out.json when that path is given."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from pyarrowspace_b200 import api, synth  # noqa: E402
from pyarrowspace_b200.api import ArrowSpaceBuilder  # noqa: E402
from pyarrowspace_b200.distributed import CudaEngine  # noqa: E402
from pyarrowspace_b200 import _lib  # noqa: E402

STATS = ("knn_stage1_ms", "knn_stage2_ms", "knn_slow_rows", "knn_rows_two_term", "knn_rows_one_term_wasted", "knn_rescored_per_row",
         "knn_stage1_is_tc")


def brute(x, rows, k):
    """(distances, indices) of the k+1 nearest items of each row, f64 Gram form, self removed afterwards."""
    nsq = (x * x).sum(1)
    d_all, i_all = [], []
    for c0 in range(0, len(rows), 250):
        r = rows[c0:c0 + 250]
        d2 = (nsq[r, None] + nsq[None, :] - 2.0 * x[r] @ x.T).clamp_min_(0.0)
        d2[torch.arange(len(r)), r] = float("inf")
        v, i = torch.topk(d2, k + 8, dim=1, largest=False)
        d_all.append(v.sqrt().cpu().numpy()); i_all.append(i.cpu().numpy())
    return np.concatenate(d_all), np.concatenate(i_all)


def check_rows(x, rows, k, eps, idx, dst, cnt):
    """Rows whose list differs from the brute force: count min(k, #{d <= eps}) (either side of a 1e-9 band around eps),
    distances to 1e-9, and every neighbour a brute-force candidate within 1e-9 of its distance."""
    bd, bi = brute(x, torch.from_numpy(rows).cuda(), k)
    bad = 0
    for r in range(len(rows)):
        c = int(cnt[r])
        lo = min(k, int((bd[r] <= eps * (1 - 1e-9)).sum()))
        hi = min(k, int((bd[r] <= eps * (1 + 1e-9)).sum()))
        ok = lo <= c <= hi and np.allclose(dst[r, :c], bd[r, :c], rtol=1e-9, atol=0)
        for j, d in zip(idx[r, :c], dst[r, :c]):
            near = np.abs(bd[r] - d) <= 1e-9 * max(d, 1e-300)
            ok = ok and int(j) in set(int(v) for v in bi[r][near])
        bad += 0 if ok else 1
    return bad


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
    sample = int(sys.argv[2]) if len(sys.argv) > 2 else 1000
    c = synth.config("C4")
    f = c["f"]
    x = torch.from_numpy(synth.make_items(n, f, c["seed"], c["scale"])).cuda()
    k = 25
    rng = np.random.default_rng(7)
    rows2k = rng.choice(n, 2000, replace=False)
    bd, _ = brute(x, torch.from_numpy(rows2k).cuda(), k)
    kth = bd[:, k - 1]
    eps_list = [float(np.percentile(kth, q)) for q in (10, 50, 90)]
    out = {"n": n, "f": f, "k": k, "gpu": torch.cuda.get_device_name(0), "eps_percentiles_10_50_90": eps_list, "runs": []}
    check_rows_idx = np.sort(rng.choice(n, sample, replace=False)).astype(np.int64)
    eng = CudaEngine(0)
    space = eng.full_space(x)

    def one(distance, eps):
        gp = {"eps": eps, "k": k, "topk": 10, "p": 2.0, "sigma": None}
        walls = []
        for rep in range(2):
            torch.cuda.synchronize(); t0 = time.time()
            aspace, gl = ArrowSpaceBuilder.build_item_graph(gp, x, distance=distance)
            torch.cuda.synchronize(); walls.append(time.time() - t0)
            st = {s: api.stat(s) for s in STATS}
            nnz = int(gl.nnz)
            del aspace, gl
        run = {"distance": distance, "eps": eps, "wall_s": walls[-1], "wall_s_first": walls[0], "nnz": nnz, **st}
        if distance == "l2":
            cgp = _lib.make_params(eps, k, 10, 2.0, None)
            sw = _lib.make_switches(distance="l2")
            # the neighbour lists of every row (asp_item_knn_rows), the sampled ones against the brute force
            i_all, d_all, c_all = eng.knn_rows(space, cgp, 0, n, sw)
            i_s, d_s, c_s = (t[torch.from_numpy(check_rows_idx).cuda()].cpu().numpy() for t in (i_all, d_all, c_all))
            bad = check_rows(x, check_rows_idx, k, eps, i_s, d_s, c_s)
            run["checked_rows"] = int(sample)
            run["check_mismatches"] = int(bad)
        print(json.dumps(run), flush=True)
        out["runs"].append(run)

    one("cosine", c["graph_params"]["eps"])
    for eps in eps_list:
        one("l2", eps)
    one("cosine", c["graph_params"]["eps"])                          # again, after the l2 runs: same process, same state
    print(json.dumps(out), flush=True)
    if len(sys.argv) > 3:
        with open(sys.argv[3], "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
