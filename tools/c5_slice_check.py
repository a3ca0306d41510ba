"""BASELINE.json config C5, the oracle leg (SURVEY.md 8(d): "oracle checks a 100k-row slice only"): rows [0, SLICE) of the
8.8M x 768 matrix of tools/c5_sweep.py (same device generator, same seed / block offsets) as a stand-alone item graph on ONE
GPU, for every eps of the sweep {5, 10, 15} (/root/reference/tests/test_5_msmarco_eps_sweep.py:19-23), against the CPU
oracle's item graph of the same rows: CSR structure identical, values within 1e-9.

    python tools/c5_slice_check.py [SLICE=100000] [eps list=5,10,15]      -> gpurun_out/c5_slice_check.json"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import c5_sweep  # noqa: E402
import oracle  # noqa: E402
from pyarrowspace_b200 import api  # noqa: E402
from pyarrowspace_b200.api import ArrowSpaceBuilder  # noqa: E402


def main():
    m = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
    eps_list = [float(e) for e in (sys.argv[2] if len(sys.argv) > 2 else "5,10,15").split(",")]
    distance = sys.argv[3] if len(sys.argv) > 3 else "cosine"         # third argument: cosine | l2 | l2sq (recorded in the JSON)
    n, f = 8_800_000, 768
    dev = torch.device("cuda", 0)
    centres = torch.randn(c5_sweep.NCL, f, generator=torch.Generator(device=dev).manual_seed(c5_sweep.SEED), device=dev, dtype=torch.float64)
    x = c5_sweep.gen_rows(0, m, n, f, centres, dev)
    xh = x.cpu().numpy()
    try:
        oracle.set_num_threads(len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    out = {"slice_rows": m, "f": f, "distance": distance, "of_n": n, "runs": [], "oracle_threads": oracle.num_threads()}
    ok = True
    for eps in eps_list:
        gp = {"eps": eps, "k": 25, "topk": 10, "p": 2.0, "sigma": None}
        torch.cuda.synchronize(); t0 = time.time()
        aspace, gl = ArrowSpaceBuilder.build_item_graph(gp, x, distance=distance)
        torch.cuda.synchronize(); t_gpu = time.time() - t0
        st = {k: api.stat(k) for k in ("knn_stage1_ms", "knn_stage2_ms", "knn_slow_rows", "knn_rows_two_term", "knn_rescored_per_row")}
        t0 = time.time()
        s, g = oracle.build(gp, xh, nodes="items", distance=distance)
        t_cpu = time.time() - t0
        ip, ix, dt = gl.csr()
        oip, oix, odt = g.csr()
        same = bool(np.array_equal(ip, oip) and np.array_equal(ix, oix))
        rel = float(np.max(np.abs(dt - odt) / np.maximum(np.abs(odt), 1e-300))) if same else None
        run = {"eps": eps, "structure_equal": same, "data_max_rel_err": rel, "nnz": int(gl.nnz), "gpu_s": t_gpu, "oracle_s": t_cpu, **st}
        ok = ok and same and rel is not None and rel <= 1e-9
        print("C5 slice", json.dumps(run), flush=True)
        out["runs"].append(run)
        del aspace, gl, s, g
    out["ok"] = ok
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "c5_slice_check.json"), "w"), indent=1)
    print("C5_SLICE_CHECK", "OK" if ok else "FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
