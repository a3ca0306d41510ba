"""Times the item-graph build (nodes = items) on device-generated data: tcgen05 candidate pass vs FP64 DMMA.
    python tools/knn_time.py [n] [f] [modes=tc,fp64] [distance=cosine|l2|l2sq]
(l2 / l2sq: the "fp64" mode is the batched exact scan on every row; eps=... in the environment sets eps.)"""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from pyarrowspace_b200 import api
from pyarrowspace_b200.api import ArrowSpaceBuilder
n = int(sys.argv[1]) if len(sys.argv) > 1 else 200000
f = int(sys.argv[2]) if len(sys.argv) > 2 else 384
modes = sys.argv[3].split(",") if len(sys.argv) > 3 else ["tc", "fp64"]
distance = sys.argv[4] if len(sys.argv) > 4 else "cosine"
g = torch.Generator(device="cuda").manual_seed(1)
ncl = int(os.environ.get("NCL", 256))             # fewer clusters = denser neighbourhoods (C5 regime: 34k items per cluster)
centres = torch.randn(ncl, f, generator=g, device="cuda", dtype=torch.float64)
lab = torch.randint(0, ncl, (n,), generator=g, device="cuda")
x = centres[lab] + 0.3 * torch.randn(n, f, generator=g, device="cuda", dtype=torch.float64)
x = x / x.norm(dim=1, keepdim=True) * 100.0 + 25.0
gp = {"eps": 10.0, "k": 25, "topk": 10, "p": 2.0, "sigma": None}
if os.environ.get("SYNTH"):                      # the bench's C4 matrix
    from pyarrowspace_b200 import synth
    c = synth.config("C4")
    x = torch.from_numpy(synth.make_items(n, f, c["seed"], c["scale"])).cuda()
    gp = c["graph_params"]
if os.environ.get("EPS"):
    gp = dict(gp, eps=float(os.environ["EPS"]))
out = {"n": n, "f": f, "distance": distance, "eps": gp["eps"]}
for mode in modes:
    os.environ["ASP_KNN_STAGE1"] = mode
    for rep in range(2):
        torch.cuda.synchronize(); t0 = time.time()
        aspace, gl = ArrowSpaceBuilder.build_item_graph(gp, x, distance=distance)
        torch.cuda.synchronize(); dt = time.time() - t0
        st = {k: api.stat(k) for k in ("knn_stage1_ms", "knn_stage2_ms", "knn_slow_rows", "knn_rows_two_term", "knn_rows_one_term_wasted", "knn_rescored_per_row", "knn_stage1_is_tc")}
        print(mode, rep, "wall %.3f s" % dt, st, "nnz", gl.nnz if hasattr(gl, "nnz") else None, flush=True)
        del aspace, gl
    out[mode] = dict(st, wall_s=dt)
json.dump(out, open(os.path.join(ROOT, "gpurun_out", "knn_time.json"), "w"), indent=1)
