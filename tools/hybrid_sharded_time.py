"""torchrun --nproc-per-node G tools/hybrid_sharded_time.py [out.json]

Queries/s of search_hybrid_batch at C4 (1M x 384, topk = 10, tau = 0.62) on G GPUs for the search layouts R = 8, 2, 1 item
shards that divide G (build_sharded(item_shards=R)), 16384 host queries per call, pool 20 and 31, each beside search_batch
at topk = pool on the same layout in the same run (the sharded hybrid exchanges R * pool * 24 bytes per query, the sharded
search R * pool * 16).  Per case: the median and the spread of REPS timed calls after one warm-up call, each call between
two barriers with every device synchronised.  The hybrid answers of every layout must be the same bits as the first
layout's.  Rank 0 prints one JSON line per case, with the GPU model and power limit; the whole result is written to
out.json when a path is given.  The item matrix (3 GB) is larger than L2."""
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from pyarrowspace_b200 import shard_rows, synth  # noqa: E402
from pyarrowspace_b200.api import ArrowSpaceBuilder  # noqa: E402

NQ = 16384
REPS = 7
POOLS = (20, 31)


def timed(fn):
    fn()                                                      # warm-up: every shape of the timed calls
    ts = []
    for _ in range(REPS):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        dist.barrier()
        ts.append(time.perf_counter() - t0)
    return sorted(ts), out


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                         capture_output=True, text=True).stdout.strip()
    cfg = synth.config("C4")
    n, f, tau = cfg["n"], cfg["f"], cfg["tau"]
    r0, r1 = shard_rows(n, world, rank)
    shard = synth.make_items(n, f, cfg["seed"], cfg["scale"], rows=(r0, r1))
    q, _ = synth.make_queries(synth.make_items(n, f, cfg["seed"], cfg["scale"], rows=(0, 65536)), NQ, cfg["seed"], cfg["scale"])
    out = {"gpu": gpu, "gpus": world, "n": n, "f": f, "topk": cfg["graph_params"]["topk"], "tau": tau,
           "queries_per_call": NQ, "reps": REPS, "cases": []}
    first = {}
    for R in [r for r in (8, 2, 1) if r <= world and world % r == 0]:
        aspace, gl = ArrowSpaceBuilder.build_sharded(cfg["graph_params"], shard, n, device=local, item_shards=R)
        for pool in POOLS:
            th, (hi, hs) = timed(lambda: aspace.search_hybrid_batch(q, gl, tau, pool=pool))
            crc = zlib.crc32(hi.tobytes() + hs.tobytes())
            same = first.setdefault(pool, crc) == crc
            a2, g2 = ArrowSpaceBuilder.build_sharded(dict(cfg["graph_params"], topk=pool), shard, n, device=local,
                                                     item_shards=R)
            tsr, _ = timed(lambda: a2.search_batch(q, g2, tau))
            del a2, g2
            t = torch.tensor([1 if same else 0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            case = {"item_shards": R, "query_slots": world // R, "pool": pool,
                    "hybrid_ms_median": 1e3 * float(np.median(th)), "hybrid_ms_min_max": [1e3 * th[0], 1e3 * th[-1]],
                    "hybrid_queries_per_s": NQ / float(np.median(th)),
                    "search_topk_eq_pool_ms_median": 1e3 * float(np.median(tsr)),
                    "search_topk_eq_pool_ms_min_max": [1e3 * tsr[0], 1e3 * tsr[-1]],
                    "search_topk_eq_pool_queries_per_s": NQ / float(np.median(tsr)),
                    "hybrid_over_search_time": float(np.median(th) / np.median(tsr)),
                    "hybrid_bits_equal_first_layout_all_ranks": bool(t.item())}
            out["cases"].append(case)
            if rank == 0:
                print(json.dumps(dict(case, gpu=gpu, gpus=world)), flush=True)
        del aspace, gl
        dist.barrier()
    if rank == 0 and len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            json.dump(out, fh, indent=1)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
