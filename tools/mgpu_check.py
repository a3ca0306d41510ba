"""torchrun --nproc-per-node N tools/mgpu_check.py : multi-GPU build + search over NCCL against the CPU oracle and against
the single-GPU result (bit identical), for EVERY layout of the search grid (R item shards x N / R query slots: R = N fully
item-sharded ... R = 1 items replicated), with host and with device-resident query batches, and search_hybrid (host
batches, default shortlist and pool 40) against the single-GPU result (bit identical) and the oracle, and search_range_batch
(with and without a mask) against the single-GPU result (bit identical) and the definition over the oracle.

    BIG=1      adds the 1M x 384 case (BASELINE.json C4 shape; oracle check on a 96-query sample)
    CHECK_PEER=1 also runs the peer-memory merge (csrc/peer.cu) on the fully item-sharded layout
    QUICK=1    skips the item-graph part
Prints one line per check and MGPU_CHECK OK / FAILED; exit code 0 / 1."""
import os
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from pyarrowspace_b200 import shard_rows, synth  # noqa: E402
from pyarrowspace_b200.api import ArrowSpaceBuilder  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_filtered_search_cpu import want_hybrid, want_search  # noqa: E402  (the filtered searches by definition)
from test_range_search_cpu import want_range  # noqa: E402  (the range search by definition)

HYBRID_POOLS = (None, 40)     # search_hybrid shortlists: the default (tensor-core candidates) and the batched exact scan


def filter_mask(n):
    """The allowed= mask of the filtered checks: half the items, and none of the last rank's rows, the same on every rank."""
    mask = np.random.default_rng(n).random(n) < 0.5
    mask[shard_rows(n, dist.get_world_size(), dist.get_world_size() - 1)[0]:] = False
    return mask


def all_ranks(flag):
    t = torch.tensor([1 if flag else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    cases = [(20000, 96, {"eps": 0.5, "k": 6, "topk": 10, "p": 2.0, "sigma": 0.25}, 500, 500),
             (3001, 384, {"eps": 10.0, "k": 25, "topk": 10, "p": 2.0, "sigma": None}, 333, 333)]
    if os.environ.get("BIG"):
        c = synth.config("C4")
        cases.append((c["n"], c["f"], c["graph_params"], 65536, 96))
    for n, f, gp, nq, n_oracle in cases:
        big = n >= 500000
        r0, r1 = shard_rows(n, world, rank)
        seed, scale = (44, 100.0) if big else (9, 100.0)
        kw = {} if big else {"n_clusters": 16}
        shard = synth.make_items(n, f, seed, scale, rows=(r0, r1), **kw)
        qsrc = synth.make_items(n, f, seed, scale, rows=(0, min(n, 65536)), **kw)
        q, _ = synth.make_queries(qsrc, nq, seed, scale)
        q_dev = torch.from_numpy(q).cuda()
        ref = None
        if rank == 0:                                          # the single-GPU answer and the oracle's, once per case
            import oracle
            full = synth.make_items(n, f, seed, scale, **kw)
            a1, g1 = ArrowSpaceBuilder.build(gp, full, device=local)
            idx1, sc1 = a1.search_batch(q, g1, 0.62)
            pick = np.unique(np.linspace(0, nq - 1, n_oracle).astype(np.int64))
            s, g = oracle.build(gp, full)
            oidx, osc, _ = s.search_batch(q[pick], g, 0.62)
            ref = dict(idx1=idx1, sc1=sc1, lam1=a1.lambdas(), csr1=g1.csr(), pick=pick, oidx=oidx, osc=osc, olam=s.lambdas(), oedges=g.edges())
            for pool in HYBRID_POOLS:                         # search_hybrid: one GPU and the oracle's restatement
                ref["hyb1", pool] = a1.search_hybrid_batch(q, g1, 0.62, pool=pool)
                ref["hybo", pool] = s.search_hybrid_batch(q[pick], g, 0.62, pool or 0)[:2]
            fmask = filter_mask(n)                            # filtered search and hybrid: one GPU and the oracle
            ref["filt1"] = a1.search_batch(q, g1, 0.62, allowed=fmask)
            ref["filto"] = want_search(s, q[pick], s.search_batch(q[pick], g, 0.62)[2], 0.62, fmask, gp["topk"])
            ref["fhyb1"] = a1.search_hybrid_batch(q, g1, 0.62, allowed=fmask)
            ref["fhybo"] = want_hybrid(s, q[pick], s.search_hybrid_batch(q[pick], g, 0.62, 0)[2], 0.62, 0, fmask, gp["topk"])
            thr = float(np.median(sc1[:, -1]))                # range search: about topk hits per query
            olq = s.search_batch(q[pick], g, 0.62)[2]
            for m_ in (None, fmask):
                ref["rng1", m_ is None] = a1.search_range_batch(q, g1, 0.62, thr, allowed=m_)
                ref["rngo", m_ is None] = [want_range(s, q[i], olq[j], 0.62, thr, m_) for j, i in enumerate(pick)]
            ref["thr"] = thr
            ar, gr = ArrowSpaceBuilder.build(gp, full, device=local, reduction=True)      # pre-graph reduction, one GPU
            ref.update(red_csr=gr.csr(), red_lam=ar.lambdas(), red_cent=gr.centroids(), red_info=gr.reduction)
            del a1, g1, s, g, full, ar, gr
        dist.barrier()
        # pre-graph reduction across the ranks: sampled rows all-gathered, replicated k-means == the single-GPU one
        aspace, gl = ArrowSpaceBuilder.build_sharded(gp, shard, n, device=local, item_shards=world, reduction=True)
        cent, lam, lr0 = gl.centroids(), aspace.lambdas(), aspace.row_offset
        same = True
        if rank == 0:
            same = (np.array_equal(cent, ref["red_cent"]) and all(np.array_equal(a, b) for a, b in zip(gl.csr(), ref["red_csr"]))
                    and np.array_equal(lam, ref["red_lam"][lr0:lr0 + len(lam)]) and str(gl.reduction) == str(ref["red_info"]))
            print("world %d n %d f %d reduced build (K = %d, %d rows sampled): centroids / graph / lambdas / statistics == single GPU "
                  "(bitwise) %s" % (world, n, f, gl.reduction["n_clusters"], gl.reduction["n_sampled"], same), flush=True)
        ok = ok and same
        del aspace, gl
        dist.barrier()
        shards = [r for r in (world, 4, 2, 1) if r <= world and world % r == 0]
        for R in dict.fromkeys(shards):
            t0 = time.time()
            aspace, gl = ArrowSpaceBuilder.build_sharded(gp, shard, n, device=local, item_shards=R)
            idx, sc = aspace.search_batch(q, gl, 0.62)                       # host batch
            idx_d, sc_d = aspace.search_batch(q_dev, gl, 0.62)               # device-resident batch
            same_dev = all_ranks(np.array_equal(idx_d.cpu().numpy(), idx) and np.array_equal(sc_d.cpu().numpy(), sc))
            lam = aspace.lambdas()
            lr0 = aspace.row_offset
            if rank == 0:
                e_or = [np.array_equal(gl.edges(), ref["oedges"]), np.array_equal(idx[ref["pick"]], ref["oidx"]),
                        bool(np.allclose(sc[ref["pick"]], ref["osc"], rtol=1e-9, atol=0)),
                        bool(np.allclose(lam, ref["olam"][lr0:lr0 + len(lam)], rtol=1e-9, atol=0))]
                e_1 = [all(np.array_equal(a, b) for a, b in zip(gl.csr(), ref["csr1"])), np.array_equal(idx, ref["idx1"]),
                       np.array_equal(sc, ref["sc1"]), np.array_equal(lam, ref["lam1"][lr0:lr0 + len(lam)])]
                print("world %d n %d f %d grid %d item shard(s) x %d query slot(s): edges/idx/score/lambda vs oracle (%d queries) %s, "
                      "vs single GPU bitwise %s, device batch == host batch on all ranks %s  [%.1f s]"
                      % (world, n, f, R, world // R, len(ref["pick"]), e_or, e_1, same_dev, time.time() - t0), flush=True)
                ok = ok and all(e_or) and all(e_1)
            ok = ok and same_dev
            for pool in HYBRID_POOLS:                         # collective on item shards; every rank returns the whole batch
                hi, hs = aspace.search_hybrid_batch(q, gl, 0.62, pool=pool)
                crc = torch.tensor([zlib.crc32(hi.tobytes() + hs.tobytes())], dtype=torch.int64, device="cuda")
                lo, hi_crc = crc.clone(), crc.clone()
                dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                dist.all_reduce(hi_crc, op=dist.ReduceOp.MAX)
                if rank == 0:
                    i1, s1 = ref["hyb1", pool]
                    oi, os_ = ref["hybo", pool]
                    e = [np.array_equal(hi, i1) and np.array_equal(hs, s1, equal_nan=True),
                         np.array_equal(hi[ref["pick"]], oi) and bool(np.allclose(hs[ref["pick"]], os_, rtol=1e-9, atol=0)),
                         bool(lo.item() == hi_crc.item())]
                    print("world %d n %d f %d grid %d item shard(s) x %d query slot(s): search_hybrid pool %s == single GPU "
                          "(bitwise) %s, == oracle (%d queries) %s, same bits on every rank %s"
                          % (world, n, f, R, world // R, pool, e[0], len(ref["pick"]), e[1], e[2]), flush=True)
                    ok = ok and all(e)
            fmask = filter_mask(n)                            # collective, the same mask on every rank
            checks = [("search", aspace.search_batch(q, gl, 0.62, allowed=fmask), "filt"),
                      ("search_hybrid", aspace.search_hybrid_batch(q, gl, 0.62, allowed=fmask), "fhyb")]
            for name, (fi, fs), key in checks:
                fi, fs = (t.cpu().numpy() if torch.is_tensor(t) else t for t in (fi, fs))
                if rank == 0:
                    i1, s1 = ref[key + "1"]
                    oi, os_ = ref[key + "o"]
                    ok_o = oi >= 0
                    e = [np.array_equal(fi, i1) and np.array_equal(fs, s1, equal_nan=True),
                         np.array_equal(fi[ref["pick"]], oi) and bool(np.allclose(fs[ref["pick"]][ok_o], os_[ok_o], rtol=1e-9, atol=0)),
                         bool(fmask[fi[fi >= 0]].all())]
                    print("world %d n %d f %d grid %d item shard(s) x %d query slot(s): filtered %s == single GPU (bitwise) %s, "
                          "== oracle (%d queries) %s, only allowed items %s" % (world, n, f, R, world // R, name, e[0],
                                                                                len(ref["pick"]), e[1], e[2]), flush=True)
                    ok = ok and all(e)
            thr = torch.tensor([ref["thr"] if rank == 0 else 0.0], dtype=torch.float64, device="cuda")
            dist.broadcast(thr, 0)
            for m_ in (None, fmask):                          # range search, collective: every rank returns the whole batch
                rp, ri, rs = aspace.search_range_batch(q, gl, 0.62, float(thr.item()), allowed=m_)
                crc = torch.tensor([zlib.crc32(rp.tobytes() + ri.tobytes() + rs.tobytes())], dtype=torch.int64, device="cuda")
                lo, hi_crc = crc.clone(), crc.clone()
                dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                dist.all_reduce(hi_crc, op=dist.ReduceOp.MAX)
                if rank == 0:
                    p1, i1, s1 = ref["rng1", m_ is None]
                    e_o = True
                    for j, i in enumerate(ref["pick"]):
                        wi, ws = ref["rngo", m_ is None][j]
                        e_o = e_o and np.array_equal(ri[rp[i]:rp[i + 1]], wi) and bool(np.allclose(rs[rp[i]:rp[i + 1]], ws, rtol=1e-9, atol=0))
                    e = [np.array_equal(rp, p1) and np.array_equal(ri, i1) and np.array_equal(rs, s1), e_o, bool(lo.item() == hi_crc.item())]
                    print("world %d n %d f %d grid %d item shard(s) x %d query slot(s): search_range%s (%.1f hits/query) == single "
                          "GPU (bitwise) %s, == definition (%d queries) %s, same bits on every rank %s"
                          % (world, n, f, R, world // R, "" if m_ is None else " masked", rp[-1] / nq, e[0], len(ref["pick"]),
                             e[1], e[2]), flush=True)
                    ok = ok and all(e)
            if os.environ.get("CHECK_PEER") and R == world and world > 1:    # csrc/peer.cu: P2P exchange + flag-driven merge
                os.environ["ASP_PEER_MERGE"] = "1"
                same = True
                for rep in range(3):                              # three calls: both parities and a reused slot
                    idx_p, sc_p = aspace.search_batch(q, gl, 0.62)
                    same = same and np.array_equal(idx_p, idx) and np.array_equal(sc_p, sc)
                os.environ.pop("ASP_PEER_MERGE")
                same = all_ranks(same)
                if rank == 0:
                    print("world", world, "n", n, "peer-memory merge == NCCL merge on every rank (bitwise):", same, flush=True)
                ok = ok and same
            del aspace, gl
            dist.barrier()
    if os.environ.get("QUICK"):                               # build / search / merge checks only
        ok = all_ranks(ok)
        if rank == 0:
            print("MGPU_CHECK", "OK" if ok else "FAILED")
        dist.destroy_process_group()
        sys.exit(0 if ok else 1)
    # item graph across the ranks: halo all-gather of the item shards, rows resolved per rank on the tensor cores,
    # all-gather of the neighbour lists; every rank must end with the single-GPU graph (bitwise) == the oracle's edges
    for n, f, gp in [(24000, 96, {"eps": 0.3, "k": 12, "topk": 3, "p": 2.0, "sigma": None}),
                     (int(os.environ.get("IG_N", 60000)), 384, {"eps": 10.0, "k": 25, "topk": 3, "p": 2.0, "sigma": None})]:
        per = (n + world - 1) // world
        r0, r1 = min(rank * per, n), min((rank + 1) * per, n)
        full = synth.make_items(n, f, 11, n_clusters=16)
        shard = torch.from_numpy(full[r0:r1].copy()).cuda()
        torch.cuda.synchronize(); dist.barrier(); t0 = time.time()
        aspace, gl = ArrowSpaceBuilder.build_item_graph_sharded(gp, shard, n, r0, device=local)
        torch.cuda.synchronize(); dist.barrier(); dt = time.time() - t0
        os.environ["ASP_KNN_STAGE1"] = "tc"
        torch.cuda.synchronize(); t1 = time.time()
        a1, g1 = ArrowSpaceBuilder.build_item_graph(gp, torch.from_numpy(full).cuda(), device=local)
        torch.cuda.synchronize(); d1 = time.time() - t1
        os.environ.pop("ASP_KNN_STAGE1", None)
        same = all_ranks(all(np.array_equal(a, b) for a, b in zip(gl.csr(), g1.csr())))
        if rank == 0:
            e = [same]
            if n <= 30000:
                import oracle
                s, g = oracle.build(gp, full, nodes="items")
                e.append(np.array_equal(gl.edges(), g.edges()))
            print("world", world, "item graph n", n, "f", f, "sharded %.3f s, single GPU %.3f s" % (dt, d1),
                  "all ranks == single GPU (bitwise):", e[0], "" if len(e) < 2 else "== oracle edges: %s" % e[1], flush=True)
            ok = ok and all(e)
        del aspace, gl, a1, g1
        dist.barrier()
    ok = all_ranks(ok)
    if rank == 0:
        print("MGPU_CHECK", "OK" if ok else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
