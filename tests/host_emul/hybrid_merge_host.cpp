// CPU walk of the cross-shard merge of pyarrowspace_b200/csrc/hybrid.cuh (test infrastructure: tests/test_hybrid_sharded_cpu.py):
// the -1 fill of the merged shortlist, hybrid_merge_kernel and hybrid_select_kernel, as asp_hybrid_merge runs them, every
// thread index walked in an order that differs from the GPU's only where threads are independent.
// Build: g++ -O2 -ffp-contract=off -shared -fPIC.
#include <string.h>

#include "../../pyarrowspace_b200/csrc/hybrid.cuh"

extern "C" void hyb_merge_emulate(int parts, int64_t nq, int64_t m, int64_t topk, const int64_t *idx, const double *cosv,
                                  const double *score, int64_t *pool_idx, double *pool_score, int64_t *out_idx,
                                  double *out_score)
{
    memset(pool_idx, 0xff, sizeof(int64_t) * (size_t)(nq * m));
    const int64_t total = parts * nq * m;
    const int64_t threads_m = 5 * 256;                       // hybrid_merge_kernel: grid-stride, a grid smaller than the work
    for (int64_t tid = threads_m - 1; tid >= 0; --tid)
        for (int64_t t = tid; t < total; t += threads_m)
            asp_hybrid::merge_slot(t, parts, nq, m, idx, cosv, score, pool_idx, pool_score);
    const int64_t threads_s = 2 * 128;                       // hybrid_select_kernel
    for (int64_t tid = threads_s - 1; tid >= 0; --tid)
        for (int64_t qi = tid; qi < nq; qi += threads_s)
            asp_hybrid::select_query(qi, m, topk, pool_idx, pool_score, out_idx, out_score);
}
