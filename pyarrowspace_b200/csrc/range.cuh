// range.cuh -- the parts of the range search (asp_search_range_batch, csrc/range.cu) that tests walk on the CPU.
//
// A range search returns, per query, EVERY item whose reference-order score is >= min_score, ordered by (score desc, index
// asc).  Its per-query lists have different lengths, so results are CSR pieces: counts per query, then the hits query-major.
// Row-sharded spaces answer per shard and merge with asp_range_merge:
//   range_merge_kernel  one thread per hit of the concatenated per-shard pieces: the hit's position in the one-GPU list is
//                       the query's output offset + its position in its own (sorted) segment + the number of hits of each
//                       other shard's segment of the same query that come before it (binary search by (score desc, index
//                       asc)).  Shards hold disjoint, contiguous global row ranges, so no two hits compare equal and the
//                       positions are a permutation: the result does not depend on the number of shards or their order.
//
// The per-thread body and the host-side offset tables are plain functions so that tests/test_range_search_cpu.py can compile
// this header with g++ (-ffp-contract=off) and walk the thread grid on the CPU.
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define ASP_RNG_FN __host__ __device__ __forceinline__
#else
#define ASP_RNG_FN static inline
#endif

namespace asp_range {

// (s, i) comes strictly before (os, oi) in the order (score desc, index asc)
ASP_RNG_FN bool before(double s, int64_t i, double os, int64_t oi) { return (s > os) || (s == os && i < oi); }

// Order-preserving 64-bit key of a score for the sort: key(a) < key(b) iff a > b.  -0.0 is mapped to +0.0 first so that the
// two zeros tie (and then order by index) as they do under the double comparison.
ASP_RNG_FN uint64_t desc_key(double s)
{
    if (s == 0.0) s = 0.0;
    uint64_t u;
#if defined(__CUDA_ARCH__)
    u = (uint64_t)__double_as_longlong(s);
#else
    memcpy(&u, &s, sizeof(u));
#endif
    const uint64_t asc = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    return ~asc;
}

ASP_RNG_FN double key_score(uint64_t k)
{
    const uint64_t asc = ~k;
    const uint64_t u = (asc >> 63) ? (asc & 0x7fffffffffffffffull) : ~asc;
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double s;
    memcpy(&s, &u, sizeof(s));
    return s;
#endif
}

// Host: offset tables of a merge.  counts [parts][nq] (each part query-major).  part_off [parts][nq + 1]: absolute start of
// (part, query) in the concatenated parts; out_off [nq + 1]: start of query q in the merged result.  Returns the total.
static inline int64_t merge_tables(int parts, int64_t nq, const int64_t *counts, int64_t *part_off, int64_t *out_off)
{
    int64_t base = 0;
    for (int p = 0; p < parts; ++p)
        for (int64_t q = 0; q <= nq; ++q) {
            part_off[(int64_t)p * (nq + 1) + q] = base;
            if (q < nq) base += counts[(int64_t)p * nq + q];
        }
    int64_t o = 0;
    for (int64_t q = 0; q <= nq; ++q) {
        out_off[q] = o;
        if (q < nq)
            for (int p = 0; p < parts; ++p) o += counts[(int64_t)p * nq + q];
    }
    return base;
}

// Hit t of the concatenated parts (t < total) to its place in the merged result.
ASP_RNG_FN void merge_elem(int64_t t, int parts, int64_t nq, const int64_t *part_off, const int64_t *out_off,
                           const int64_t *idx, const double *score, int64_t *out_idx, double *out_score)
{
    int p = 0;
    while (p + 1 < parts && t >= part_off[(int64_t)(p + 1) * (nq + 1)]) ++p;   // the part holding t (parts <= 8 in practice)
    const int64_t *po = part_off + (int64_t)p * (nq + 1);
    int64_t lo = 0, hi = nq;                                                   // the query: po[q] <= t < po[q + 1]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (po[mid] <= t) lo = mid; else hi = mid;
    }
    const int64_t q = lo;
    const double s = score[t];
    const int64_t id = idx[t];
    int64_t pos = out_off[q] + (t - po[q]);
    for (int o = 0; o < parts; ++o) {
        if (o == p) continue;
        const int64_t b0 = part_off[(int64_t)o * (nq + 1) + q], b1 = part_off[(int64_t)o * (nq + 1) + q + 1];
        int64_t a = b0, b = b1;                                                // hits of part o before (s, id): a prefix
        while (a < b) {
            const int64_t mid = (a + b) >> 1;
            if (before(score[mid], idx[mid], s, id)) a = mid + 1; else b = mid;
        }
        pos += a - b0;
    }
    out_idx[pos] = id;
    out_score[pos] = s;
}

#if defined(__CUDACC__) && !defined(ASP_RANGE_KEYS_ONLY)          // (large_k.cuh takes the keys only: one kernel definition)
__global__ void __launch_bounds__(256)
range_merge_kernel(int64_t total, int parts, int64_t nq, const int64_t *__restrict__ part_off, const int64_t *__restrict__ out_off,
                   const int64_t *__restrict__ idx, const double *__restrict__ score, int64_t *__restrict__ out_idx,
                   double *__restrict__ out_score)
{
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
        merge_elem(t, parts, nq, part_off, out_off, idx, score, out_idx, out_score);
}
#endif

}  // namespace asp_range
