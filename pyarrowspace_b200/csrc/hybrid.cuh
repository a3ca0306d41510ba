// hybrid.cuh -- re-ranking of a cosine shortlist: the second half of asp_search_hybrid_batch (SURVEY.md 8(f)-2).
//
// Replaces the crate's search_lambda_aware_hybrid as called by ArrowSpace.search_hybrid (src/lib.rs:182-219).  Its body is
// not in the reference (PARITY UNPINNED); the restatement H1-H3 is in include/arrowspace_b200.h and oracle/oracle.c.  The
// shortlist itself (H2) is the validated search at tau = 1 with topk = pool (search_tc.cu / search.cu); this file holds H3:
//   hybrid_rescore_kernel  one thread per (query, shortlist slot): the cosine re-evaluated in the oracle's order (left to
//                          right, product rounded then added) and the lambda-aware score in the oracle's expression, so the
//                          scores are the oracle's bit for bit;
//   hybrid_select_kernel   one thread per query: the best topk slots by (score desc, index asc).
// Both are a few hundred steps per query next to a scan of every item for the shortlist; no shared memory, no barriers.
//
// Row-sharded spaces (asp_search_hybrid_shard + asp_hybrid_merge) add one step between the two:
//   hybrid_merge_kernel    one thread per (shard, query, slot) of the per-shard shortlists: the slot's rank among the union
//                          of the query's shortlists by (cosine desc, index asc), by binary search in each other list.  The
//                          global top-m by cosine is contained in that union (each shard holds its own top-m), so a slot of
//                          rank < m is one of the m entries the one-GPU shortlist holds, and it is written to position
//                          `rank` of that shortlist.  hybrid_select_kernel then picks from it exactly as on one GPU.
//
// The per-thread bodies are plain functions so that tests/test_hybrid_host.py and tests/test_hybrid_sharded_cpu.py can
// compile this header with g++ (-ffp-contract=off) and walk the thread grid on the CPU against the oracle.
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define ASP_HYB_FN __host__ __device__ __forceinline__
#else
#define ASP_HYB_FN static inline
#endif

namespace asp_hybrid {

ASP_HYB_FN double mul_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
ASP_HYB_FN double add_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
ASP_HYB_FN double sub_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
ASP_HYB_FN double div_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

// H3 for shortlist slot t = qi * pool + j.  pool_idx holds GLOBAL row indices (-1 = padding: fewer items than slots).
// Scores of padding slots are NaN and never selected.
ASP_HYB_FN void rescore_slot(int64_t t, int64_t pool, const double *q, int qpitch, const double *items, int pitch, int f,
                             int64_t row0, const double *norm_x, const double *lam_x, const double *norm_q,
                             const double *lam_q, double tau, const int64_t *pool_idx, double *pool_score)
{
    const int64_t qi = t / pool;
    const int64_t id = pool_idx[t];
    if (id < 0) { pool_score[t] = NAN; return; }
    const int64_t li = id - row0;
    const double *qv = q + (size_t)qi * qpitch;
    const double *xv = items + (size_t)li * pitch;
    double dot = 0.0;
    for (int c = 0; c < f; ++c) dot = add_rn(dot, mul_rn(qv[c], xv[c]));          // oracle.c seq_dot
    const double den = mul_rn(norm_q[qi], norm_x[li]);
    const double cs = (den == 0.0) ? 0.0 : div_rn(dot, den);                        // README.md:69 arithmetic
    const double prox = div_rn(1.0, add_rn(1.0, fabs(sub_rn(lam_q[qi], lam_x[li]))));
    pool_score[t] = add_rn(mul_rn(tau, cs), mul_rn(sub_rn(1.0, tau), prox));       // TAUMODE.md:33
}

// The best topk of query qi's shortlist by (score desc, index asc); pool_idx is scratch (taken slots are overwritten with -1).
// Output rows are padded with -1 / NaN like asp_search_batch.
ASP_HYB_FN void select_query(int64_t qi, int64_t pool, int64_t topk, int64_t *pool_idx, const double *pool_score,
                             int64_t *out_idx, double *out_score)
{
    int64_t *ids = pool_idx + (size_t)qi * pool;
    const double *sc = pool_score + (size_t)qi * pool;
    for (int64_t r = 0; r < topk; ++r) {
        int64_t best = -1;
        for (int64_t j = 0; j < pool; ++j) {
            if (ids[j] < 0) continue;
            if (best < 0 || sc[j] > sc[best] || (sc[j] == sc[best] && ids[j] < ids[best])) best = j;
        }
        if (best < 0) {
            out_idx[qi * topk + r] = -1;
            out_score[qi * topk + r] = NAN;
        } else {
            out_idx[qi * topk + r] = ids[best];
            out_score[qi * topk + r] = sc[best];
            ids[best] = -1;
        }
    }
}

// Slot t = (r * nq + qi) * m + p of `parts` per-shard shortlists ([parts][nq][m]: GLOBAL indices, their cosines and H3
// scores, each list sorted by (cosine desc, index asc) and padded with -1).  A slot whose rank in the union of the query's
// lists is below m goes to position `rank` of the query's merged shortlist pool_idx / pool_score ([nq][m], filled with -1
// beforehand).  Ranks are distinct because the shards hold disjoint rows, so every position is written at most once.
ASP_HYB_FN void merge_slot(int64_t t, int parts, int64_t nq, int64_t m, const int64_t *idx, const double *cosv,
                           const double *score, int64_t *pool_idx, double *pool_score)
{
    const int64_t id = idx[t];
    if (id < 0) return;
    const int64_t per = nq * m;
    const int r = (int)(t / per);
    const int64_t qi = (t - r * per) / m;
    const double c = cosv[t];
    int64_t rank = t - r * per - qi * m;                       // the entries before it in its own list
    for (int o = 0; o < parts && rank < m; ++o) {
        if (o == r) continue;
        const int64_t *oi = idx + o * per + qi * m;
        const double *oc = cosv + o * per + qi * m;
        int64_t lo = 0, hi = m;                                // entries of list o before (c, id): a prefix of the list
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (oi[mid] >= 0 && (oc[mid] > c || (oc[mid] == c && oi[mid] < id))) lo = mid + 1;
            else hi = mid;
        }
        rank += lo;
    }
    if (rank < m) {
        pool_idx[qi * m + rank] = id;
        pool_score[qi * m + rank] = score[t];
    }
}

#if defined(__CUDACC__)
__global__ void __launch_bounds__(256)
hybrid_merge_kernel(int64_t total, int parts, int64_t nq, int64_t m, const int64_t *__restrict__ idx,
                    const double *__restrict__ cosv, const double *__restrict__ score, int64_t *__restrict__ pool_idx,
                    double *__restrict__ pool_score)
{
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
        merge_slot(t, parts, nq, m, idx, cosv, score, pool_idx, pool_score);
}

__global__ void __launch_bounds__(256)
hybrid_rescore_kernel(int64_t total, int64_t pool, const double *__restrict__ q, int qpitch, const double *__restrict__ items,
                      int pitch, int f, int64_t row0, const double *__restrict__ norm_x, const double *__restrict__ lam_x,
                      const double *__restrict__ norm_q, const double *__restrict__ lam_q, double tau,
                      const int64_t *__restrict__ pool_idx, double *__restrict__ pool_score)
{
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
        rescore_slot(t, pool, q, qpitch, items, pitch, f, row0, norm_x, lam_x, norm_q, lam_q, tau, pool_idx, pool_score);
}

__global__ void __launch_bounds__(128)
hybrid_select_kernel(int64_t nq, int64_t pool, int64_t topk, int64_t *pool_idx, const double *__restrict__ pool_score,
                     int64_t *__restrict__ out_idx, double *__restrict__ out_score)
{
    for (int64_t qi = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; qi < nq; qi += (int64_t)gridDim.x * blockDim.x)
        select_query(qi, pool, topk, pool_idx, pool_score, out_idx, out_score);
}
#endif

}  // namespace asp_hybrid
