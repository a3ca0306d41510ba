// search.cu -- K4 / K4' / K5: batched lambda-aware search
//   score_i = tau * cos(q, x_i) + (1 - tau) / (1 + |lambda_q - lambda_i|)        (TAUMODE.md:33)
// top-`topk` per query by (score desc, index asc)  (replaces ArrowSpace::search_lambda_aware,
// call site /root/reference/src/lib.rs:173; SURVEY.md Appendix A9).
//
// Two stages, so that the answer equals the one computed with left-to-right f64 dot products:
//   stage 1  candidate generation.  Scores with tensor-core dot products (different summation order,
//            |s~ - s| <= DELTA), per query the best LIST candidates:
//              search_gemm_kernel  (nq > 8)   FP64 DMMA 128x128 tiles fed by TMA, fused scoring +
//                                             warp-local threshold/top-LIST epilogue in shared memory.
//                                             Bound: FP64 tensor pipe, 2*nq*n*f FLOP.
//              search_gemv_kernel  (nq <= 8)  the reference's one-query-per-call shape.  Bound: HBM,
//                                             8*n*f bytes per pass.
//   stage 2  rescore_kernel.  The LIST candidates of a query are re-scored in the reference order
//            (sequential dot, the oracle's exact expression), sorted, top-k emitted.  The candidate set is
//            complete iff  s~(LIST) < s~(k) - 2 DELTA  (or the shard has <= LIST items); otherwise the
//            query takes the exact full scan (exact_scan.cuh, SearchScanPolicy).
//   K5       topk_merge_kernel: merge of per-shard results (cross-GPU), (score desc, index asc).
// Filtered search (FILTER instantiations, `allowed` = packed item mask): stage 1 skips a row that is not allowed before it can
// enter a list, so every threshold is the k-th score of k allowed rows and the completeness test above holds over the allowed
// set; the exact scan marks such rows invalid.  Stage 2 needs no change.
#include "gemm_topk.cuh"
#include "exact_scan.cuh"

#include <math.h>
#include <type_traits>

namespace {

using namespace asp_gemm;

// ============================================================================ stage 1: GEMV (nq <= 8)

constexpr int GV_MAXQ = 8;
constexpr int GV_WARPS = 8;

template <int LIST, int FPL, bool FILTER>
__global__ void __launch_bounds__(GV_WARPS * 32)
search_gemv_kernel(const double *__restrict__ q, int qpitch, int nq, const double *__restrict__ items, int64_t n_local,
                   int f, int pitch, const double *__restrict__ inv_nx, const double *__restrict__ lam_x,
                   const double *__restrict__ inv_nq, const double *__restrict__ lam_q, double tau,
                   double *__restrict__ cand_score, int32_t *__restrict__ cand_idx, const uint32_t *__restrict__ allowed)
{
    constexpr int CAP = 2 * LIST;
    constexpr int NPL = CAP / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *qs = reinterpret_cast<double *>(smem_raw);                              // nq * FPL * 32
    double *w_sc = qs + (size_t)GV_MAXQ * FPL * 32;                                 // [warp][q][CAP]
    int32_t *w_ix = reinterpret_cast<int32_t *>(w_sc + GV_WARPS * GV_MAXQ * CAP);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int i = threadIdx.x; i < nq * FPL * 32; i += blockDim.x) {
        const int qi = i / (FPL * 32), ff = i % (FPL * 32);
        qs[i] = (ff < f) ? q[(size_t)qi * qpitch + ff] : 0.0;
    }
    __syncthreads();

    int cnt[GV_MAXQ];
    double theta[GV_MAXQ];
#pragma unroll
    for (int qi = 0; qi < GV_MAXQ; ++qi) { cnt[qi] = 0; theta[qi] = -INFINITY; }
    const double beta = 1.0 - tau;
    double *my_sc = w_sc + (size_t)warp * GV_MAXQ * CAP;
    int32_t *my_ix = w_ix + (size_t)warp * GV_MAXQ * CAP;

    auto compact = [&](int qi) {
        Cand e[NPL];
#pragma unroll
        for (int t = 0; t < NPL; ++t) {
            const int i = lane + 32 * t;
            if (i < cnt[qi]) { e[t].s = my_sc[qi * CAP + i]; e[t].i = my_ix[qi * CAP + i]; }
            else e[t] = asp::cand_empty();
        }
        asp::warp_sort_best_first<NPL>(e, lane);
#pragma unroll
        for (int t = 0; t < NPL; ++t) {
            const int i = lane + 32 * t;
            if (i < LIST) { my_sc[qi * CAP + i] = e[t].s; my_ix[qi * CAP + i] = e[t].i; }
        }
        const double last = __shfl_sync(0xffffffffu, e[(LIST - 1) / 32].s, (LIST - 1) & 31);
        theta[qi] = (cnt[qi] >= LIST) ? last : -INFINITY;
        cnt[qi] = cnt[qi] < LIST ? cnt[qi] : LIST;
        __syncwarp();
    };

    const int64_t gw = (int64_t)blockIdx.x * GV_WARPS + warp, nw = (int64_t)gridDim.x * GV_WARPS;
    for (int64_t item = gw; item < n_local; item += nw) {
        if (FILTER && !asp_allowed(allowed, item)) continue;                         // warp-uniform: one item per warp
        const double *row = items + item * pitch;
        double xv[FPL];
#pragma unroll
        for (int j = 0; j < FPL; ++j) {
            const int ff = lane + 32 * j;
            xv[j] = (ff < f) ? asp::ld_nc_f64(row + ff) : 0.0;
        }
        const double inx = inv_nx[item], lmx = lam_x[item];
#pragma unroll
        for (int qi = 0; qi < GV_MAXQ; ++qi) {
            if (qi < nq) {
                double d = 0.0;
#pragma unroll
                for (int j = 0; j < FPL; ++j) d = fma(xv[j], qs[(qi * FPL + j) * 32 + lane], d);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
                const double cs = tau * inv_nq[qi] * d * inx;
                if (cs + beta > theta[qi]) {
                    const double sc = cs + beta / (1.0 + fabs(lam_q[qi] - lmx));
                    if (sc > theta[qi]) {                       // warp-uniform branch
                        if (lane == 0) { my_sc[qi * CAP + cnt[qi]] = sc; my_ix[qi * CAP + cnt[qi]] = (int32_t)item; }
                        cnt[qi]++;
                        __syncwarp();
                        if (cnt[qi] == CAP) compact(qi);
                    }
                }
            }
        }
    }
    // per-warp lists -> per-block list: warp qi merges query qi's GV_WARPS lists
#pragma unroll
    for (int qi = 0; qi < GV_MAXQ; ++qi)
        if (qi < nq) compact(qi);
    __shared__ int s_cnt[GV_WARPS][GV_MAXQ];
    if (lane == 0)
        for (int qi = 0; qi < GV_MAXQ; ++qi) s_cnt[warp][qi] = cnt[qi];
    __syncthreads();
    for (int qi = warp; qi < nq; qi += GV_WARPS) {
        Cand best[NPL];
#pragma unroll
        for (int t = 0; t < NPL; ++t) best[t] = asp::cand_empty();
        for (int w = 0; w < GV_WARPS; ++w) {
            // slots [LIST, CAP) of the merge buffer <- list of warp w; slots [0, LIST) keep the running best
#pragma unroll
            for (int t = 0; t < NPL; ++t) {
                const int i = lane + 32 * t;
                if (i >= LIST) {
                    const int j = i - LIST;
                    if (j < s_cnt[w][qi]) {
                        best[t].s = w_sc[((size_t)w * GV_MAXQ + qi) * CAP + j];
                        best[t].i = w_ix[((size_t)w * GV_MAXQ + qi) * CAP + j];
                    } else best[t] = asp::cand_empty();
                }
            }
            asp::warp_sort_best_first<NPL>(best, lane);
        }
#pragma unroll
        for (int t = 0; t < NPL; ++t) {
            const int i = lane + 32 * t;
            if (i < LIST) {
                const size_t o = ((size_t)qi * gridDim.x + blockIdx.x) * LIST + i;
                cand_score[o] = best[t].s;
                cand_idx[o] = (best[t].s == -INFINITY && best[t].i == 0x7fffffff) ? -1 : best[t].i;
            }
        }
    }
}

__global__ void reciprocal_kernel(const double *__restrict__ x, int64_t n, double *__restrict__ out)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (x[i] > 0.0) ? 1.0 / x[i] : 0.0;
}

// ============================================================================ stage 2: rescore

// the oracle's score expression (oracle.c orc_scores), no contraction
__device__ __forceinline__ double exact_score(double dot, double nq, double nx, double tau, double lq, double lx)
{
    const double den = __dmul_rn(nq, nx);
    const double c = (den == 0.0) ? 0.0 : __ddiv_rn(dot, den);
    const double prox = __ddiv_rn(1.0, __dadd_rn(1.0, fabs(__dsub_rn(lq, lx))));
    return __dadd_rn(__dmul_rn(tau, c), __dmul_rn(__dsub_rn(1.0, tau), prox));
}

constexpr int RS_WARPS = 4;

template <int LIST>
__global__ void __launch_bounds__(RS_WARPS * 32)
rescore_kernel(const double *__restrict__ q, int qpitch, int64_t nq, const double *__restrict__ items, int64_t n_local,
               int f, int pitch, int64_t row0, const double *__restrict__ norm_x, const double *__restrict__ lam_x,
               const double *__restrict__ norm_q, const double *__restrict__ lam_q, double tau, int topk, int nparts,
               const double *__restrict__ cand_score, const int32_t *__restrict__ cand_idx, double delta,
               int64_t *__restrict__ out_idx, double *__restrict__ out_score, int32_t *slow_list, int32_t *slow_count)
{
    constexpr int CAP = 2 * LIST;
    constexpr int NPL = CAP / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *qs_all = reinterpret_cast<double *>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *qs = qs_all + (size_t)warp * f;
    const int64_t qi = (int64_t)blockIdx.x * RS_WARPS + warp;
    if (qi >= nq) return;

    for (int j = lane; j < f; j += 32) qs[j] = q[qi * qpitch + j];
    __syncwarp();

    // merge the partial lists: running best in slots [0, LIST), incoming in [LIST, CAP)
    Cand best[NPL];
#pragma unroll
    for (int t = 0; t < NPL; ++t) best[t] = asp::cand_empty();
    for (int p = 0; p < nparts; ++p) {
        const size_t base = ((size_t)qi * nparts + p) * LIST;
#pragma unroll
        for (int t = 0; t < NPL; ++t) {
            const int i = lane + 32 * t;
            if (i >= LIST) {
                const int32_t ci = cand_idx[base + i - LIST];
                if (ci >= 0) { best[t].s = cand_score[base + i - LIST]; best[t].i = ci; }
                else best[t] = asp::cand_empty();
            }
        }
        asp::warp_sort_best_first<NPL>(best, lane);
    }
    // element e lives in lane e%32 slot e/32.  Completeness test on the approximate scores.
    const int kk = topk < n_local ? topk : (int)n_local;
    const double a_k = __shfl_sync(0xffffffffu, best[(kk - 1) / 32].s, (kk - 1) & 31);
    const double a_L = __shfl_sync(0xffffffffu, best[(LIST - 1) / 32].s, (LIST - 1) & 31);
    const bool complete = (n_local <= LIST) || (a_L == -INFINITY) || (a_L < a_k - 2.0 * delta);
    if (!complete || kk > LIST) {
        if (lane == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)qi;
        return;
    }
    // exact rescoring of the LIST candidates (one lane each), reference order
    const double nqv = norm_q[qi], lqv = lam_q[qi];
#pragma unroll
    for (int t = 0; t < NPL; ++t) {
        const int i = lane + 32 * t;
        if (i < LIST && best[t].i != 0x7fffffff) {
            const int64_t it = best[t].i;
            const double d = seq_dot_row(qs, items + it * pitch, f);
            best[t].s = exact_score(d, nqv, norm_x[it], tau, lqv, lam_x[it]);
        } else best[t] = asp::cand_empty();
    }
    asp::warp_sort_best_first<NPL>(best, lane);
#pragma unroll
    for (int t = 0; t < NPL; ++t) {
        const int i = lane + 32 * t;
        if (i < topk) {
            const bool ok = (i < kk) && best[t].i != 0x7fffffff;
            out_idx[qi * topk + i] = ok ? row0 + best[t].i : -1;
            out_score[qi * topk + i] = ok ? best[t].s : NAN;
        }
    }
}

// ============================================================================ slow path: exact full scan (exact_scan.cuh)
// value = the reference-order score; every item is admissible (FILTER: the allowed ones)
template <bool FILTER>
struct SearchScanPolicy {
    const double *q; int qpitch; const int32_t *slow_list;
    const double *norm_x, *lam_x, *norm_q, *lam_q; double tau;
    int64_t row0; int topk; int64_t *out_idx; double *out_score; const uint32_t *allowed;
    struct Row { double nq, lq; };
    struct Item { double nx, lx; };
    __device__ const double *query(int slot) const { return q + (int64_t)slow_list[slot] * qpitch; }
    __device__ Row row(int slot) const { const int64_t qi = slow_list[slot]; return Row{norm_q[qi], lam_q[qi]}; }
    __device__ Item item(int64_t it) const { return Item{norm_x[it], lam_x[it]}; }
    __device__ double value(const Row &r, const Item &i, double dot, int64_t it, bool &valid) const
    {
        valid = !FILTER || asp_allowed(allowed, it);
        return exact_score(dot, r.nq, i.nx, tau, r.lq, i.lx);
    }
    __device__ void emit(int slot, int r, bool ok, double v, int64_t it) const
    {
        const int64_t qi = slow_list[slot];
        out_idx[qi * topk + r] = ok ? row0 + it : -1;
        out_score[qi * topk + r] = ok ? v : NAN;
    }
    __device__ void finish(int, int) const {}
};

// ============================================================================ K5: cross-shard merge

struct MKey { double s; int64_t i; };
__device__ __forceinline__ bool mkey_better(const MKey &x, const MKey &y)
{
    return (x.s > y.s) || (x.s == y.s && x.i < y.i);
}

// one block per query; bitonic sort of parts*topk entries in shared memory
__global__ void topk_merge_kernel(const int64_t *__restrict__ idx, const double *__restrict__ score, int parts, int64_t nq,
                                  int topk, int p2, int64_t *__restrict__ out_idx, double *__restrict__ out_score)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    MKey *keys = reinterpret_cast<MKey *>(smem_raw);
    const int64_t qi = blockIdx.x;
    const int total = parts * topk;
    for (int i = threadIdx.x; i < p2; i += blockDim.x) {
        MKey k; k.s = -INFINITY; k.i = INT64_MAX;
        if (i < total) {
            const int p = i / topk, j = i % topk;
            const int64_t id = idx[((size_t)p * nq + qi) * topk + j];
            if (id >= 0) { k.s = score[((size_t)p * nq + qi) * topk + j]; k.i = id; }
        }
        keys[i] = k;
    }
    for (int size = 2; size <= p2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < p2 / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool first = ((lo & size) == 0);
                const MKey a = keys[lo], b = keys[hi];
                if (first ? mkey_better(b, a) : mkey_better(a, b)) { keys[lo] = b; keys[hi] = a; }
            }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < topk; i += blockDim.x) {
        const bool ok = (i < p2) && keys[i].i != INT64_MAX;
        out_idx[qi * topk + i] = ok ? keys[i].i : -1;
        out_score[qi * topk + i] = ok ? keys[i].s : NAN;
    }
}

template <int LIST, bool FILTER>
int launch_gemm(const asp_space *s, const CUtensorMap &tmap_q, const double *q_dev, int64_t nq, const double *inv_nq,
                const double *lam_q, double tau, int nchunks, double *cand_score, int32_t *cand_idx, const uint32_t *allowed)
{
    asp_ctx *ctx = s->ctx;
    constexpr int STAGES = (LIST == 16) ? 4 : 3;
    const size_t smem = (size_t)STAGES * STAGE_DOUBLES_S * 8 + sizeof(ListSmem<LIST>) + 128;
    dim3 grid((unsigned)asp_ceil_div(nq, QT), nchunks);
    if (ctx->use_tma) {
        auto k = search_gemm_kernel<LIST, STAGES, true, 0, FILTER>;
        ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k<<<grid, MMA_WARPS * 32, smem, ctx->stream>>>(tmap_q, s->tmap_rows, q_dev, s->items, nq, s->n_local, s->fp,
                                                           s->inv_norms, s->lambdas, inv_nq, lam_q, tau, 0.0, nchunks, cand_score,
                                                           cand_idx, allowed);
    } else {
        auto k = search_gemm_kernel<LIST, STAGES, false, 0, FILTER>;
        ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k<<<grid, MMA_WARPS * 32, smem, ctx->stream>>>(tmap_q, s->tmap_rows, q_dev, s->items, nq, s->n_local, s->fp,
                                                     s->inv_norms, s->lambdas, inv_nq, lam_q, tau, 0.0, nchunks, cand_score,
                                                     cand_idx, allowed);
    }
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}

template <int LIST, bool FILTER>
int launch_gemv(const asp_space *s, const double *q_dev, int qpitch, int nq, const double *inv_nq, const double *lam_q,
                double tau, int nblocks, double *cand_score, int32_t *cand_idx, const uint32_t *allowed)
{
    asp_ctx *ctx = s->ctx;
    constexpr int CAP = 2 * LIST;
    const int f = s->f;
    int fpl = (f + 31) / 32;
    auto smem_for = [&](int FPL) { return (size_t)GV_MAXQ * FPL * 32 * 8 + (size_t)GV_WARPS * GV_MAXQ * CAP * 12; };
#define ASP_GEMV_CASE(FPLV)                                                                                         \
    {                                                                                                               \
        auto k = search_gemv_kernel<LIST, FPLV, FILTER>;                                                            \
        const size_t smem = smem_for(FPLV);                                                                         \
        ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                  \
        k<<<nblocks, GV_WARPS * 32, smem, ctx->stream>>>(q_dev, qpitch, nq, s->items, s->n_local, f, s->fp,         \
                                                        s->inv_norms, s->lambdas, inv_nq, lam_q, tau, cand_score,   \
                                                        cand_idx, allowed);                                         \
    }
    if (fpl <= 4) ASP_GEMV_CASE(4)
    else if (fpl <= 12) ASP_GEMV_CASE(12)
    else if (fpl <= 24) ASP_GEMV_CASE(24)
    else if (fpl <= 48) ASP_GEMV_CASE(48)
    else ASP_FAIL(ASP_ERR_UNSUPPORTED, "single-query search supports at most 1536 features (got %d)", f);
#undef ASP_GEMV_CASE
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}

}  // namespace

int asp_launch_reciprocal(asp_ctx *ctx, const double *x, int64_t n, double *out)
{
    reciprocal_kernel<<<(unsigned)(asp_ceil_div(n, 256) < 1024 ? asp_ceil_div(n, 256) : 1024), 256, 0, ctx->stream>>>(x, n, out);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}

// exact full scan of the listed queries (completeness test failed / emission buffer full)
int asp_search_slow_path(const asp_space *s, const double *q_dev, int32_t qpitch, const double *lambda_q_dev,
                         const double *qnorm_dev, double tau, int64_t topk, const int32_t *slow_list, int nslow,
                         int64_t *out_idx_dev, double *out_score_dev, const uint32_t *allowed)
{
    asp_ctx *ctx = s->ctx;
    auto scan = [&](auto pol) {
        return asp_xs::run(ctx->stream, ctx->num_sms, pol, nslow, s->items, s->n_local, s->f, s->fp, topk,
                           [&](int k) { ctx->launches += k; });
    };
    const int rc = allowed ? scan(SearchScanPolicy<true>{q_dev, qpitch, slow_list, s->norms, s->lambdas, qnorm_dev, lambda_q_dev,
                                                         tau, s->row0, (int)topk, out_idx_dev, out_score_dev, allowed})
                           : scan(SearchScanPolicy<false>{q_dev, qpitch, slow_list, s->norms, s->lambdas, qnorm_dev, lambda_q_dev,
                                                          tau, s->row0, (int)topk, out_idx_dev, out_score_dev, nullptr});
    if (rc == 1) ASP_FAIL(ASP_ERR_UNSUPPORTED, "exact scan supports topk <= %d (got %lld)", asp_xs::TOPK_MAX, (long long)topk);
    if (rc == 2) ASP_FAIL(ASP_ERR_UNSUPPORTED, "exact scan: %d features x topk %lld do not fit in shared memory", s->f, (long long)topk);
    if (rc == 3) ASP_FAIL(ASP_ERR_NOMEM, "out of device memory in the exact scan");
    if (rc != 0) ASP_FAIL(ASP_ERR_CUDA, "exact scan launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return ASP_OK;
}

int asp_search_impl(const asp_space *s, const asp_graph *g, const double *q_dev, int64_t nq, int32_t qpitch,
                    const double *lambda_q_dev, const double *qnorm_dev, double tau, int64_t topk, int64_t *out_idx_dev,
                    double *out_score_dev, const uint32_t *allowed)
{
    (void)g;
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    if (nq == 0 || topk == 0) return ASP_OK;
    const int f = s->f;
    const int LISTSEL = (topk <= 12) ? 16 : 32;
    // rounding band of one approximate score: dot products of f terms in two orders, both norms,
    // the blend: (4 f + 64) u  scaled by |tau| + |1 - tau|
    const double u = 1.1102230246251565e-16;
    const double delta = (4.0 * f + 64.0) * u * (fabs(tau) + fabs(1.0 - tau) + 1.0);

    // 1/norm of the queries
    asp_scratch sc(st);
    double *inv_nq = nullptr;
    ASP_CHECK(sc.get(&inv_nq, (size_t)nq));
    ASP_CHECK(asp_launch_reciprocal(ctx, qnorm_dev, nq, inv_nq));

    int32_t *slow_list = nullptr, *slow_count = nullptr;
    ASP_CHECK(sc.get(&slow_list, (size_t)nq + 1));
    ASP_CHECK(sc.get(&slow_count, 1));
    ASP_CUDA(cudaMemsetAsync(slow_count, 0, sizeof(int32_t), st));

    int nparts = 0;
    double *cand_score = nullptr;
    int32_t *cand_idx = nullptr;
    ASP_CUDA(cudaEventRecord(ctx->ev0, st));
    if (nq <= GV_MAXQ && f <= 1536) {            // the GEMV kernel keeps a query in registers: wider vectors take the DMMA tile kernel
        int64_t want = asp_ceil_div(s->n_local, GV_WARPS * 16);
        nparts = (int)(want < ctx->num_sms * 2 ? (want > 0 ? want : 1) : ctx->num_sms * 2);
        ASP_CHECK(sc.get(&cand_score, (size_t)nq * nparts * LISTSEL));
        ASP_CHECK(sc.get(&cand_idx, (size_t)nq * nparts * LISTSEL));
        auto gemv = [&](auto list, auto filter) {
            return launch_gemv<decltype(list)::value, decltype(filter)::value>(s, q_dev, qpitch, (int)nq, inv_nq, lambda_q_dev, tau,
                                                                               nparts, cand_score, cand_idx, allowed);
        };
        using L16 = std::integral_constant<int, 16>; using L32 = std::integral_constant<int, 32>;
        using F0 = std::false_type; using F1 = std::true_type;
        ASP_CHECK(LISTSEL == 16 ? (allowed ? gemv(L16(), F1()) : gemv(L16(), F0())) : (allowed ? gemv(L32(), F1()) : gemv(L32(), F0())));
    } else {
        const int64_t tiles_total = asp_ceil_div(s->n_local, IT);
        const int64_t qblocks = asp_ceil_div(nq, QT);
        // CTAs = qblocks x chunks; pick the chunk count whose CTA total fills whole waves of SMs
        // (1 CTA per SM): smallest wave count w with >= 97 % of w * num_sms CTAs, else the best seen.
        int64_t best_chunks = 1;
        double best_eff = 0.0;
        for (int w = 1; w <= 16; ++w) {
            int64_t c = ((int64_t)w * ctx->num_sms) / qblocks;
            if (c < 1) continue;
            if (c > tiles_total) c = tiles_total;
            const int64_t ctas = c * qblocks;
            const double eff = (double)ctas / (double)(asp_ceil_div(ctas, ctx->num_sms) * ctx->num_sms);
            if (eff > best_eff + 1e-9) { best_eff = eff; best_chunks = c; }
            if (eff >= 0.97 || c == tiles_total) break;
        }
        nparts = (int)best_chunks;
        CUtensorMap tmap_q;
        ASP_CHECK(asp_make_items_tmap(&tmap_q, q_dev, nq, qpitch, QT, KSTEP / 4));
        ASP_CHECK(sc.get(&cand_score, (size_t)nq * nparts * LISTSEL));
        ASP_CHECK(sc.get(&cand_idx, (size_t)nq * nparts * LISTSEL));
        auto gemm = [&](auto list, auto filter) {
            return launch_gemm<decltype(list)::value, decltype(filter)::value>(s, tmap_q, q_dev, nq, inv_nq, lambda_q_dev, tau,
                                                                               nparts, cand_score, cand_idx, allowed);
        };
        using L16 = std::integral_constant<int, 16>; using L32 = std::integral_constant<int, 32>;
        using F0 = std::false_type; using F1 = std::true_type;
        ASP_CHECK(LISTSEL == 16 ? (allowed ? gemm(L16(), F1()) : gemm(L16(), F0())) : (allowed ? gemm(L32(), F1()) : gemm(L32(), F0())));
    }
    ASP_CUDA(cudaEventRecord(ctx->ev1, st));

    {
        const size_t smem = (size_t)RS_WARPS * f * 8;
        const unsigned grid = (unsigned)asp_ceil_div(nq, RS_WARPS);
        if (LISTSEL == 16) {
            ASP_CUDA(cudaFuncSetAttribute(rescore_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            rescore_kernel<16><<<grid, RS_WARPS * 32, smem, st>>>(q_dev, qpitch, nq, s->items, s->n_local, f, s->fp, s->row0,
                                                                 s->norms, s->lambdas, qnorm_dev, lambda_q_dev, tau, (int)topk,
                                                                 nparts, cand_score, cand_idx, delta, out_idx_dev,
                                                                 out_score_dev, slow_list, slow_count);
        } else {
            ASP_CUDA(cudaFuncSetAttribute(rescore_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            rescore_kernel<32><<<grid, RS_WARPS * 32, smem, st>>>(q_dev, qpitch, nq, s->items, s->n_local, f, s->fp, s->row0,
                                                                 s->norms, s->lambdas, qnorm_dev, lambda_q_dev, tau, (int)topk,
                                                                 nparts, cand_score, cand_idx, delta, out_idx_dev,
                                                                 out_score_dev, slow_list, slow_count);
        }
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }

    int32_t nslow = 0;
    ASP_CUDA(cudaMemcpyAsync(&nslow, slow_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->stats["search_stage1_ms"] = ms;
    ctx->stats["search_slow_queries"] = nslow;
    ctx->stats["search_stage1_is_tc"] = 0.0;
    if (nslow > 0)
        ASP_CHECK(asp_search_slow_path(s, q_dev, qpitch, lambda_q_dev, qnorm_dev, tau, topk, slow_list, nslow, out_idx_dev,
                                       out_score_dev, allowed));
    return ASP_OK;
}

int asp_topk_merge_impl(asp_ctx *ctx, const int64_t *idx_dev, const double *score_dev, int parts, int64_t nq, int64_t topk,
                        int64_t *out_idx_dev, double *out_score_dev)
{
    if (nq == 0 || topk == 0) return ASP_OK;
    int p2 = 1;
    while (p2 < parts * topk) p2 <<= 1;
    const size_t smem = (size_t)p2 * sizeof(MKey);
    if (smem > 200 * 1024) ASP_FAIL(ASP_ERR_UNSUPPORTED, "topk merge of %d x %lld entries does not fit in shared memory", parts, (long long)topk);
    ASP_CUDA(cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topk_merge_kernel<<<(unsigned)nq, 128, smem, ctx->stream>>>(idx_dev, score_dev, parts, nq, (int)topk, p2, out_idx_dev,
                                                                out_score_dev);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}
