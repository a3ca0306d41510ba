// graph_select.cu -- K1 epilogue for the feature graph: rectified-cosine distances from the Gram,
// eps-radius filter, k smallest neighbours by (distance, index)
// (GRAPH_VARIABLES.md:7-8; SURVEY.md Appendix A3-A4; crate call site /root/reference/src/lib.rs:289).
//
// Exactness contract.  The oracle decides on left-to-right f64 sums; the Gram here comes from DMMA
// chains in a different order.  Every approximate distance carries the rounding band DELTA
// (|d~ - d_oracle| <= DELTA, see asp_feature_select).  Decisions outside the band are safe; the
// pairs inside it are reported ("need exact"), recomputed in the oracle's own order by
// exact_pairs_kernel and fed back, so the selected edge set equals the oracle's:
//   * eps test:   |d~ - eps| <= DELTA                      -> need the pair
//   * k-th test:  T = k-th smallest d~ of the candidates; if the (k+1)-th lies within T + 2 DELTA,
//                 every candidate with |d~ - T| <= 2 DELTA is needed.  Elements below the band are
//                 in the true top-k, elements above are not, and sorting the band members by their
//                 exact values fills the remaining slots (proof in DESIGN.md).
// The band is always derived from the approximate values only, so the request set is the same
// on every pass and the host loop terminates after at most three passes.
//
// Distance variants (asp_switches.distance, an UNPINNED choice of SURVEY.md 8(c)): besides the documented rectified cosine
// (GRAPH_VARIABLES.md:7) the Gram-form Euclidean distance d^2 = <a,a> + <b,b> - 2<a,b> (clamped at 0) and its square
// root.  Their rounding band is per pair, 2 rel (<a,a> + <b,b>) on d^2 (and d~ - sqrt(d~^2 - band) on d); the
// row uses the largest band of its pairs, which keeps the uniform-band argument above valid.
#include "common.cuh"

#include <math.h>

namespace {

struct Key { double d; int idx; };

__device__ __forceinline__ bool key_less(const Key &x, const Key &y)
{
    return (x.d < y.d) || (x.d == y.d && x.idx < y.idx);
}

__device__ void block_bitonic_sort(Key *keys, int p2)
{
    for (int size = 2; size <= p2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < p2 / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1));
                const int hi = lo + stride;
                const bool asc = ((lo & size) == 0);
                Key a = keys[lo], b = keys[hi];
                const bool swap = asc ? key_less(b, a) : key_less(a, b);
                if (swap) { keys[lo] = b; keys[hi] = a; }
            }
        }
    }
    __syncthreads();
}

// exact d from left-to-right sums, the oracle's own expression (oracle.c node_distance)
__device__ __forceinline__ double exact_distance(double sab, double saa, double sbb, int distance)
{
    if (distance != ASP_DISTANCE_COSINE) {
        double d2 = __dsub_rn(__dadd_rn(saa, sbb), __dmul_rn(2.0, sab));
        if (!(d2 > 0.0)) d2 = 0.0;
        return distance == ASP_DISTANCE_L2 ? __dsqrt_rn(d2) : d2;
    }
    const double na = __dsqrt_rn(saa), nb = __dsqrt_rn(sbb);
    double c = 0.0;
    if (na != 0.0 && nb != 0.0) c = __ddiv_rn(sab, __dmul_rn(na, nb));
    return __dsub_rn(1.0, c > 0.0 ? c : 0.0);
}

// approximate distance of the pair from the (DMMA) Gram + the band that contains the oracle's value
__device__ __forceinline__ double approx_distance(double gab, double gaa, double gbb, int distance, double rel, double *band,
                                                  bool *surely_one)
{
    *surely_one = false;
    if (distance != ASP_DISTANCE_COSINE) {
        double d2 = (gaa + gbb) - 2.0 * gab;
        if (!(d2 > 0.0)) d2 = 0.0;
        const double b2 = rel * 2.0 * (gaa + gbb) + 1e-300;       // 2 sum|x_a x_b| <= <a,a> + <b,b>
        if (distance == ASP_DISTANCE_L2SQ) { *band = b2; return d2; }
        const double d = sqrt(d2), lo2 = d2 - b2;
        *band = (d - (lo2 > 0.0 ? sqrt(lo2) : 0.0)) * (1.0 + 1e-12) + 8.0 * 1.1102230246251565e-16 * d + 1e-300;
        return d;
    }
    *band = rel;
    const double na = sqrt(gaa), nb = sqrt(gbb);
    if (na == 0.0 || nb == 0.0) { *surely_one = true; return 1.0; }
    const double c = gab / (na * nb);
    if (c < -rel) *surely_one = true;                                   // surely rectified: d == 1 exactly
    return 1.0 - (c > 0.0 ? c : 0.0);
}

__device__ int find_exact(const int32_t *pairs, int64_t n, int a, int b)
{
    if (a > b) { const int t = a; a = b; b = t; }
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int pa = pairs[2 * mid], pb = pairs[2 * mid + 1];
        if (pa < a || (pa == a && pb < b)) lo = mid + 1; else hi = mid;
    }
    if (lo < n && pairs[2 * lo] == a && pairs[2 * lo + 1] == b) return (int)lo;
    return -1;
}

__device__ void emit_need(int a, int b, int32_t *need_pairs, int64_t need_cap, int32_t *need_count)
{
    if (a > b) { const int t = a; a = b; b = t; }
    const int slot = atomicAdd(need_count, 1);
    if (slot < need_cap) { need_pairs[2 * slot] = a; need_pairs[2 * slot + 1] = b; }
}

// One block per node a.  smem: Key keys[p2]; double vexact[f] (NaN = none)
__global__ void feature_select_kernel(const double *__restrict__ gram, int f, double eps, int kk, double rel, int distance,
                                      const int32_t *__restrict__ exact_pairs, const double *__restrict__ exact_sums,
                                      int64_t n_exact, int p2, int32_t *__restrict__ out_idx,
                                      double *__restrict__ out_dist, int32_t *__restrict__ out_cnt,
                                      int32_t *need_pairs, int64_t need_cap, int32_t *need_count)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Key *keys = reinterpret_cast<Key *>(smem_raw);
    double *vexact = reinterpret_cast<double *>(keys + p2);
    __shared__ int s_incomplete, s_cnt, s_band;
    __shared__ double s_T;
    __shared__ unsigned long long s_delta;

    const int a = blockIdx.x;
    if (threadIdx.x == 0) { s_incomplete = 0; s_cnt = 0; s_band = 0; s_delta = 0ull; }
    __syncthreads();

    const double gaa = gram[(size_t)a * f + a];

    // ---- A0: the row's band = the largest band of its pairs (non-negative doubles order like their bit patterns)
    double delta = rel;
    if (distance != ASP_DISTANCE_COSINE) {
        double mx = 0.0;
        for (int b = threadIdx.x; b < f; b += blockDim.x) {
            if (b == a) continue;
            double band; bool one;
            approx_distance(gram[(size_t)a * f + b], gaa, gram[(size_t)b * f + b], distance, rel, &band, &one);
            mx = fmax(mx, band);
        }
        atomicMax(&s_delta, (unsigned long long)__double_as_longlong(mx));
        __syncthreads();
        delta = __longlong_as_double((long long)s_delta);
    }

    // ---- A: approximate distance, exact value if known, eps status
    for (int b = threadIdx.x; b < p2; b += blockDim.x) {
        Key k; k.d = INFINITY; k.idx = 0x7fffffff;
        if (b < f) vexact[b] = NAN;
        if (b < f && b != a) {
            double band;
            bool known = false;          // exact value known without a resolve pass
            const double dap = approx_distance(gram[(size_t)a * f + b], gaa, gram[(size_t)b * f + b], distance, rel, &band, &known);
            double dex = known ? 1.0 : NAN;
            if (!known && n_exact > 0) {
                const int e = find_exact(exact_pairs, n_exact, a, b);
                if (e >= 0) { known = true; dex = exact_distance(exact_sums[3 * e], exact_sums[3 * e + 1], exact_sums[3 * e + 2], distance); }
            }
            bool in;
            if (known) in = (dex <= eps);
            else if (fabs(dap - eps) <= delta) { in = false; emit_need(a, b, need_pairs, need_cap, need_count); s_incomplete = 1; }
            else in = (dap < eps);
            if (in) { k.d = dap; k.idx = b; vexact[b] = known ? dex : NAN; atomicAdd(&s_cnt, 1); }
        }
        keys[b] = k;
    }
    __syncthreads();
    if (s_incomplete) { if (threadIdx.x == 0) out_cnt[a] = -1; return; }
    const int cnt = s_cnt;
    const int keep = cnt < kk ? cnt : kk;
    if (keep == 0) { if (threadIdx.x == 0) out_cnt[a] = 0; return; }

    // ---- C: order by the approximate values, locate the band around the k-th
    block_bitonic_sort(keys, p2);
    if (cnt > kk) {
        if (threadIdx.x == 0) {
            s_T = keys[kk - 1].d;
            s_band = (keys[kk].d <= keys[kk - 1].d + 2.0 * delta) ? 1 : 0;
        }
        __syncthreads();
        if (s_band) {
            const double T = s_T;
            for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
                const Key k = keys[i];
                if (fabs(k.d - T) <= 2.0 * delta && isnan(vexact[k.idx])) {
                    emit_need(a, k.idx, need_pairs, need_cap, need_count);
                    s_incomplete = 1;
                }
            }
            __syncthreads();
            if (s_incomplete) { if (threadIdx.x == 0) out_cnt[a] = -1; return; }
            // ---- D: every band member is exact now: re-sort on the mixed values
            for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
                const double ve = vexact[keys[i].idx];
                if (!isnan(ve)) keys[i].d = ve;
            }
            block_bitonic_sort(keys, p2);
        }
    }
    for (int i = threadIdx.x; i < keep; i += blockDim.x) {
        const Key k = keys[i];
        const double ve = vexact[k.idx];
        out_idx[(size_t)a * kk + i] = k.idx;
        out_dist[(size_t)a * kk + i] = isnan(ve) ? k.d : ve;
    }
    if (threadIdx.x == 0) out_cnt[a] = keep;
}

// Left-to-right continuation of <a,b>, <a,a>, <b,b> over the shard rows: product rounded, then added
// (the oracle's order, oracle.c dots_block_full / orc_graph_from_nodes_t).  One thread per pair.
__global__ void exact_pairs_kernel(const double *__restrict__ items, int64_t n_local, int pitch,
                                   const int32_t *__restrict__ pairs, int64_t n_pairs, double *__restrict__ sums)
{
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const int a = pairs[2 * p], b = pairs[2 * p + 1];
    double sab = sums[3 * p], saa = sums[3 * p + 1], sbb = sums[3 * p + 2];
    const double *pa = items + a, *pb = items + b;
    int64_t r = 0;
    for (; r + 8 <= n_local; r += 8) {
        double xa[8], xb[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { xa[u] = pa[(r + u) * pitch]; xb[u] = pb[(r + u) * pitch]; }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            sab = __dadd_rn(sab, __dmul_rn(xa[u], xb[u]));
            saa = __dadd_rn(saa, __dmul_rn(xa[u], xa[u]));
            sbb = __dadd_rn(sbb, __dmul_rn(xb[u], xb[u]));
        }
    }
    for (; r < n_local; ++r) {
        const double xa = pa[r * pitch], xb = pb[r * pitch];
        sab = __dadd_rn(sab, __dmul_rn(xa, xb));
        saa = __dadd_rn(saa, __dmul_rn(xa, xa));
        sbb = __dadd_rn(sbb, __dmul_rn(xb, xb));
    }
    sums[3 * p] = sab; sums[3 * p + 1] = saa; sums[3 * p + 2] = sbb;
}

}  // namespace

int asp_feature_select(asp_ctx *ctx, const double *gram_dev, int32_t f, int64_t n_total, const asp_graph_params *gp,
                       const asp_switches *sw, const int32_t *exact_pairs_dev, const double *exact_sums_dev, int64_t n_exact,
                       asp_knn_lists *lists, int32_t *need_pairs_dev, int64_t need_cap, int32_t *need_count_dev)
{
    if (f > 8192) ASP_FAIL(ASP_ERR_UNSUPPORTED, "feature graph supports at most 8192 features (got %d)", f);
    const int64_t kk = asp_neighbour_cap(gp, sw, f);
    ASP_CHECK(lists->alloc(ctx->stream, f, (int32_t)(kk > 0 ? kk : 1)));
    if (kk == 0) {
        ASP_CUDA(cudaMemsetAsync(lists->cnt, 0, sizeof(int32_t) * (size_t)f, ctx->stream));
        return ASP_OK;
    }
    // Rounding band of a cosine computed from two different summation orders of n_total terms
    // (both within gamma_n of the real value, numerator and both norms): 4*gamma_n + O(u), doubled.
    const double u = 1.1102230246251565e-16;
    const double delta = (8.0 * (double)n_total + 128.0) * u;
    int p2 = 1;
    while (p2 < f) p2 <<= 1;
    const size_t smem = (size_t)p2 * sizeof(Key) + (size_t)f * sizeof(double);
    ASP_CUDA(cudaFuncSetAttribute(feature_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    feature_select_kernel<<<f, 256, smem, ctx->stream>>>(gram_dev, f, gp->eps, (int)kk, delta, sw ? sw->distance : 0, exact_pairs_dev,
                                                         exact_sums_dev, n_exact, p2, lists->idx, lists->dist,
                                                         lists->cnt, need_pairs_dev, need_cap, need_count_dev);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}

int asp_launch_exact_pairs(asp_space *s, const int32_t *pairs_dev, int64_t n_pairs, double *sums_dev)
{
    if (n_pairs == 0) return ASP_OK;
    exact_pairs_kernel<<<(unsigned)asp_ceil_div(n_pairs, 64), 64, 0, s->ctx->stream>>>(s->items, s->n_local, s->fp,
                                                                                         pairs_dev, n_pairs, sums_dev);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(s->ctx);
    return ASP_OK;
}
