// knn.cu -- K1, item orientation (nodes = items): eps-radius / k-NN lists on the rectified-cosine distance (default) or the
// Euclidean one (l2 / l2sq, the Gram form of oracle.c node_distance) for every item against every item (GRAPH_VARIABLES.md:7-8; SURVEY.md Appendix A2 `nodes = items`,
// A3-A4; the graph-build workload of BASELINE.json configs C4/C5).
//
// Bound: FP64 tensor pipe, 2*M^2*D FLOP (every ordered pair, as the reference's per-row scan does).
//
// Same two-stage contract as the search:
//   stage 1  search_gemm_kernel<MODE 1>: DMMA 128x128 tiles of X X^T fed by TMA, epilogue keeps per row the
//            LIST best rectified cosines >= 1 - eps - band (self excluded) in shared memory.
//   stage 2  knn_rescore_kernel: the candidates' distances are recomputed in the oracle's order
//            (left-to-right dot, d = 1 - max(0, dot/(|a||b|))), d <= eps is decided on those values, the k
//            smallest by (d, index) are kept.  Complete iff s~(LIST) < s~(k) - 2 band; otherwise the row takes
//            the exact scan (exact_scan.cuh, KnnScanPolicy).
// Output: neighbour lists for csr.cu (K2).
#include "gemm_topk.cuh"
#include "exact_scan.cuh"

namespace {

using namespace asp_gemm;
using asp::Cand;

// left-to-right norms (the oracle's: sqrt of the sequential sum of squares), one thread per row; nsq (if given) keeps the
// sum of squares itself, which the Euclidean distance uses (it is not norm^2: the two differ in the last bits)
__global__ void row_norms_kernel(const double *__restrict__ items, int64_t n, int f, int pitch, double *__restrict__ norms,
                                 double *__restrict__ inv_norms, double *__restrict__ nsq)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double *row = items + i * pitch;
        const double n2 = seq_dot_row(row, row, f);
        const double nr = sqrt(n2);
        norms[i] = nr;
        inv_norms[i] = nr > 0.0 ? 1.0 / nr : 0.0;
        if (nsq) nsq[i] = n2;
    }
}

__global__ void iota_rows_kernel(int32_t *__restrict__ p, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = (int32_t)i;
}

// the oracle's distance expression (oracle.c select_neighbours)
__device__ __forceinline__ double exact_dist(double dot, double na, double nb)
{
    double c = 0.0;
    if (na != 0.0 && nb != 0.0) c = __ddiv_rn(dot, __dmul_rn(na, nb));
    return __dsub_rn(1.0, c > 0.0 ? c : 0.0);
}

// oracle.c node_distance for every distance kind: cosine as above; l2 / l2sq from the left-to-right sums
// saa = <a,a>, sbb = <b,b>, dot = <a,b>:  d2 = (saa + sbb) - 2 dot clamped at 0, and its square root for l2
__device__ __forceinline__ double exact_node_dist(int distance, double dot, double na, double nb, double saa, double sbb)
{
    if (distance == ASP_DISTANCE_COSINE) return exact_dist(dot, na, nb);
    double d2 = __dsub_rn(__dadd_rn(saa, sbb), __dmul_rn(2.0, dot));
    if (!(d2 > 0.0)) d2 = 0.0;
    return distance == ASP_DISTANCE_L2 ? __dsqrt_rn(d2) : d2;
}

constexpr int KR_WARPS = 4;

template <int LIST>
__global__ void __launch_bounds__(KR_WARPS * 32)
knn_rescore_kernel(const double *__restrict__ items, int64_t n, int f, int pitch, const double *__restrict__ norms,
                   double eps, int kk, int nparts, const double *__restrict__ cand_score,
                   const int32_t *__restrict__ cand_idx, double delta, int32_t *__restrict__ out_idx,
                   double *__restrict__ out_dist, int32_t *__restrict__ out_cnt, int32_t *slow_list, int32_t *slow_count)
{
    constexpr int CAP = 2 * LIST;
    constexpr int NPL = CAP / 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *xs_all = reinterpret_cast<double *>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *xs = xs_all + (size_t)warp * f;
    const int64_t i = (int64_t)blockIdx.x * KR_WARPS + warp;
    if (i >= n) return;
    for (int j = lane; j < f; j += 32) xs[j] = items[i * pitch + j];
    __syncwarp();

    Cand best[NPL];
#pragma unroll
    for (int t = 0; t < NPL; ++t) best[t] = asp::cand_empty();
    for (int p = 0; p < nparts; ++p) {
        const size_t base = ((size_t)i * nparts + p) * LIST;
#pragma unroll
        for (int t = 0; t < NPL; ++t) {
            const int e = lane + 32 * t;
            if (e >= LIST) {
                const int32_t ci = cand_idx[base + e - LIST];
                if (ci >= 0) { best[t].s = cand_score[base + e - LIST]; best[t].i = ci; }
                else best[t] = asp::cand_empty();
            }
        }
        asp::warp_sort_best_first<NPL>(best, lane);
    }
    const double a_k = __shfl_sync(0xffffffffu, best[(kk - 1) / 32].s, (kk - 1) & 31);
    const double a_L = __shfl_sync(0xffffffffu, best[(LIST - 1) / 32].s, (LIST - 1) & 31);
    const bool complete = (a_L == -INFINITY) || (a_L < a_k - 2.0 * delta);
    if (!complete) {
        if (lane == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)i;
        return;
    }
    const double ni = norms[i];
#pragma unroll
    for (int t = 0; t < NPL; ++t) {
        const int e = lane + 32 * t;
        if (e < LIST && best[t].i != 0x7fffffff) {
            const int64_t j = best[t].i;
            const double d = exact_dist(seq_dot_row(xs, items + j * pitch, f), ni, norms[j]);
            best[t].s = (d <= eps) ? -d : -INFINITY;            // GRAPH_VARIABLES.md:7
            if (!(d <= eps)) best[t].i = 0x7fffffff;
        } else best[t] = asp::cand_empty();
    }
    asp::warp_sort_best_first<NPL>(best, lane);                  // (-d desc, index asc) == (d asc, index asc)
    int nvalid = 0;
#pragma unroll
    for (int t = 0; t < NPL; ++t) nvalid += __popc(__ballot_sync(0xffffffffu, best[t].i != 0x7fffffff));
    const int keep = nvalid < kk ? nvalid : kk;
#pragma unroll
    for (int t = 0; t < NPL; ++t) {
        const int e = lane + 32 * t;
        if (e < keep) { out_idx[i * kk + e] = best[t].i; out_dist[i * kk + e] = -best[t].s; }
    }
    if (lane == 0) out_cnt[i] = keep;
}

// slow path (exact_scan.cuh): value = -d(i, j), admissible = another item within eps; the k best by (d asc, index asc).
// Also the whole route of a Euclidean graph below the tensor-core size (every row takes it).
struct KnnScanPolicy {
    const double *items; int pitch; const double *norms; double eps; const int32_t *slow_list;
    int kk; int32_t *out_idx; double *out_dist; int32_t *out_cnt;
    const double *nsq; int distance;                                            // nsq: l2 / l2sq only
    struct Row { double ni, si; int64_t self; };
    struct Item { double nj, sj; };
    __device__ const double *query(int slot) const { return items + (int64_t)slow_list[slot] * pitch; }
    __device__ Row row(int slot) const
    {
        const int64_t i = slow_list[slot];
        return Row{norms[i], distance != ASP_DISTANCE_COSINE ? nsq[i] : 0.0, i};
    }
    __device__ Item item(int64_t j) const { return Item{norms[j], distance != ASP_DISTANCE_COSINE ? nsq[j] : 0.0}; }
    __device__ double value(const Row &r, const Item &it, double dot, int64_t j, bool &valid) const
    {
        const double d = exact_node_dist(distance, dot, r.ni, it.nj, r.si, it.sj);
        valid = (j != r.self) && (d <= eps);                                    // GRAPH_VARIABLES.md:7
        return -d;
    }
    __device__ void emit(int slot, int r, bool ok, double v, int64_t j) const
    {
        if (!ok) return;
        const int64_t row = slow_list[slot];
        out_idx[row * kk + r] = (int32_t)j;
        out_dist[row * kk + r] = -v;
    }
    __device__ void finish(int slot, int count) const { out_cnt[slow_list[slot]] = count; }
};

// ---------------------------------------------------------------- tcgen05 candidate pass (search_tc.cu) + exact stage 2
// Stage 1 is the search's tensor-core kernel with tau = 1 (score = cosine; DIST = l2 / l2sq: the score kind -d^2~), the
// items themselves as queries, lists of k + 1 (the item finds itself) and an emission floor at 1 - eps (-eps^2 | -eps); this
// kernel is the item-graph stage 2, one warp per row:
//   cut    (k+1)-th largest approximate score over all emitted candidates, minus 2 x the row's band
//   (A)    survivors re-scored in f64 with a coalesced warp-cooperative dot product (cosine, or -(|a|^2 + |b|^2 - 2 dot)
//          from the left-to-right sums of squares), best 32 kept
//   (B)    the candidates within 2 eps_fast of the (k+1)-th best get the oracle's distance (left-to-right dot,
//          exact_node_dist); self dropped, d <= eps decided on those values, k smallest by (d, index).
// A band that may extend beyond the 32 kept, a k-th neighbour whose cosine is not clearly positive (cosine only:
// rectification ties at d = 1 are ordered by index over ALL such items) or a full emission buffer send the row to the
// exact scan.  For l2 / l2sq eps_fast scales with |a|^2 + max |b|^2 (the dot's rounding is relative to the norms).
constexpr int KT_QUEUE = 96;

// Sums of FOUR per-lane values over the warp with 12 shuffles instead of 40: the halves of the warp first trade two values,
// the quarters one, then three plain butterfly steps.  Lanes 8u .. 8u+7 end with the total of value u.
__device__ __forceinline__ double warp_sum4_transposed(const double (&d)[4], int lane)
{
    const bool hi = (lane & 16) != 0;
    const double k0 = hi ? d[2] : d[0], k1 = hi ? d[3] : d[1];
    const double s0 = hi ? d[0] : d[2], s1 = hi ? d[1] : d[3];
    const double e0 = k0 + __shfl_xor_sync(0xffffffffu, s0, 16), e1 = k1 + __shfl_xor_sync(0xffffffffu, s1, 16);
    const bool mid = (lane & 8) != 0;
    double f = (mid ? e1 : e0) + __shfl_xor_sync(0xffffffffu, mid ? e0 : e1, 8);
#pragma unroll
    for (int off = 4; off > 0; off >>= 1) f += __shfl_xor_sync(0xffffffffu, f, off);
    return f;
}

template <int DIST>
__global__ void __launch_bounds__(KR_WARPS * 32)
knn_tc_rescore_kernel(const double *__restrict__ items, int64_t n, int f, int pitch, const double *__restrict__ norms,
                      const double *__restrict__ nsq, double nsq_max, double eps, int kk, int64_t b0, int64_t nq, int nsub, int capb, const float *__restrict__ delta_q,
                      double eps_fast, const float *__restrict__ emit_sc, const int32_t *__restrict__ emit_ix,
                      const int32_t *__restrict__ emit_cnt, const int32_t *__restrict__ qperm, const int32_t *__restrict__ row_map,
                      int64_t out_row0,
                      int32_t *__restrict__ out_idx, double *__restrict__ out_dist, int32_t *__restrict__ out_cnt,
                      int32_t *slow_list, int32_t *slow_count, unsigned long long *survivor_total)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *xs = reinterpret_cast<double *>(smem_raw) + (size_t)warp * pitch;
    int32_t *queue = reinterpret_cast<int32_t *>(reinterpret_cast<double *>(smem_raw) + (size_t)KR_WARPS * pitch) + warp * KT_QUEUE;
    const int64_t qi = (int64_t)blockIdx.x * KR_WARPS + warp;                    // visiting position inside the batch
    if (qi >= nq) return;
    const int64_t qp = qperm ? (int64_t)qperm[qi] : qi;                          // position in the batch as passed
    const int64_t i = row_map ? (int64_t)row_map[qp] : b0 + qp;                  // the row (item) this warp resolves
    for (int j = lane; j < pitch; j += 32) xs[j] = items[i * pitch + j];         // rows are zero padded to the pitch
    const int kq = kk + 1;                                                       // the item finds itself

    bool overflow = false;
    for (int c = lane; c < nsub; c += 32) overflow |= emit_cnt[qi * nsub + c] > capb;
    if (__any_sync(0xffffffffu, overflow)) {
        if (lane == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)i;
        return;
    }
    float cutoff;
    {
        float top[2] = {-INFINITY, -INFINITY};
        float floor32 = -INFINITY;
        for (int c = 0; c < nsub; ++c) {
            const int cnt = emit_cnt[qi * nsub + c];
            const size_t base = ((size_t)qi * nsub + c) * (size_t)capb;
            for (int e0 = 0; e0 < cnt; e0 += 32) {
                const int e = e0 + lane;
                const float v = (e < cnt) ? emit_sc[base + e] : -INFINITY;
                if (!__any_sync(0xffffffffu, v > floor32)) continue;
                top[1] = v;
                asp::warp_sort_desc_f32x2(top, lane);
                floor32 = __shfl_sync(0xffffffffu, top[0], 31);
            }
        }
        const float kth = __shfl_sync(0xffffffffu, top[0], kq - 1);              // -inf when fewer than k+1 were emitted
        cutoff = kth - 2.0f * delta_q[qi];
    }
    const double ni = norms[i];
    const double si = (DIST != ASP_DISTANCE_COSINE) ? nsq[i] : 0.0;
    const double eps_row = (DIST != ASP_DISTANCE_COSINE) ? eps_fast * (si + nsq_max) : eps_fast;
    __syncwarp();

    Cand best[2];
    best[0] = asp::cand_empty();
    best[1] = asp::cand_empty();
    int qn = 0;
    unsigned long long nsurv = 0;
    auto flush = [&](int count) {
        Cand mine = asp::cand_empty();
        double my_dot = 0.0;
        int my_item = -1;
        for (int s0 = 0; s0 < count; s0 += 4) {
            int ii[4];
            const double *rr[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { ii[u] = queue[(s0 + u < count) ? s0 + u : s0]; rr[u] = items + (int64_t)ii[u] * pitch; }
            double d[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 2
            for (int j = 2 * lane; j < pitch; j += 64) {
                const double2 qq = *reinterpret_cast<const double2 *>(xs + j);
                double2 a[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) a[u] = *reinterpret_cast<const double2 *>(rr[u] + j);
#pragma unroll
                for (int u = 0; u < 4; ++u) { d[u] = fma(qq.x, a[u].x, d[u]); d[u] = fma(qq.y, a[u].y, d[u]); }
            }
            const double tot = warp_sum4_transposed(d, lane);                    // lanes 8u .. 8u+7: the dot of row s0 + u
            const int u_mine = lane - s0;
            const double dd = __shfl_sync(0xffffffffu, tot, 8 * (u_mine & 3));
            if (u_mine >= 0 && u_mine < 4 && lane < count) {
                my_dot = dd;
                my_item = (u_mine == 0) ? ii[0] : (u_mine == 1) ? ii[1] : (u_mine == 2) ? ii[2] : ii[3];
            }
        }
        if (my_item >= 0) {
            if (DIST != ASP_DISTANCE_COSINE) {
                mine.s = -((si + nsq[my_item]) - 2.0 * my_dot);                  // fast -d^2
            } else {
                const double den = ni * norms[my_item];
                mine.s = (den != 0.0) ? my_dot / den : 0.0;                      // fast cosine
            }
            mine.i = my_item;
        }
        best[1] = mine;
        asp::warp_sort_best_first<2>(best, lane);
    };
    for (int c = 0; c < nsub; ++c) {
        const int cnt = emit_cnt[qi * nsub + c];
        const size_t base = ((size_t)qi * nsub + c) * (size_t)capb;
        for (int e0 = 0; e0 < cnt; e0 += 32) {
            const int e = e0 + lane;
            const bool keep = (e < cnt) && (emit_sc[base + e] >= cutoff);
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) queue[qn + __popc(m & ((1u << lane) - 1))] = emit_ix[base + e];
            qn += __popc(m);
            __syncwarp();
            if (qn >= 32) {
                flush(32);
                nsurv += 32;
                __syncwarp();
                if (lane < qn - 32) queue[lane] = queue[32 + lane];
                qn -= 32;
                __syncwarp();
            }
        }
    }
    if (qn > 0) { flush(qn); nsurv += qn; }

    const double kth = __shfl_sync(0xffffffffu, best[0].s, kq - 1);              // -inf when fewer than k+1 survivors
    const bool valid = best[0].i != 0x7fffffff;
    const bool in_band = valid && (best[0].s >= kth - 2.0 * eps_row);
    const unsigned band = __ballot_sync(0xffffffffu, in_band);
    if (band == 0xffffffffu || (DIST == ASP_DISTANCE_COSINE && kth != -INFINITY && kth <= 4.0 * eps_fast)) {
        if (lane == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)i;
        return;
    }
    Cand fin[1];
    fin[0] = asp::cand_empty();
    if (in_band && best[0].i != (int32_t)i) {
        const int64_t j = best[0].i;
        const double d = exact_node_dist(DIST, seq_dot_row(xs, items + j * pitch, f), ni, norms[j], si,
                                         (DIST != ASP_DISTANCE_COSINE) ? nsq[j] : 0.0);
        if (d <= eps) { fin[0].s = -d; fin[0].i = (int32_t)j; }                   // GRAPH_VARIABLES.md:7
    }
    asp::warp_sort_best_first<1>(fin, lane);                                     // (-d desc, index asc) == (d asc, index asc)
    const int nvalid = __popc(__ballot_sync(0xffffffffu, fin[0].i != 0x7fffffff));
    const int keep = nvalid < kk ? nvalid : kk;
    const int64_t orow = i - out_row0;
    if (lane < keep) { out_idx[orow * kk + lane] = fin[0].i; out_dist[orow * kk + lane] = -fin[0].s; }
    if (lane == 0) { out_cnt[orow] = keep; atomicAdd(survivor_total, nsurv); }
}

}  // namespace

// exact scan of the rows listed in slow_list (device) into lists indexed by item row
static int knn_slow_rows(asp_space *s, const asp_graph_params *gp, int distance, int64_t kk, const int32_t *slow_list, int nslow,
                         int32_t *idx, double *dist, int32_t *cnt)
{
    asp_ctx *ctx = s->ctx;
    const KnnScanPolicy pol{s->items, s->fp, s->norms, gp->eps, slow_list, (int)kk, idx, dist, cnt, s->nsq, distance};
    const int rc = asp_xs::run(ctx->stream, ctx->num_sms, pol, nslow, s->items, s->n_local, s->f, s->fp, kk,
                               [&](int k) { ctx->launches += k; });
    if (rc == 3) ASP_FAIL(ASP_ERR_NOMEM, "out of device memory in the exact scan of the item graph");
    if (rc == 1 || rc == 2) ASP_FAIL(ASP_ERR_UNSUPPORTED, "item graph: exact scan does not fit (k = %lld, %d features)", (long long)kk, s->f);
    if (rc != 0) ASP_FAIL(ASP_ERR_CUDA, "item graph: exact scan launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return ASP_OK;
}

static int item_knn_fp64(asp_space *s, const asp_graph_params *gp, asp_knn_lists *lists)
{
    constexpr int LIST = 32;
    constexpr int STAGES = 3;
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = s->n_local;
    const int f = s->f;
    if (n > 2147483647LL) ASP_FAIL(ASP_ERR_UNSUPPORTED, "item graph supports at most 2^31-1 items");
    int64_t kk = gp->k;
    if (kk > n - 1) kk = n - 1;
    if (kk < 0) kk = 0;
    if (kk > LIST - 4) ASP_FAIL(ASP_ERR_UNSUPPORTED, "item graph supports k <= %d (got %lld)", LIST - 4, (long long)gp->k);
    ASP_CHECK(lists->alloc(st, n, (int32_t)(kk > 0 ? kk : 1)));
    ASP_CUDA(cudaMemsetAsync(lists->cnt, 0, sizeof(int32_t) * (size_t)n, st));
    if (kk == 0) return ASP_OK;

    row_norms_kernel<<<(unsigned)(asp_ceil_div(n, 128) < 65535 ? asp_ceil_div(n, 128) : 65535), 128, 0, st>>>(
        s->items, n, f, s->fp, s->norms, s->inv_norms, nullptr);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);

    // rounding band of one approximate cosine (two summation orders of f terms, both norms) + the 1 - c rounding
    const double u = 1.1102230246251565e-16;
    const double delta = (4.0 * f + 64.0) * u;
    const double smin = 1.0 - gp->eps - delta;

    const int64_t tiles_total = asp_ceil_div(n, IT);
    const int64_t qblocks = asp_ceil_div(n, QT);
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
    const int nparts = (int)best_chunks;

    asp_scratch sc(st);
    double *cand_score = nullptr;
    int32_t *cand_idx = nullptr, *slow_list = nullptr, *slow_count = nullptr;
    ASP_CHECK(sc.get(&cand_score, (size_t)n * nparts * LIST));
    ASP_CHECK(sc.get(&cand_idx, (size_t)n * nparts * LIST));
    ASP_CHECK(sc.get(&slow_list, (size_t)n + 1));
    ASP_CHECK(sc.get(&slow_count, 1));
    ASP_CUDA(cudaMemsetAsync(slow_count, 0, sizeof(int32_t), st));

    ASP_CUDA(cudaEventRecord(ctx->ev0, st));
    {
        const size_t smem = (size_t)STAGES * STAGE_DOUBLES_S * 8 + sizeof(ListSmem<LIST>) + 128;
        dim3 grid((unsigned)qblocks, nparts);
        if (ctx->use_tma) {
            auto k = search_gemm_kernel<LIST, STAGES, true, 1>;
            ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k<<<grid, MMA_WARPS * 32, smem, st>>>(s->tmap_rows, s->tmap_rows, s->items, s->items, n, n, s->fp, s->inv_norms,
                                                   nullptr, s->inv_norms, nullptr, 1.0, smin, nparts, cand_score, cand_idx, nullptr);
        } else {
            auto k = search_gemm_kernel<LIST, STAGES, false, 1>;
            ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k<<<grid, MMA_WARPS * 32, smem, st>>>(s->tmap_rows, s->tmap_rows, s->items, s->items, n, n, s->fp, s->inv_norms,
                                                   nullptr, s->inv_norms, nullptr, 1.0, smin, nparts, cand_score, cand_idx, nullptr);
        }
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    ASP_CUDA(cudaEventRecord(ctx->ev1, st));
    {
        const size_t smem = (size_t)KR_WARPS * f * 8;
        ASP_CUDA(cudaFuncSetAttribute(knn_rescore_kernel<LIST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        knn_rescore_kernel<LIST><<<(unsigned)asp_ceil_div(n, KR_WARPS), KR_WARPS * 32, smem, st>>>(
            s->items, n, f, s->fp, s->norms, gp->eps, (int)kk, nparts, cand_score, cand_idx, delta, lists->idx, lists->dist,
            lists->cnt, slow_list, slow_count);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    int32_t nslow = 0;
    ASP_CUDA(cudaMemcpyAsync(&nslow, slow_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->stats["knn_stage1_ms"] = ms;
    ctx->stats["knn_slow_rows"] = nslow;
    ctx->stats["knn_stage1_is_tc"] = 0.0;
    if (nslow > 0) ASP_CHECK(knn_slow_rows(s, gp, ASP_DISTANCE_COSINE, kk, slow_list, nslow, lists->idx, lists->dist, lists->cnt));
    return ASP_OK;
}

// Item-graph neighbour lists on the tensor cores: batches of 64k rows through asp_tc_stage1, exact stage 2 above.
__global__ void gather_rows_kernel(const double *__restrict__ items, int pitch, const double *__restrict__ norms,
                                   const int32_t *__restrict__ rows, int64_t nrows, double *__restrict__ out, double *__restrict__ out_norms)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < nrows; r += nwarps) {
        const int64_t src = rows[r];
        for (int j = lane; j < pitch; j += 32) out[r * pitch + j] = items[src * pitch + j];
        if (lane == 0) out_norms[r] = norms[src];
    }
}

// rows [row_begin, row_end) against all items of the space; lists->idx/dist/cnt hold (row_end - row_begin) rows.
//   pass 1  every row, candidate pass with as few MMA terms as the residual norms allow (usually ONE fp16 term)
//   pass 2  the rows whose emission lists or bands overflowed (dense neighbourhoods: the 1-term band of ~1e-4 in cosine
//           can hold hundreds of neighbours) are gathered and redone with the two-term split (band ~1e-6)
//   pass 3  what is still unresolved (long runs of exact ties around the k-th neighbour) takes the exact scan
static int item_knn_tc(asp_space *s, const asp_graph_params *gp, int distance, int64_t kk, int64_t row_begin, int64_t row_end,
                       asp_knn_lists *lists)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = s->n_local;
    const int f = s->f;
    const double u = 1.1102230246251565e-16;
    const double eps_fast = (4.0 * f + 64.0) * u * 2.0;
    const bool l2 = distance != ASP_DISTANCE_COSINE;
    double floor = (gp->eps < 2.0) ? 1.0 - gp->eps - eps_fast : -INFINITY;         // cos < 1 - eps can never be a neighbour
    double nsq_max = 0.0;
    if (l2) {
        // score -d^2: d <= eps needs -d^2 >= -eps^2 (l2) | -eps (l2sq); the stage-1 score is f32, so the norms must square
        // well inside its range
        double norm_max = 0.0;
        ASP_CHECK(asp_device_max(ctx, s->norms, n, &norm_max));
        ASP_CHECK(asp_device_max(ctx, s->nsq, n, &nsq_max));
        if (!(norm_max <= 1e18))
            ASP_FAIL(ASP_ERR_UNSUPPORTED, "Euclidean item graph: norms up to %g exceed the f32 range of the tensor-core pass (limit 1e18)", norm_max);
        const double e2 = (distance == ASP_DISTANCE_L2) ? gp->eps * gp->eps : gp->eps;
        floor = (gp->eps >= 0.0 && e2 < 1e300) ? -(e2 * (1.0 + 1e-12)) : -INFINITY;
    }
    const int64_t rows = row_end - row_begin;
    asp_scratch sc(st);
    int32_t *slow1 = nullptr, *slow2 = nullptr, *counts = nullptr;                  // counts[0], counts[1]
    unsigned long long *counter = nullptr;
    ASP_CHECK(sc.get(&slow1, (size_t)rows + 1));
    ASP_CHECK(sc.get(&slow2, (size_t)rows + 1));
    ASP_CHECK(sc.get(&counts, 2));
    ASP_CHECK(sc.get(&counter, 1));
    ASP_CUDA(cudaMemsetAsync(counts, 0, sizeof(int32_t) * 2, st));
    ASP_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), st));
    const size_t rsmem = (size_t)KR_WARPS * s->fp * 8 + KR_WARPS * KT_QUEUE * 4;
    auto rescore = (distance == ASP_DISTANCE_L2) ? knn_tc_rescore_kernel<ASP_DISTANCE_L2>
                 : (distance == ASP_DISTANCE_L2SQ) ? knn_tc_rescore_kernel<ASP_DISTANCE_L2SQ> : knn_tc_rescore_kernel<ASP_DISTANCE_COSINE>;
    ASP_CUDA(cudaFuncSetAttribute(rescore, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem));
    int64_t batch = 65536;
    if (const char *e = getenv("ASP_KNN_BATCH")) { const long v = atol(e); if (v >= 128) batch = v; }
    double stage1_ms = 0.0, stage2_ms = 0.0;
    int rc = ASP_OK, terms_pass1 = 0;

    // one batch of query rows: q = their vectors (contiguous), row_map = their item indices (nullptr: b0 + position)
    auto run_batch = [&](const double *q, const double *qn, int64_t nq, int64_t b0, const int32_t *row_map, int terms,
                         int32_t *slow_list, int32_t *slow_count, int *terms_used) -> int {
        asp_tc_batch b;
        int r = asp_tc_stage1(s, q, nq, s->fp, nullptr, qn, 1.0, kk + 1, floor, terms, 2048, nullptr, &b, l2);
        if (r == ASP_OK) {
            rescore<<<(unsigned)asp_ceil_div(nq, KR_WARPS), KR_WARPS * 32, rsmem, st>>>(
                s->items, n, f, s->fp, s->norms, s->nsq, nsq_max, gp->eps, (int)kk, b0, nq, b.nsub, b.capb, b.delta_q, eps_fast, b.emit_sc, b.emit_ix,
                b.emit_cnt, b.qperm, row_map, row_begin, lists->idx, lists->dist, lists->cnt, slow_list, slow_count, counter);
            if (cudaGetLastError() != cudaSuccess) { asp_set_error("knn_tc_rescore_kernel launch failed"); r = ASP_ERR_CUDA; }
            ASP_LAUNCHED(ctx);
            cudaEventRecord(ctx->ev2, st);
            cudaEventSynchronize(ctx->ev2);
            float m1 = 0.f, m2 = 0.f;
            cudaEventElapsedTime(&m1, ctx->ev0, ctx->ev1);
            cudaEventElapsedTime(&m2, ctx->ev1, ctx->ev2);
            stage1_ms += m1; stage2_ms += m2;
            *terms_used = b.nterms;
        }
        return r;
    };

    // Dense neighbourhoods (C5: 34k items per cluster in 768 dimensions, where the distances inside a cluster concentrate)
    // overflow the 1-term band on EVERY row: when more than half of the first batch does, the remaining batches go
    // straight to the two-term split instead of paying for a pass that decides nothing.
    bool direct3 = false;
    int64_t rows_direct3 = 0;
    int32_t h_counts[2] = {0, 0};
    for (int64_t b0 = row_begin; b0 < row_end && rc == ASP_OK; b0 += batch) {
        const int64_t nq = (row_end - b0 < batch) ? row_end - b0 : batch;
        if (direct3) {
            int used = 0;
            rc = run_batch(s->items + b0 * s->fp, s->norms + b0, nq, b0, nullptr, 3, slow2, counts + 1, &used);
            rows_direct3 += nq;
            continue;
        }
        // the first batch picks the number of MMA terms from its residual norms; the later batches are held to the same
        // choice (their per-row bands stay valid either way), so that `slow1` holds rows of ONE kind: all of them still owed
        // the two-term pass (1 term) or all of them owed the exact scan (3 terms)
        rc = run_batch(s->items + b0 * s->fp, s->norms + b0, nq, b0, nullptr, b0 == row_begin ? 0 : terms_pass1, slow1, counts, &terms_pass1);
        if (rc == ASP_OK && b0 == row_begin && terms_pass1 == 1 && b0 + batch < row_end) {
            ASP_CUDA(cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, st));
            ASP_CUDA(cudaStreamSynchronize(st));
            direct3 = (int64_t)h_counts[0] * 2 > nq;
        }
    }
    if (rc == ASP_OK) {
        ASP_CUDA(cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
    }
    const int32_t n_pass2 = (terms_pass1 == 1) ? h_counts[0] : 0;
    const int32_t *final_list = direct3 ? slow2 : slow1;
    int32_t n_final = direct3 ? h_counts[1] : h_counts[0];
    if (rc == ASP_OK && n_pass2 > 0) {
        asp_scratch qsc(st);
        double *qbuf = nullptr, *qnorm = nullptr;
        const int64_t chunk = n_pass2 < batch ? n_pass2 : batch;
        ASP_CHECK(qsc.get(&qbuf, (size_t)chunk * s->fp));
        ASP_CHECK(qsc.get(&qnorm, (size_t)chunk));
        for (int64_t c0 = 0; c0 < n_pass2 && rc == ASP_OK; c0 += chunk) {
            const int64_t nq = (n_pass2 - c0 < chunk) ? n_pass2 - c0 : chunk;
            gather_rows_kernel<<<ctx->num_sms * 4, 256, 0, st>>>(s->items, s->fp, s->norms, slow1 + c0, nq, qbuf, qnorm);
            ASP_LAUNCHED(ctx);
            int used = 0;
            rc = run_batch(qbuf, qnorm, nq, 0, slow1 + c0, 3, slow2, counts + 1, &used);
        }
        if (rc == ASP_OK) {
            ASP_CUDA(cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, st));
            ASP_CUDA(cudaStreamSynchronize(st));
        }
        final_list = slow2;
        n_final = h_counts[1];
    }
    unsigned long long nsurv = 0;
    if (rc == ASP_OK) {
        ASP_CUDA(cudaMemcpyAsync(&nsurv, counter, sizeof(nsurv), cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
        ctx->stats["knn_stage1_ms"] = stage1_ms;
        ctx->stats["knn_stage2_ms"] = stage2_ms;
        ctx->stats["knn_rows_two_term"] = (double)n_pass2 + (double)rows_direct3;
        ctx->stats["knn_rows_one_term_wasted"] = n_pass2;
        ctx->stats["knn_slow_rows"] = n_final;
        ctx->stats["knn_stage1_is_tc"] = 1.0;
        ctx->stats["knn_rescored_per_row"] = (double)nsurv / (double)(rows > 0 ? rows : 1);
        if (n_final > 262144) {                                          // the batched scan does ~3000 rows/s at 1M x 384
            asp_set_error("item graph: %d rows need the exact scan even after the two-term pass (long runs of ties around the "
                          "k-th neighbour?); use ASP_KNN_STAGE1=fp64", n_final);
            rc = ASP_ERR_UNSUPPORTED;
        } else if (n_final > 0) {                                     // the exact kernels index the lists by GLOBAL row
            rc = knn_slow_rows(s, gp, distance, kk, final_list, n_final, lists->idx - row_begin * kk, lists->dist - row_begin * kk,
                               lists->cnt - row_begin);
        }
    }
    return rc;
}

// norms (and, for the Euclidean distances, the sums of squares) of every item
static int knn_row_norms(asp_space *s, int distance)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = s->n_local;
    if (distance != ASP_DISTANCE_COSINE && !s->nsq) ASP_CUDA(cudaMallocAsync(&s->nsq, sizeof(double) * (size_t)(n > 0 ? n : 1), st));
    row_norms_kernel<<<(unsigned)(asp_ceil_div(n, 128) < 65535 ? asp_ceil_div(n, 128) : 65535), 128, 0, st>>>(
        s->items, n, s->f, s->fp, s->norms, s->inv_norms, distance != ASP_DISTANCE_COSINE ? s->nsq : nullptr);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}

// Euclidean graph below the tensor-core size (or ASP_KNN_STAGE1=fp64): every row takes the batched exact scan
static int item_knn_scan_all(asp_space *s, const asp_graph_params *gp, int distance, int64_t kk, asp_knn_lists *lists)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = s->n_local;
    asp_scratch sc(st);
    int32_t *rows = nullptr;
    ASP_CHECK(sc.get(&rows, (size_t)n));
    iota_rows_kernel<<<ctx->num_sms * 4, 256, 0, st>>>(rows, n);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    const int rc = knn_slow_rows(s, gp, distance, kk, rows, (int)n, lists->idx, lists->dist, lists->cnt);
    ctx->stats["knn_stage1_ms"] = 0.0;
    ctx->stats["knn_slow_rows"] = (double)n;
    ctx->stats["knn_stage1_is_tc"] = 0.0;
    return rc;
}

int asp_item_knn(asp_space *s, const asp_graph_params *gp, int distance, asp_knn_lists *lists)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = s->n_local;
    int64_t kk = gp->k;
    if (kk > n - 1) kk = n - 1;
    if (kk < 0) kk = 0;
    const char *force = getenv("ASP_KNN_STAGE1");
    const bool want_fp64 = force && force[0] == 'f', want_tc = force && force[0] == 't';
    const bool tc_ok = kk >= 1 && kk + 1 <= 31 && n < 2147483647LL && s->fp <= 6144;
    const bool l2 = distance != ASP_DISTANCE_COSINE;
    const bool small = want_fp64 || (!want_tc && n < 8192);
    if (!l2 && (!tc_ok || small)) return item_knn_fp64(s, gp, lists);
    if (l2 && kk > 30) ASP_FAIL(ASP_ERR_UNSUPPORTED, "the Euclidean item graph supports k <= 30 (got %lld)", (long long)gp->k);
    if (l2 && !small && !tc_ok)
        ASP_FAIL(ASP_ERR_UNSUPPORTED, "the Euclidean item graph on the tensor cores supports at most 6144 features (got %d)", s->f);

    ASP_CHECK(lists->alloc(st, n, (int32_t)(kk > 0 ? kk : 1)));
    ASP_CUDA(cudaMemsetAsync(lists->cnt, 0, sizeof(int32_t) * (size_t)n, st));
    ASP_CHECK(knn_row_norms(s, distance));
    if (kk == 0) return ASP_OK;
    if (small) return item_knn_scan_all(s, gp, distance, kk, lists);
    return item_knn_tc(s, gp, distance, kk, 0, n, lists);
}

// neighbour lists of rows [row_begin, row_end) only (multi-GPU item graph: every rank holds all items and resolves
// its own rows); tensor-core pass only
int asp_item_knn_rows_impl(asp_space *s, const asp_graph_params *gp, int distance, int64_t row_begin, int64_t row_end,
                           asp_knn_lists *lists)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = s->n_local, rows = row_end - row_begin;
    int64_t kk = gp->k;
    if (kk > n - 1) kk = n - 1;
    if (row_begin < 0 || row_end > n || rows < 0) ASP_FAIL(ASP_ERR_ARG, "row range [%lld, %lld) outside [0, %lld)", (long long)row_begin, (long long)row_end, (long long)n);
    if (kk < 1 || kk + 1 > 31 || n >= 2147483647LL || s->fp > 6144)
        ASP_FAIL(ASP_ERR_UNSUPPORTED, "the row-range item graph needs 1 <= k <= 30 (got %lld) and <= 6144 features", (long long)gp->k);
    ASP_CHECK(lists->alloc(st, rows, (int32_t)kk));
    ASP_CUDA(cudaMemsetAsync(lists->cnt, 0, sizeof(int32_t) * (size_t)(rows > 0 ? rows : 1), st));
    ASP_CHECK(knn_row_norms(s, distance));
    if (rows == 0) return ASP_OK;
    return item_knn_tc(s, gp, distance, kk, row_begin, row_end, lists);
}
