// range.cu -- range search: per query EVERY (allowed) item with score >= min_score, ordered by (score desc, index asc), the
// scores the oracle's bit for bit (asp_search_range_batch).
//
// Stage 1 is the tcgen05 candidate pass of the search (search_tc.cu, asp_tc_stage1) run with topk = 0 and score_floor =
// min_score (clamped to [-2, 2]): its running lists never fill, so the emission threshold of a query row stays at
// score_floor - delta_q, delta_q being the row's bound on |s~ - s|.  A hit has s >= min_score, hence s~ >= min_score - delta_q:
// it is emitted (or the query's emission buffer overflows).  Membership is then decided on the exact value alone -- no band,
// no tie question.  Everything after stage 1 lives here:
//   tc_range_count_kernel  one warp per query (lambda_q visiting order, mapped through qperm as tc_rescore_kernel does): a
//                          query with an overflowing emission buffer goes to the slow list; otherwise every emitted candidate
//                          gets its reference-order score (one candidate per lane: left-to-right __dmul_rn / __dadd_rn dot,
//                          the oracle's expression) and is kept iff score >= min_score.  Scores are kept beside the emission
//                          lists; per-query hit counts go to the host.
//   tc_range_fill_kernel   the same walk, kept hits compacted (ballot) into the query's CSR segment.
//   range_scan_kernel      the exact range scan of the slow list (and of every query when the tensor-core route does not
//                          apply): block (x, y) = item range x of QPB queries, each thread one item row at a time, read once
//                          for the QPB ordered dots.  A count pass, a host-side exclusive scan, a fill pass with a shared
//                          cursor per (query, item range); the sort fixes the order.  No topk limit: a row holds up to
//                          n_local hits.
//   sort                   per query segment by (score desc, index asc) on an order-preserving 64-bit key of the score plus
//                          the index: segments of up to SORT_S entries by one CTA (bitonic network in shared memory), longer
//                          ones as SORT_S-blocks followed by merge passes (each element finds its rank in the partner run by
//                          binary search).
// The scan's value and validity are those of the search's exact scan (search.cu, SearchScanPolicy): the same score expression,
// a row that is not allowed is skipped.
#include "common.cuh"
#include "range.cuh"

#include <math.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>

namespace {

constexpr int RW = 4;                 // warps (queries) per CTA of the tensor-core stage 2
constexpr int SC_THREADS = 256, SC_CHUNK = 1024;
constexpr int SORT_S = 8192;          // longest segment one CTA sorts: 8192 x 16 B = 128 KB of shared memory
constexpr int64_t SUB_BATCH = 32768;  // queries per sub-batch (see asp_range_sub_batch)

__device__ __forceinline__ double exact_score(double dot, double nq, double nx, double tau, double lq, double lx)
{
    const double den = __dmul_rn(nq, nx);
    const double c = (den == 0.0) ? 0.0 : __ddiv_rn(dot, den);
    const double prox = __ddiv_rn(1.0, __dadd_rn(1.0, fabs(__dsub_rn(lq, lx))));
    return __dadd_rn(__dmul_rn(tau, c), __dmul_rn(__dsub_rn(1.0, tau), prox));
}

__device__ __forceinline__ double seq_dot(const double *__restrict__ qv, const double *__restrict__ row, int f)
{
    double d = 0.0;
    int j = 0;
    for (; j + 2 <= f; j += 2) {
        const double2 x = *reinterpret_cast<const double2 *>(row + j);
        d = __dadd_rn(d, __dmul_rn(qv[j], x.x));
        d = __dadd_rn(d, __dmul_rn(qv[j + 1], x.y));
    }
    for (; j < f; ++j) d = __dadd_rn(d, __dmul_rn(qv[j], row[j]));
    return d;
}

// ------------------------------------------------------------------ stage 2 of the tensor-core route
__global__ void __launch_bounds__(RW * 32)
tc_range_count_kernel(const double *__restrict__ q, int qpitch, int64_t nq, const double *__restrict__ items, int f, int pitch,
                      const double *__restrict__ norm_x, const double *__restrict__ lam_x, const double *__restrict__ norm_q,
                      const double *__restrict__ lam_q, double tau, double min_score, int nstreams, int capb,
                      const int32_t *__restrict__ emit_ix, const int32_t *__restrict__ emit_cnt, const int32_t *__restrict__ qperm,
                      double *__restrict__ exact, int64_t *__restrict__ counts, int32_t *slow_list, int32_t *slow_count)
{
    extern __shared__ __align__(16) double rq_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t qi = (int64_t)blockIdx.x * RW + warp;                          // visiting position
    if (qi >= nq) return;
    const int64_t oq = qperm ? (int64_t)qperm[qi] : qi;                          // the caller's query
    double *qs = rq_smem + (size_t)warp * pitch;
    for (int j = lane; j < f; j += 32) qs[j] = q[oq * qpitch + j];
    bool overflow = false;
    for (int c = lane; c < nstreams; c += 32) overflow |= emit_cnt[qi * nstreams + c] > capb;
    if (__any_sync(0xffffffffu, overflow)) {
        if (lane == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)oq;
        return;
    }
    __syncwarp();
    const double nqv = norm_q[oq], lqv = lam_q[oq];
    int64_t kept = 0;
    for (int c = 0; c < nstreams; ++c) {
        const int cnt = emit_cnt[qi * nstreams + c];
        const size_t base = ((size_t)qi * nstreams + c) * (size_t)capb;
        for (int e = lane; e - lane < cnt; e += 32) {
            bool keep = false;
            if (e < cnt) {
                const int32_t it = emit_ix[base + e];
                const double sc = exact_score(seq_dot(qs, items + (int64_t)it * pitch, f), nqv, norm_x[it], tau, lqv, lam_x[it]);
                keep = sc >= min_score;
                exact[base + e] = keep ? sc : NAN;
            }
            kept += __popc(__ballot_sync(0xffffffffu, keep));
        }
    }
    if (lane == 0) counts[oq] = kept;
}

__global__ void __launch_bounds__(RW * 32)
tc_range_fill_kernel(int64_t nq, int nstreams, int capb, const int32_t *__restrict__ emit_ix, const int32_t *__restrict__ emit_cnt,
                     const int32_t *__restrict__ qperm, const double *__restrict__ exact, const int64_t *__restrict__ offsets,
                     int64_t row0, int64_t *__restrict__ out_idx, double *__restrict__ out_score)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t qi = (int64_t)blockIdx.x * RW + warp;
    if (qi >= nq) return;
    bool overflow = false;
    for (int c = lane; c < nstreams; c += 32) overflow |= emit_cnt[qi * nstreams + c] > capb;
    if (__any_sync(0xffffffffu, overflow)) return;                               // answered by the scan
    const int64_t oq = qperm ? (int64_t)qperm[qi] : qi;
    int64_t pos = offsets[oq];
    for (int c = 0; c < nstreams; ++c) {
        const int cnt = emit_cnt[qi * nstreams + c];
        const size_t base = ((size_t)qi * nstreams + c) * (size_t)capb;
        for (int e = lane; e - lane < cnt; e += 32) {
            const double sc = (e < cnt) ? exact[base + e] : NAN;
            const bool keep = !isnan(sc);
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int64_t o = pos + __popc(m & ((1u << lane) - 1u));
                out_idx[o] = row0 + emit_ix[base + e];
                out_score[o] = sc;
            }
            pos += __popc(m);
        }
    }
}

// ------------------------------------------------------------------ exact range scan
// FILL == false: part_cnt[slot][x] = hits of query list[slot] among the rows of item range x.
// FILL == true:  the hits written at offsets[list[slot]] + part_cnt[slot][x] (part_cnt then holds the exclusive prefix over x).
template <int QPB, bool FILL, bool FILTER>
__global__ void __launch_bounds__(SC_THREADS)
range_scan_kernel(const double *__restrict__ q, int qpitch, const int32_t *__restrict__ list, int first, int nslow,
                  const double *__restrict__ items, int64_t n_local, int f, int pitch, const double *__restrict__ norm_x,
                  const double *__restrict__ lam_x, const double *__restrict__ norm_q, const double *__restrict__ lam_q, double tau,
                  double min_score, const uint32_t *__restrict__ allowed, int64_t *__restrict__ part_cnt,
                  const int64_t *__restrict__ offsets, int64_t row0, int64_t *__restrict__ out_idx, double *__restrict__ out_score)
{
    extern __shared__ __align__(16) double sc_smem[];
    double *qs = sc_smem;                                                        // [QPB][f]
    __shared__ unsigned long long cur[QPB];
    const int slot0 = first + blockIdx.y * QPB;
    double nqv[QPB], lqv[QPB];
    bool live[QPB];
#pragma unroll
    for (int u = 0; u < QPB; ++u) {
        live[u] = slot0 + u < first + nslow;
        const int64_t oq = list[live[u] ? slot0 + u : first];
        nqv[u] = norm_q[oq];
        lqv[u] = lam_q[oq];
    }
    for (int j = threadIdx.x; j < QPB * f; j += SC_THREADS) {
        const int u = j / f, t = j - u * f;
        qs[j] = live[u] ? q[(int64_t)list[slot0 + u] * qpitch + t] : 0.0;
    }
    if (threadIdx.x < QPB) cur[threadIdx.x] = 0ull;
    __syncthreads();
    const int64_t per = (n_local + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = blockIdx.x * per, r1 = (r0 + per < n_local) ? r0 + per : n_local;
    int64_t base[QPB];
    if (FILL) {
#pragma unroll
        for (int u = 0; u < QPB; ++u)
            base[u] = live[u] ? offsets[list[slot0 + u]] + part_cnt[(size_t)(slot0 + u - first) * gridDim.x + blockIdx.x] : 0;
    }
    for (int64_t it = r0 + threadIdx.x; it < r1; it += SC_THREADS) {
        if (FILTER && !asp_allowed(allowed, it)) continue;
        const double *row = items + it * pitch;
        double d[QPB];
#pragma unroll
        for (int u = 0; u < QPB; ++u) d[u] = 0.0;
        int j = 0;
        for (; j + 2 <= f; j += 2) {                                             // one load of the row for the QPB ordered sums
            const double2 xv = *reinterpret_cast<const double2 *>(row + j);
#pragma unroll
            for (int u = 0; u < QPB; ++u) {
                d[u] = __dadd_rn(d[u], __dmul_rn(qs[u * f + j], xv.x));
                d[u] = __dadd_rn(d[u], __dmul_rn(qs[u * f + j + 1], xv.y));
            }
        }
        for (; j < f; ++j)
#pragma unroll
            for (int u = 0; u < QPB; ++u) d[u] = __dadd_rn(d[u], __dmul_rn(qs[u * f + j], row[j]));
        const double nx = norm_x[it], lx = lam_x[it];
#pragma unroll
        for (int u = 0; u < QPB; ++u) {
            if (!live[u]) continue;
            const double sc = exact_score(d[u], nqv[u], nx, tau, lqv[u], lx);
            if (!(sc >= min_score)) continue;
            const unsigned long long p = atomicAdd(&cur[u], 1ull);
            if (FILL) { out_idx[base[u] + p] = row0 + it; out_score[base[u] + p] = sc; }
        }
    }
    if (!FILL) {
        __syncthreads();
        if (threadIdx.x < QPB && live[threadIdx.x])
            part_cnt[(size_t)(slot0 + threadIdx.x - first) * gridDim.x + blockIdx.x] = (int64_t)cur[threadIdx.x];
    }
}

// per slow query: its item ranges' counts -> exclusive prefix (in place), the total -> counts[query]
__global__ void scan_prefix_kernel(int nslow, int nparts, const int32_t *__restrict__ list, int64_t *__restrict__ part_cnt,
                                   int64_t *__restrict__ counts)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nslow; i += gridDim.x * blockDim.x) {
        int64_t *pc = part_cnt + (size_t)i * nparts;
        int64_t run = 0;
        for (int x = 0; x < nparts; ++x) { const int64_t c = pc[x]; pc[x] = run; run += c; }
        counts[list[i]] = run;
    }
}

__global__ void iota32_kernel(int32_t *__restrict__ p, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = (int32_t)i;
}

// ------------------------------------------------------------------ sort
struct SKey { uint64_t k; int64_t i; };
__device__ __forceinline__ bool skey_less(const SKey &a, const SKey &b) { return a.k < b.k || (a.k == b.k && a.i < b.i); }

// one CTA sorts entries [start, start + len) (len <= SORT_S) of (out_idx, out_score) in place by (score desc, index asc)
__device__ void cta_sort(int64_t start, int len, int64_t *__restrict__ out_idx, double *__restrict__ out_score, SKey *keys)
{
    int p2 = 2;
    while (p2 < len) p2 <<= 1;
    for (int i = threadIdx.x; i < p2; i += blockDim.x) {
        SKey k;
        if (i < len) { k.k = asp_range::desc_key(out_score[start + i]); k.i = out_idx[start + i]; }
        else { k.k = ~0ull; k.i = INT64_MAX; }
        keys[i] = k;
    }
    for (int size = 2; size <= p2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < p2 / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const SKey a = keys[lo], b = keys[hi];
                if (up ? skey_less(b, a) : skey_less(a, b)) { keys[lo] = b; keys[hi] = a; }
            }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
        out_idx[start + i] = keys[i].i;
        out_score[start + i] = asp_range::key_score(keys[i].k);
    }
}

// one CTA per query whose segment holds 2 .. SORT_S entries
__global__ void sort_segments_kernel(int64_t nq, const int64_t *__restrict__ offsets, int64_t *__restrict__ out_idx,
                                     double *__restrict__ out_score)
{
    extern __shared__ __align__(16) unsigned char sort_smem[];
    for (int64_t qi = blockIdx.x; qi < nq; qi += gridDim.x) {
        const int64_t a = offsets[qi], len = offsets[qi + 1] - a;
        if (len < 2 || len > SORT_S) continue;
        cta_sort(a, (int)len, out_idx, out_score, reinterpret_cast<SKey *>(sort_smem));
        __syncthreads();
    }
}

// one CTA per SORT_S-block of the long segments: blocks[2 b] = start, blocks[2 b + 1] = length
__global__ void sort_blocks_kernel(const int64_t *__restrict__ blocks, int64_t *__restrict__ out_idx, double *__restrict__ out_score)
{
    extern __shared__ __align__(16) unsigned char sort_smem[];
    cta_sort(blocks[2 * blockIdx.x], (int)blocks[2 * blockIdx.x + 1], out_idx, out_score, reinterpret_cast<SKey *>(sort_smem));
}

// One merge pass over the long segments (segs[2 s] = start, segs[2 s + 1] = length): sorted runs of width w are merged in
// pairs from (si, ss) into (di, ds).  An element's place = its pair's start + its position in its run + the number of
// elements of the partner run before it (no two entries of a query compare equal: the indices differ).
__global__ void merge_pass_kernel(int nseg, const int64_t *__restrict__ segs, int64_t w, const int64_t *__restrict__ si,
                                  const double *__restrict__ ss, int64_t *__restrict__ di, double *__restrict__ ds)
{
    for (int sg = blockIdx.y; sg < nseg; sg += gridDim.y) {
        const int64_t start = segs[2 * sg], len = segs[2 * sg + 1];
        for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < len; e += (int64_t)gridDim.x * blockDim.x) {
            const int64_t run = e / w, pair0 = (run >> 1) * 2 * w;
            const bool in_a = (run & 1) == 0;
            const int64_t o0 = in_a ? pair0 + w : pair0;                         // the partner run [o0, o1)
            const int64_t o1 = in_a ? ::min(pair0 + 2 * w, len) : pair0 + w;
            const double s = ss[start + e];
            const int64_t id = si[start + e];
            int64_t lo = ::min(o0, len), hi = ::min(o1, len);
            const int64_t b0 = lo;
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (asp_range::before(ss[start + mid], si[start + mid], s, id)) lo = mid + 1; else hi = mid;
            }
            const int64_t own = in_a ? e - pair0 : e - (pair0 + w);
            const int64_t pos = pair0 + own + (lo - b0);
            di[start + pos] = id;
            ds[start + pos] = s;
        }
    }
}

template <int QPB, bool FILL, bool FILTER>
int launch_scan(const asp_space *s, const double *q_dev, int32_t qpitch, const int32_t *list, int nslow, int nparts,
                const double *lam_dev, const double *norm_dev, double tau, double min_score, const uint32_t *allowed,
                int64_t *part_cnt, const int64_t *offsets, int64_t *out_idx, double *out_score)
{
    asp_ctx *ctx = s->ctx;
    auto k = range_scan_kernel<QPB, FILL, FILTER>;
    const size_t smem = sizeof(double) * (size_t)QPB * s->f;
    ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ngroups = asp_ceil_div(nslow, QPB);
    for (int64_t g0 = 0; g0 < ngroups; g0 += 65535) {
        const int64_t ng = std::min<int64_t>(65535, ngroups - g0);
        const int first = (int)(g0 * QPB);
        const int count = (int)std::min<int64_t>(ng * QPB, nslow - first);
        k<<<dim3((unsigned)nparts, (unsigned)ng), SC_THREADS, smem, ctx->stream>>>(
            q_dev, qpitch, list, first, count, s->items, s->n_local, s->f, s->fp, s->norms, s->lambdas, norm_dev, lam_dev, tau,
            min_score, allowed, part_cnt, offsets, s->row0, out_idx, out_score);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    return ASP_OK;
}

template <bool FILL>
int run_scan(const asp_space *s, const double *q_dev, int32_t qpitch, const int32_t *list, int nslow, int nparts,
             const double *lam_dev, const double *norm_dev, double tau, double min_score, const uint32_t *allowed,
             int64_t *part_cnt, const int64_t *offsets, int64_t *out_idx, double *out_score)
{
    const bool wide = sizeof(double) * 4 * (size_t)s->f <= 200 * 1024;
#define ASP_RANGE_SCAN(QPB, FILTER) \
    launch_scan<QPB, FILL, FILTER>(s, q_dev, qpitch, list, nslow, nparts, lam_dev, norm_dev, tau, min_score, allowed, part_cnt, \
                                   offsets, out_idx, out_score)
    if (wide) return allowed ? ASP_RANGE_SCAN(4, true) : ASP_RANGE_SCAN(4, false);
    return allowed ? ASP_RANGE_SCAN(1, true) : ASP_RANGE_SCAN(1, false);
#undef ASP_RANGE_SCAN
}

// sorts every query segment of (out_idx, out_score) by (score desc, index asc); h_off: the offsets on the host
int sort_segments(asp_ctx *ctx, int64_t nq, const int64_t *h_off, const int64_t *d_off, int64_t nnz, int64_t *out_idx,
                  double *out_score)
{
    cudaStream_t st = ctx->stream;
    int64_t max_short = 0;
    std::vector<int64_t> segs, blocks;                          // long segments: (start, len); their SORT_S-blocks
    for (int64_t q = 0; q < nq; ++q) {
        const int64_t len = h_off[q + 1] - h_off[q];
        if (len <= SORT_S) { max_short = std::max(max_short, len); continue; }
        segs.push_back(h_off[q]);
        segs.push_back(len);
        for (int64_t b = 0; b < len; b += SORT_S) { blocks.push_back(h_off[q] + b); blocks.push_back(std::min<int64_t>(SORT_S, len - b)); }
    }
    if (max_short >= 2) {
        int p2 = 2;
        while (p2 < max_short) p2 <<= 1;
        const size_t smem = sizeof(SKey) * (size_t)p2;
        const int threads = std::max(32, std::min(512, p2 / 2));
        ASP_CUDA(cudaFuncSetAttribute(sort_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        sort_segments_kernel<<<(unsigned)std::min<int64_t>(nq, 1 << 20), threads, smem, st>>>(nq, d_off, out_idx, out_score);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    if (segs.empty()) return ASP_OK;
    asp_scratch sc(st);
    int64_t *d_segs = nullptr, *d_blocks = nullptr, *t_idx = nullptr;
    double *t_score = nullptr;
    ASP_CHECK(sc.get(&d_segs, segs.size()));
    ASP_CHECK(sc.get(&d_blocks, blocks.size()));
    ASP_CHECK(sc.get(&t_idx, (size_t)nnz));
    ASP_CHECK(sc.get(&t_score, (size_t)nnz));
    ASP_CUDA(cudaMemcpyAsync(d_segs, segs.data(), sizeof(int64_t) * segs.size(), cudaMemcpyHostToDevice, st));
    ASP_CUDA(cudaMemcpyAsync(d_blocks, blocks.data(), sizeof(int64_t) * blocks.size(), cudaMemcpyHostToDevice, st));
    const size_t smem = sizeof(SKey) * SORT_S;
    ASP_CUDA(cudaFuncSetAttribute(sort_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sort_blocks_kernel<<<(unsigned)(blocks.size() / 2), 512, smem, st>>>(d_blocks, out_idx, out_score);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    int64_t longest = 0;
    for (size_t i = 1; i < segs.size(); i += 2) longest = std::max(longest, segs[i]);
    const int nseg = (int)(segs.size() / 2);
    int64_t *si = out_idx, *di = t_idx;
    double *ss = out_score, *ds = t_score;
    const unsigned gx = (unsigned)std::min<int64_t>(asp_ceil_div(longest, 256), 1024), gy = (unsigned)std::min(nseg, 65535);
    for (int64_t w = SORT_S; w < longest; w *= 2) {
        merge_pass_kernel<<<dim3(gx, gy), 256, 0, st>>>(nseg, d_segs, w, si, ss, di, ds);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
        std::swap(si, di);
        std::swap(ss, ds);
    }
    if (si != out_idx)                                          // odd number of passes: one more with a run as wide as any segment
    {
        merge_pass_kernel<<<dim3(gx, gy), 256, 0, st>>>(nseg, d_segs, longest, si, ss, di, ds);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    ASP_CUDA(cudaStreamSynchronize(st));                        // the scratch is released on return
    return ASP_OK;
}

}  // namespace

int64_t asp_range_sub_batch() { return SUB_BATCH; }

int asp_range_merge_impl(asp_ctx *ctx, int parts, int64_t nq, const int64_t *h_counts, const int64_t *idx_dev,
                         const double *score_dev, int64_t *out_idx_dev, double *out_score_dev)
{
    cudaStream_t st = ctx->stream;
    std::vector<int64_t> part_off((size_t)parts * (nq + 1)), out_off((size_t)nq + 1);
    const int64_t total = asp_range::merge_tables(parts, nq, h_counts, part_off.data(), out_off.data());
    if (total == 0) return ASP_OK;
    asp_scratch sc(st);
    int64_t *d_po = nullptr, *d_oo = nullptr;
    ASP_CHECK(sc.get(&d_po, part_off.size()));
    ASP_CHECK(sc.get(&d_oo, out_off.size()));
    ASP_CUDA(cudaMemcpyAsync(d_po, part_off.data(), sizeof(int64_t) * part_off.size(), cudaMemcpyHostToDevice, st));
    ASP_CUDA(cudaMemcpyAsync(d_oo, out_off.data(), sizeof(int64_t) * out_off.size(), cudaMemcpyHostToDevice, st));
    asp_range::range_merge_kernel<<<(unsigned)std::min<int64_t>(asp_ceil_div(total, 256), (int64_t)ctx->num_sms * 16), 256, 0, st>>>(
        total, parts, nq, d_po, d_oo, idx_dev, score_dev, out_idx_dev, out_score_dev);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaStreamSynchronize(st));
    return ASP_OK;
}

int asp_range_impl(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lam_dev, const double *norm_dev,
                   double tau, double min_score, const uint32_t *allowed_dev, int64_t max_hits, int64_t hits_before, int64_t q_base,
                   int64_t *h_counts, asp_range_result::Piece *out)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    if (nq == 0) return ASP_OK;
    // the f32 emission floor: from a value inside [-2, 2] (every score lies in [-1, 1] for tau in [0, 1]; > 1 gives empty rows)
    const double emit_floor = std::min(2.0, std::max(-2.0, min_score));
    bool use_tc = tau > 1e-3 && tau <= 1.0 && s->fp <= 6144 && s->n_local >= 1 && s->n_local < 2147483647LL;
    if (const char *e = getenv("ASP_RANGE_STAGE1")) { if (e[0] == 's') use_tc = false; }   // test knob: both routes, same bits
    asp_scratch sc(st);
    int64_t *d_counts = nullptr, *d_off = nullptr;
    int32_t *slow_list = nullptr, *slow_count = nullptr;
    ASP_CHECK(sc.get(&d_counts, nq));
    ASP_CHECK(sc.get(&d_off, nq + 1));
    ASP_CHECK(sc.get(&slow_list, nq));
    ASP_CHECK(sc.get(&slow_count, 1));
    ASP_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(int64_t) * nq, st));
    ASP_CUDA(cudaMemsetAsync(slow_count, 0, sizeof(int32_t), st));
    asp_tc_batch b;
    double *exact = nullptr;
    int nslow = 0;
    float ms1 = 0.f;
    if (use_tc) {
        ASP_CHECK(asp_tc_stage1(s, q_dev, nq, qpitch, lam_dev, norm_dev, tau, 0, emit_floor, 0, 0, nullptr, &b, false, allowed_dev));
        ASP_CHECK(sc.get(&exact, (size_t)nq * b.nsub * b.capb));
        const size_t smem = sizeof(double) * (size_t)RW * s->fp;
        ASP_CUDA(cudaFuncSetAttribute(tc_range_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc_range_count_kernel<<<(unsigned)asp_ceil_div(nq, RW), RW * 32, smem, st>>>(
            q_dev, qpitch, nq, s->items, s->f, s->fp, s->norms, s->lambdas, norm_dev, lam_dev, tau, min_score, b.nsub, b.capb,
            b.emit_ix, b.emit_cnt, b.qperm, exact, d_counts, slow_list, slow_count);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
        ASP_CUDA(cudaMemcpyAsync(&nslow, slow_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
        cudaEventElapsedTime(&ms1, ctx->ev0, ctx->ev1);
    } else {
        ASP_CUDA(cudaEventRecord(ctx->ev1, st));
        iota32_kernel<<<(unsigned)std::min<int64_t>(asp_ceil_div(nq, 256), 1024), 256, 0, st>>>(slow_list, nq);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
        nslow = (int)nq;
    }
    int nparts = (int)std::min<int64_t>(std::max<int64_t>(asp_ceil_div(s->n_local, SC_CHUNK), 1), (int64_t)ctx->num_sms * 2);
    int64_t *part_cnt = nullptr;
    if (nslow > 0) {
        ASP_CHECK(sc.get(&part_cnt, (size_t)nslow * nparts));
        ASP_CHECK(run_scan<false>(s, q_dev, qpitch, slow_list, nslow, nparts, lam_dev, norm_dev, tau, min_score, allowed_dev, part_cnt,
                                  nullptr, nullptr, nullptr));
        scan_prefix_kernel<<<(unsigned)asp_ceil_div(nslow, 128), 128, 0, st>>>(nslow, nparts, slow_list, part_cnt, d_counts);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    ASP_CUDA(cudaMemcpyAsync(h_counts, d_counts, sizeof(int64_t) * nq, cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));

    // exclusive scan into the offsets, and the cap: checked before the hits get any device memory
    std::vector<int64_t> h_off((size_t)nq + 1);
    int64_t run = 0;
    for (int64_t qi = 0; qi < nq; ++qi) {
        h_off[qi] = run;
        run += h_counts[qi];
        if (max_hits > 0 && hits_before + run > max_hits)
            ASP_FAIL(ASP_ERR_LIMIT, "range search: %lld hits reached at query %lld, more than max_hits = %lld",
                     (long long)(hits_before + run), (long long)(q_base + qi), (long long)max_hits);
    }
    h_off[nq] = run;
    ctx->stats["search_slow_queries"] += nslow;
    if (run > 0) {
        ASP_CUDA(cudaMemcpyAsync(d_off, h_off.data(), sizeof(int64_t) * (nq + 1), cudaMemcpyHostToDevice, st));
        out->mem = asp_scratch(st);                               // the hits belong to the caller's piece
        int64_t *didx = nullptr;
        double *dsc = nullptr;
        ASP_CHECK(out->mem.get(&didx, (size_t)run));
        ASP_CHECK(out->mem.get(&dsc, (size_t)run));
        out->idx = didx; out->score = dsc; out->n = run;
        if (use_tc) {
            tc_range_fill_kernel<<<(unsigned)asp_ceil_div(nq, RW), RW * 32, 0, st>>>(nq, b.nsub, b.capb, b.emit_ix, b.emit_cnt, b.qperm,
                                                                                   exact, d_off, s->row0, didx, dsc);
            ASP_CUDA(cudaGetLastError());
            ASP_LAUNCHED(ctx);
        }
        if (nslow > 0)
            ASP_CHECK(run_scan<true>(s, q_dev, qpitch, slow_list, nslow, nparts, lam_dev, norm_dev, tau, min_score, allowed_dev,
                                     part_cnt, d_off, didx, dsc));
        ASP_CHECK(sort_segments(ctx, nq, h_off.data(), d_off, run, didx, dsc));
    }
    ASP_CUDA(cudaEventRecord(ctx->ev2, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    float ms2 = 0.f;
    cudaEventElapsedTime(&ms2, ctx->ev1, ctx->ev2);
    ctx->stats["range_stage1_ms"] += use_tc ? ms1 : 0.0;
    ctx->stats["range_stage2_ms"] += ms2;
    ctx->stats["range_stage1_is_tc"] = use_tc ? 1.0 : 0.0;
    return ASP_OK;
}
