// reduce.cu -- pre-graph reduction (SURVEY.md 8(f)-1; include/arrowspace_b200.h R1-R4): what the crate runs inside
// ArrowSpaceBuilder::build before graph construction (with_dims_reduction / with_seed, /root/reference/src/lib.rs:282-283;
// log evidence tests/output/1760705545_v0_16/suggested_eps.md:3-11).  Sampling is a counter-based hash (host), the two-NN
// intrinsic-dimension estimate and the k-means assignment share ONE kernel: squared Euclidean distances of a set of A rows
// against a set of B rows in the oracle's order (left to right over the features, difference, product rounded, then added),
// keeping the two smallest (distance, position) per A row.  The centroid update sums the member rows in ascending row order,
// so the centroids are bit-identical to the oracle's (oracle/oracle.c orc_reduce).
//
// Bound: FP64 FMA pipe (3 DP instructions per pair and feature, no FMA contraction allowed by the parity contract);
// algorithmic work per assignment pass 3 * |S| * K * f DP operations, bytes 8 * |S| * f (rows read once per pass; the K x f
// centroid tile is re-read from L2 by every CTA).
#include "common.cuh"

#include <math.h>
#include <limits.h>

namespace {

constexpr int RD_TA = 32;        // A rows per CTA
constexpr int RD_FC = 16;        // features per staged chunk
constexpr int RD_THREADS = 256;  // 8 warps: warp w owns A rows 4w .. 4w+3, lane l owns B rows l + 32 j

struct Min2 {
    double d1, d2;
    int32_t i1, i2;
};

__device__ __forceinline__ bool lex_less(double da, int32_t ia, double db, int32_t ib)
{
    return da < db || (da == db && ia < ib);
}

__device__ __forceinline__ void min2_init(Min2 &m)
{
    m.d1 = m.d2 = __longlong_as_double(0x7ff0000000000000LL);
    m.i1 = m.i2 = INT_MAX;
}

__device__ __forceinline__ void min2_insert(Min2 &m, double d, int32_t i)
{
    if (lex_less(d, i, m.d1, m.i1)) {
        m.d2 = m.d1; m.i2 = m.i1;
        m.d1 = d; m.i1 = i;
    } else if (lex_less(d, i, m.d2, m.i2)) {
        m.d2 = d; m.i2 = i;
    }
}

// out_d / out_i: [split][na][2].  excl[a] = B position that A row a must not match (itself), or nullptr.
template <int JB>
__global__ void __launch_bounds__(RD_THREADS)
sqdist_min2_kernel(const double *__restrict__ XA, int pitchA, const int32_t *__restrict__ a_rows, int64_t na,
                   const double *__restrict__ XB, int pitchB, const int32_t *__restrict__ b_rows, int64_t nb,
                   int64_t b_per_split, const int32_t *__restrict__ excl, int fp, double *__restrict__ out_d,
                   int32_t *__restrict__ out_i)
{
    constexpr int TB = 32 * JB;
    __shared__ double As[RD_FC][RD_TA + 1];
    __shared__ double Bs[RD_FC][TB + 1];
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int64_t a0 = (int64_t)blockIdx.x * RD_TA;
    const int64_t b_begin = (int64_t)blockIdx.y * b_per_split;
    const int64_t b_end = min(nb, b_begin + b_per_split);

    Min2 best[4];
    int32_t ex[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        min2_init(best[r]);
        const int64_t a = a0 + ty * 4 + r;
        ex[r] = (excl && a < na) ? excl[a] : -1;
    }
    // staging roles: 8 threads per row (one double2 each), 32 rows per pass
    const int lrow = tid >> 3, lq = tid & 7;
    const int64_t la = a0 + lrow;
    const double *a_src = nullptr;
    if (la < na) a_src = XA + (size_t)(a_rows ? a_rows[la] : la) * pitchA;

    for (int64_t bt = b_begin; bt < b_end; bt += TB) {
        const double *b_src[JB];
#pragma unroll
        for (int j = 0; j < JB; ++j) {
            const int64_t b = bt + lrow + 32 * j;
            b_src[j] = (b < b_end) ? XB + (size_t)(b_rows ? b_rows[b] : b) * pitchB : nullptr;
        }
        double acc[4][JB];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int j = 0; j < JB; ++j) acc[r][j] = 0.0;

        for (int f0 = 0; f0 < fp; f0 += RD_FC) {
            const int fo = f0 + 2 * lq;
            double2 va = make_double2(0.0, 0.0);
            if (a_src && fo < fp) va = *reinterpret_cast<const double2 *>(a_src + fo);
            double2 vb[JB];
#pragma unroll
            for (int j = 0; j < JB; ++j) {
                vb[j] = make_double2(0.0, 0.0);
                if (b_src[j] && fo < fp) vb[j] = *reinterpret_cast<const double2 *>(b_src[j] + fo);
            }
            __syncthreads();                      // the previous chunk has been consumed
            As[2 * lq][lrow] = va.x;
            As[2 * lq + 1][lrow] = va.y;
#pragma unroll
            for (int j = 0; j < JB; ++j) {
                Bs[2 * lq][lrow + 32 * j] = vb[j].x;
                Bs[2 * lq + 1][lrow + 32 * j] = vb[j].y;
            }
            __syncthreads();
#pragma unroll
            for (int fi = 0; fi < RD_FC; ++fi) {
                double a[4], b[JB];
#pragma unroll
                for (int r = 0; r < 4; ++r) a[r] = As[fi][ty * 4 + r];
#pragma unroll
                for (int j = 0; j < JB; ++j) b[j] = Bs[fi][tx + 32 * j];
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int j = 0; j < JB; ++j) {
                        const double d = __dsub_rn(a[r], b[j]);
                        acc[r][j] = __dadd_rn(acc[r][j], __dmul_rn(d, d));
                    }
            }
        }
        // the two smallest of this tile per A row: own columns, then a butterfly over the lanes
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            Min2 loc;
            min2_init(loc);
#pragma unroll
            for (int j = 0; j < JB; ++j) {
                const int64_t b = bt + tx + 32 * j;
                if (b < b_end && (int32_t)b != ex[r]) min2_insert(loc, acc[r][j], (int32_t)b);
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const double od1 = __shfl_xor_sync(0xffffffffu, loc.d1, off), od2 = __shfl_xor_sync(0xffffffffu, loc.d2, off);
                const int32_t oi1 = __shfl_xor_sync(0xffffffffu, loc.i1, off), oi2 = __shfl_xor_sync(0xffffffffu, loc.i2, off);
                min2_insert(loc, od1, oi1);
                min2_insert(loc, od2, oi2);
            }
            min2_insert(best[r], loc.d1, loc.i1);
            min2_insert(best[r], loc.d2, loc.i2);
        }
    }
    if (tx == 0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int64_t a = a0 + ty * 4 + r;
            if (a < na) {
                const size_t o = ((size_t)blockIdx.y * na + a) * 2;
                out_d[o] = best[r].d1; out_d[o + 1] = best[r].d2;
                out_i[o] = best[r].i1; out_i[o + 1] = best[r].i2;
            }
        }
    }
}

__global__ void min2_merge_splits_kernel(const double *__restrict__ part_d, const int32_t *__restrict__ part_i, int nsplit,
                                         int64_t na, double *__restrict__ out_d, int32_t *__restrict__ out_i)
{
    const int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (a >= na) return;
    Min2 m;
    min2_init(m);
    for (int s = 0; s < nsplit; ++s) {
        const size_t o = ((size_t)s * na + a) * 2;
        min2_insert(m, part_d[o], part_i[o]);
        min2_insert(m, part_d[o + 1], part_i[o + 1]);
    }
    out_d[2 * a] = m.d1; out_d[2 * a + 1] = m.d2;
    out_i[2 * a] = m.i1; out_i[2 * a + 1] = m.i2;
}

__global__ void assign_commit_kernel(const int32_t *__restrict__ best_i, int64_t na, int32_t *__restrict__ assign,
                                     int32_t *__restrict__ changed)
{
    const int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int ch = 0;
    if (a < na) {
        const int32_t nw = best_i[2 * a];
        ch = nw != assign[a];
        assign[a] = nw;
    }
    const int tot = __syncthreads_count(ch);
    if (threadIdx.x == 0 && tot) atomicAdd(changed, tot);
}

__global__ void init_centroids_kernel(const double *__restrict__ X, int pitch, const int32_t *__restrict__ s_rows, int64_t ns,
                                      int K, double *__restrict__ C, int fp)
{
    const int j = blockIdx.x;
    const int64_t pos = ((int64_t)j * ns) / K;
    const double *src = X + (size_t)(s_rows ? s_rows[pos] : pos) * pitch;
    for (int t = threadIdx.x; t < fp; t += blockDim.x) C[(size_t)j * fp + t] = src[t];
}

// One CTA per (centroid, 512-column group): walks the assignments in position order, compacts the members of its centroid
// in order into shared memory and adds their rows one after the other (the oracle's summation order).
constexpr int UP_THREADS = 128, UP_TILE = 1024, UP_COLS = 4;
__global__ void __launch_bounds__(UP_THREADS)
centroid_update_kernel(const double *__restrict__ X, int pitch, const int32_t *__restrict__ s_rows, int64_t ns,
                       const int32_t *__restrict__ assign, double *__restrict__ C, int fp, int32_t *__restrict__ counts)
{
    __shared__ int32_t list[UP_TILE];
    __shared__ int warp_tot[UP_THREADS / 32];
    const int c = blockIdx.x, t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int col0 = blockIdx.y * (UP_THREADS * UP_COLS) + t;
    double sum[UP_COLS];
#pragma unroll
    for (int u = 0; u < UP_COLS; ++u) sum[u] = 0.0;
    int64_t count = 0;
    for (int64_t tile = 0; tile < ns; tile += UP_TILE) {
        const int64_t p0 = tile + (int64_t)t * 8;
        int32_t a[8];
        if (p0 + 8 <= ns) {
            const int4 v0 = *reinterpret_cast<const int4 *>(assign + p0), v1 = *reinterpret_cast<const int4 *>(assign + p0 + 4);
            a[0] = v0.x; a[1] = v0.y; a[2] = v0.z; a[3] = v0.w; a[4] = v1.x; a[5] = v1.y; a[6] = v1.z; a[7] = v1.w;
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) a[e] = (p0 + e < ns) ? assign[p0 + e] : -1;
        }
        int mine = 0;
#pragma unroll
        for (int e = 0; e < 8; ++e) mine += a[e] == c;
        int incl = mine;                                   // inclusive scan over the warp, then over the 4 warps
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += v;
        }
        __syncthreads();                                   // the previous tile's list has been consumed
        if (lane == 31) warp_tot[w] = incl;
        __syncthreads();
        int base = 0, total = 0;
#pragma unroll
        for (int k = 0; k < UP_THREADS / 32; ++k) {
            if (k < w) base += warp_tot[k];
            total += warp_tot[k];
        }
        int o = base + incl - mine;
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (a[e] == c) list[o++] = s_rows ? s_rows[p0 + e] : (int32_t)(p0 + e);
        __syncthreads();
        count += total;
        int m = 0;
        for (; m + 4 <= total; m += 4) {                   // four rows in flight, added in order
            double v[4][UP_COLS];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double *row = X + (size_t)list[m + q] * pitch;
#pragma unroll
                for (int u = 0; u < UP_COLS; ++u) {
                    const int col = col0 + u * UP_THREADS;
                    v[q][u] = col < fp ? row[col] : 0.0;
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int u = 0; u < UP_COLS; ++u) sum[u] = __dadd_rn(sum[u], v[q][u]);
        }
        for (; m < total; ++m) {
            const double *row = X + (size_t)list[m] * pitch;
#pragma unroll
            for (int u = 0; u < UP_COLS; ++u) {
                const int col = col0 + u * UP_THREADS;
                if (col < fp) sum[u] = __dadd_rn(sum[u], row[col]);
            }
        }
    }
    if (count > 0) {
        const double cnt = (double)count;
#pragma unroll
        for (int u = 0; u < UP_COLS; ++u) {
            const int col = col0 + u * UP_THREADS;
            if (col < fp) C[(size_t)c * fp + col] = __ddiv_rn(sum[u], cnt);
        }
    }
    if (counts && blockIdx.y == 0 && t == 0) counts[c] = (int32_t)min((int64_t)INT_MAX, count);
}

uint64_t splitmix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

template <int JB>
void launch_min2(cudaStream_t st, dim3 grid, const double *XA, int pitchA, const int32_t *a_rows, int64_t na, const double *XB,
                 int pitchB, const int32_t *b_rows, int64_t nb, int64_t per, const int32_t *excl, int fp, double *od, int32_t *oi)
{
    sqdist_min2_kernel<JB><<<grid, RD_THREADS, 0, st>>>(XA, pitchA, a_rows, na, XB, pitchB, b_rows, nb, per, excl, fp, od, oi);
}

// two smallest (squared distance, B position) of every A row over all B rows -> fin_d / fin_i [na][2] (device)
int min2_all(asp_ctx *ctx, const double *XA, int pitchA, const int32_t *a_rows, int64_t na, const double *XB, int pitchB,
             const int32_t *b_rows, int64_t nb, const int32_t *excl, int fp, double *fin_d, int32_t *fin_i)
{
    int jb = 4;                                           // B tile = 32 * jb rows: least padding, larger tile on ties
    {
        int64_t best = -1;
        for (int c : {4, 2, 1}) {
            const int64_t padded = asp_ceil_div(nb, 32 * c) * 32 * c;
            if (best < 0 || padded < best) { best = padded; jb = c; }
        }
    }
    const int tb = 32 * jb;
    const int64_t a_tiles = asp_ceil_div(na, RD_TA);
    int64_t nsplit = 1;
    if (a_tiles < 2 * ctx->num_sms) {
        nsplit = std::min<int64_t>((2 * ctx->num_sms) / a_tiles, asp_ceil_div(nb, (int64_t)tb * 8));
        if (nsplit < 1) nsplit = 1;
    }
    if (a_tiles > 2147483647LL || nsplit > 65535) ASP_FAIL(ASP_ERR_UNSUPPORTED, "reduction: too many rows for one launch");
    const int64_t per = asp_ceil_div(asp_ceil_div(nb, nsplit), tb) * tb;
    nsplit = asp_ceil_div(nb, per);
    asp_scratch sc(ctx->stream);
    double *pd = fin_d;
    int32_t *pi = fin_i;
    if (nsplit > 1) {
        ASP_CHECK(sc.get(&pd, 2 * (size_t)na * nsplit));
        ASP_CHECK(sc.get(&pi, 2 * (size_t)na * nsplit));
    }
    const dim3 grid((unsigned)a_tiles, (unsigned)nsplit);
    if (jb == 4) launch_min2<4>(ctx->stream, grid, XA, pitchA, a_rows, na, XB, pitchB, b_rows, nb, per, excl, fp, pd, pi);
    else if (jb == 2) launch_min2<2>(ctx->stream, grid, XA, pitchA, a_rows, na, XB, pitchB, b_rows, nb, per, excl, fp, pd, pi);
    else launch_min2<1>(ctx->stream, grid, XA, pitchA, a_rows, na, XB, pitchB, b_rows, nb, per, excl, fp, pd, pi);
    ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaGetLastError());
    if (nsplit > 1) {
        min2_merge_splits_kernel<<<(unsigned)asp_ceil_div(na, 256), 256, 0, ctx->stream>>>(pd, pi, (int)nsplit, na, fin_d, fin_i);
        ASP_LAUNCHED(ctx);
        ASP_CUDA(cudaGetLastError());
    }
    return ASP_OK;
}

}  // namespace

extern "C" {

void asp_default_reduction(asp_reduction *red)
{
    if (!red) return;
    red->sample_rate = 0.6;
    red->seed = 42;
    red->n_clusters = 0;
    red->max_iters = 10;
    red->probes = 2048;
    red->reserved = 0;
}

int asp_reduction_sample(const asp_reduction *red, int64_t row0, int64_t n_local, int32_t *out_rows, int64_t *out_count)
{
    if (!red || !out_rows || !out_count || n_local < 0 || row0 < 0) ASP_FAIL(ASP_ERR_ARG, "asp_reduction_sample: bad argument");
    if (n_local > INT_MAX) ASP_FAIL(ASP_ERR_UNSUPPORTED, "asp_reduction_sample: more than 2^31 - 1 rows in one shard");
    int64_t cnt = 0;
    if (!(red->sample_rate < 1.0)) {
        for (int64_t i = 0; i < n_local; ++i) out_rows[cnt++] = (int32_t)i;
    } else {
        for (int64_t i = 0; i < n_local; ++i) {
            const uint64_t z = splitmix64(red->seed + (uint64_t)(row0 + i + 1) * 0x9E3779B97F4A7C15ULL);
            const double u = (double)(z >> 11) * (1.0 / 9007199254740992.0);
            if (u < red->sample_rate) out_rows[cnt++] = (int32_t)i;
        }
    }
    *out_count = cnt;
    return ASP_OK;
}

int asp_space_reduce(asp_space *s, const asp_reduction *red_in, int64_t n_total_for_k, asp_reduction_info *info,
                     asp_space **out_centroids)
{
    if (!s || !out_centroids) ASP_FAIL(ASP_ERR_ARG, "asp_space_reduce: NULL argument");
    if (s->world != 1) ASP_FAIL(ASP_ERR_UNSUPPORTED, "asp_space_reduce: needs a world-1 space (gather the sampled rows first)");
    if (s->n_local > INT_MAX) ASP_FAIL(ASP_ERR_UNSUPPORTED, "asp_space_reduce: more than 2^31 - 1 rows");
    asp_reduction red;
    if (red_in) red = *red_in; else asp_default_reduction(&red);
    if (!(red.sample_rate > 0.0) || red.max_iters < 0 || red.n_clusters < 0 || red.probes < 0)
        ASP_FAIL(ASP_ERR_ARG, "asp_space_reduce: sample_rate must be > 0, n_clusters / max_iters / probes >= 0");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    asp_scratch scratch(st);
    const int fp = s->fp;
    const int64_t n = s->n_local;

    // R1
    std::vector<int32_t> h_rows;
    int64_t ns = n;
    int32_t *d_rows = nullptr;                            // nullptr = every row
    if (red.sample_rate < 1.0) {
        h_rows.resize((size_t)n);
        ASP_CHECK(asp_reduction_sample(&red, s->row0, n, h_rows.data(), &ns));
        if (ns == 0) ns = n;                              // an empty sample keeps every row
        else if (ns < n) {
            h_rows.resize((size_t)ns);
            ASP_CHECK(scratch.get(&d_rows, (size_t)ns));
            ASP_CUDA(cudaMemcpyAsync(d_rows, h_rows.data(), sizeof(int32_t) * ns, cudaMemcpyHostToDevice, st));
        }
    }
    asp_reduction_info inf;
    inf.n_sampled = ns;
    inf.n_probes = 0;
    inf.two_nn_mean_ratio = NAN;
    inf.intrinsic_dim = 0;
    inf.iters = 0;
    inf.converged = 0;

    // R2
    cudaEvent_t e0, e1;
    ASP_CUDA(cudaEventCreate(&e0));
    ASP_CUDA(cudaEventCreate(&e1));
    struct EvGuard { cudaEvent_t a, b; ~EvGuard() { cudaEventDestroy(a); cudaEventDestroy(b); } } evg{e0, e1};
    ctx->stats["reduce_two_nn_ms"] = 0.0;
    if (red.probes > 0 && ns >= 3) {
        const int64_t P = std::min<int64_t>(red.probes, ns);
        std::vector<int32_t> pos((size_t)P), arow((size_t)P);
        for (int64_t j = 0; j < P; ++j) {
            pos[j] = (int32_t)((j * ns) / P);
            arow[j] = d_rows ? h_rows[pos[j]] : pos[j];
        }
        int32_t *d_pos = nullptr, *d_arow = nullptr, *fi = nullptr;
        double *fd = nullptr;
        ASP_CHECK(scratch.get(&d_pos, (size_t)P));
        ASP_CHECK(scratch.get(&d_arow, (size_t)P));
        ASP_CHECK(scratch.get(&fd, (size_t)2 * P));
        ASP_CHECK(scratch.get(&fi, (size_t)2 * P));
        ASP_CUDA(cudaMemcpyAsync(d_pos, pos.data(), sizeof(int32_t) * P, cudaMemcpyHostToDevice, st));
        ASP_CUDA(cudaMemcpyAsync(d_arow, arow.data(), sizeof(int32_t) * P, cudaMemcpyHostToDevice, st));
        ASP_CUDA(cudaEventRecord(e0, st));
        ASP_CHECK(min2_all(ctx, s->items, fp, d_arow, P, s->items, fp, d_rows, ns, d_pos, fp, fd, fi));
        ASP_CUDA(cudaEventRecord(e1, st));
        std::vector<double> hd((size_t)2 * P);
        ASP_CUDA(cudaMemcpyAsync(hd.data(), fd, sizeof(double) * 2 * P, cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        ctx->stats["reduce_two_nn_ms"] = ms;
        double acc = 0.0;
        int64_t used = 0;
        for (int64_t j = 0; j < P; ++j) {
            const double r1 = sqrt(hd[2 * j]), r2 = sqrt(hd[2 * j + 1]);
            if (!(r1 > 0.0) || !std::isfinite(r2)) continue;
            acc += r2 / r1;
            ++used;
        }
        inf.n_probes = used;
        if (used > 0) {
            const double m = acc / (double)used;
            inf.two_nn_mean_ratio = m;
            double d = (m > 1.0) ? m / (m - 1.0) : (double)s->f;
            if (!(d < (double)s->f)) d = (double)s->f;
            inf.intrinsic_dim = d < 1.0 ? 1 : (int32_t)d;
        }
    }

    // R3
    int64_t K = red.n_clusters;
    if (K <= 0) {
        const int64_t N = n_total_for_k > 0 ? n_total_for_k : s->n_total;
        K = (int64_t)ceil(sqrt((double)N / 10.0));
    }
    if (K > ns) K = ns;
    if (K < 1) K = 1;
    if (K > 65535) ASP_FAIL(ASP_ERR_UNSUPPORTED, "reduction: at most 65535 clusters (got %lld)", (long long)K);
    inf.n_clusters = (int32_t)K;

    // R4
    double *C = nullptr, *bd = nullptr;
    int32_t *bi = nullptr, *assign = nullptr, *changed = nullptr;
    ASP_CHECK(scratch.get(&C, (size_t)K * fp));
    ASP_CHECK(scratch.get(&bd, (size_t)2 * ns));
    ASP_CHECK(scratch.get(&bi, (size_t)2 * ns));
    ASP_CHECK(scratch.get(&assign, (size_t)ns));
    ASP_CHECK(scratch.get(&changed, 1));
    ASP_CUDA(cudaMemsetAsync(assign, 0xff, sizeof(int32_t) * ns, st));
    init_centroids_kernel<<<(unsigned)K, 128, 0, st>>>(s->items, fp, d_rows, ns, (int)K, C, fp);
    ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaGetLastError());
    ASP_CUDA(cudaEventRecord(e0, st));
    double assign_ms = 0.0;
    int passes = 0;
    for (int it = 0; it < red.max_iters; ++it) {
        cudaEvent_t a0, a1;
        ASP_CUDA(cudaEventCreate(&a0));
        ASP_CUDA(cudaEventCreate(&a1));
        EvGuard ag{a0, a1};
        ASP_CUDA(cudaMemsetAsync(changed, 0, sizeof(int32_t), st));
        ASP_CUDA(cudaEventRecord(a0, st));
        ASP_CHECK(min2_all(ctx, s->items, fp, d_rows, ns, C, fp, nullptr, K, nullptr, fp, bd, bi));
        ASP_CUDA(cudaEventRecord(a1, st));
        assign_commit_kernel<<<(unsigned)asp_ceil_div(ns, 256), 256, 0, st>>>(bi, ns, assign, changed);
        ASP_LAUNCHED(ctx);
        int32_t h_changed = 0;
        ASP_CUDA(cudaMemcpyAsync(&h_changed, changed, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a0, a1);
        assign_ms += ms;
        ++passes;
        if (h_changed == 0) { inf.converged = 1; break; }
        const dim3 ug((unsigned)K, (unsigned)asp_ceil_div(fp, UP_THREADS * UP_COLS));
        centroid_update_kernel<<<ug, UP_THREADS, 0, st>>>(s->items, fp, d_rows, ns, assign, C, fp, nullptr);
        ASP_LAUNCHED(ctx);
        ASP_CUDA(cudaGetLastError());
        inf.iters = it + 1;
    }
    ASP_CUDA(cudaEventRecord(e1, st));
    ASP_CUDA(cudaEventSynchronize(e1));
    {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        ctx->stats["reduce_kmeans_ms"] = ms;
        ctx->stats["reduce_assign_ms"] = assign_ms;
        ctx->stats["reduce_assign_passes"] = (double)passes;
    }

    // the centroids as a space of their own (dense copy: asp_space_create re-pitches)
    double *dense = C;
    if (fp != s->f) {
        ASP_CHECK(scratch.get(&dense, (size_t)K * s->f));
        ASP_CUDA(cudaMemcpy2DAsync(dense, sizeof(double) * s->f, C, sizeof(double) * fp, sizeof(double) * s->f, (size_t)K,
                                   cudaMemcpyDeviceToDevice, st));
    }
    ASP_CHECK(asp_space_create(ctx, dense, K, s->f, K, 1, 0, out_centroids));
    if (info) *info = inf;
    return ASP_OK;
}

}  // extern "C"
