// csr.cu -- K2: graph Laplacian CSR assembly by scan / compaction / segmented sort
// (GRAPH_VARIABLES.md:3,8-9; SURVEY.md Appendix A5-A7; crate call site /root/reference/src/lib.rs:289).
//
// Input: per-node neighbour lists (index, distance), <= kk per node.  Output: L = D - W with
// W = max(W, W^T), CSR with ascending columns and the diagonal stored.
// Bound: HBM, ~60*M*k bytes (SURVEY.md 8(d) K2): lists in, mirrored edges, CSR out.
//
//   1. weights_compact   w = 1/(1+(d/sigma)^p) | exp(-(d/sigma)^p); drop w == 0; compact each list
//  1b. symmetrise rule   (asp_switches.symmetrise, UNPINNED): max = union (default) | avg: a one-sided edge weighs w/2 in both
//                        directions | min: one-sided edges are dropped | none: the directed lists are the graph
//   2. count_mirror      for edge a->b: is a in list(b)?  if not, row b grows by one (atomic count)
//   3. exclusive scan    row lengths (own + mirrored + diagonal) -> indptr   (3-kernel block scan)
//   4. fill              own edges at their slot, mirrored edges through an atomic cursor
//   5. sort_rows         segmented sort by column (warp bitonic <= 64, block bitonic otherwise),
//                        degree = sum of weights in ascending column order, values -> -w, diag -> deg
//   6. normalise         (asp_switches.laplacian, UNPINNED): sym  L_ab = -w_ab / sqrt(deg_a deg_b), L_aa = [deg_a > 0]
//                        rw   L_ab = -w_ab / deg_a; entries towards a node of degree 0 become explicit zeros
// The atomics only decide slots inside a row; the sort makes the result deterministic.
#include "common.cuh"

#include <math.h>

namespace {

__device__ __forceinline__ double edge_weight(double d, double sigma, double p, int kernel)
{
    const double r = d / sigma;
    double t;
    if (p == 2.0) t = r * r;           // every reference config uses p = 2 (tests/test_0.py:16, README.md:46)
    else if (p == 1.0) t = r;
    else t = pow(r, p);
    return kernel == ASP_KERNEL_GAUSSIAN ? exp(-t) : 1.0 / (1.0 + t);
}

__global__ void weights_compact_kernel(int64_t m, int kk, int32_t *idx, double *val, int32_t *cnt, double sigma,
                                       double p, int kernel)
{
    for (int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; a < m; a += (int64_t)gridDim.x * blockDim.x) {
        const int c = cnt[a];
        int o = 0;
        for (int j = 0; j < c; ++j) {
            const double w = edge_weight(val[a * kk + j], sigma, p, kernel);
            const int32_t b = idx[a * kk + j];
            if (w > 0.0) { idx[a * kk + o] = b; val[a * kk + o] = w; ++o; }
        }
        cnt[a] = o;
    }
}

__device__ __forceinline__ bool list_contains(const int32_t *idx, int kk, const int32_t *cnt, int64_t row, int32_t v)
{
    const int c = cnt[row];
    for (int j = 0; j < c; ++j)
        if (idx[row * kk + j] == v) return true;
    return false;
}

// one-sided edges (a -> b with a not in list(b)): halved (avg) or marked dead with a negative weight (min)
__global__ void symmetrise_mark_kernel(int64_t m, int kk, const int32_t *idx, double *val, const int32_t *cnt, int mode)
{
    const int64_t total = m * kk;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = e / kk;
        if ((int)(e % kk) >= cnt[a]) continue;
        if (list_contains(idx, kk, cnt, idx[e], (int32_t)a)) continue;
        val[e] = (mode == ASP_SYM_AVG) ? 0.5 * val[e] : -1.0;
    }
}

__global__ void drop_marked_kernel(int64_t m, int kk, int32_t *idx, double *val, int32_t *cnt)
{
    for (int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; a < m; a += (int64_t)gridDim.x * blockDim.x) {
        const int c = cnt[a];
        int o = 0;
        for (int j = 0; j < c; ++j) {
            const double w = val[a * kk + j];
            const int32_t b = idx[a * kk + j];
            if (w >= 0.0) { idx[a * kk + o] = b; val[a * kk + o] = w; ++o; }
        }
        cnt[a] = o;
    }
}

__global__ void count_mirror_kernel(int64_t m, int kk, const int32_t *idx, const int32_t *cnt, int32_t *extra)
{
    const int64_t total = m * kk;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = e / kk;
        const int j = (int)(e % kk);
        if (j >= cnt[a]) continue;
        const int32_t b = idx[e];
        if (!list_contains(idx, kk, cnt, b, (int32_t)a)) atomicAdd(&extra[b], 1);
    }
}

// ---- exclusive scan of (cnt + extra + 1) into int64 indptr: block scan, scan of block sums, add
constexpr int SCAN_BLOCK = 1024;

__global__ void scan_blocks_kernel(int64_t m, const int32_t *cnt, const int32_t *extra, int64_t *indptr,
                                   int64_t *block_sums)
{
    __shared__ int64_t sh[SCAN_BLOCK];
    const int64_t i = blockIdx.x * (int64_t)SCAN_BLOCK + threadIdx.x;
    const int64_t v = (i < m) ? (int64_t)cnt[i] + extra[i] + 1 : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int off = 1; off < SCAN_BLOCK; off <<= 1) {
        const int64_t t = (threadIdx.x >= off) ? sh[threadIdx.x - off] : 0;
        __syncthreads();
        sh[threadIdx.x] += t;
        __syncthreads();
    }
    if (i < m) indptr[i] = sh[threadIdx.x] - v;          // exclusive, block-local
    if (threadIdx.x == SCAN_BLOCK - 1) block_sums[blockIdx.x] = sh[threadIdx.x];
}

__global__ void scan_sums_kernel(int64_t nblocks, int64_t *block_sums, int64_t *total)
{
    // single block: sequential chunks of SCAN_BLOCK with a running carry
    __shared__ int64_t sh[SCAN_BLOCK];
    __shared__ int64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nblocks; base += SCAN_BLOCK) {
        const int64_t i = base + threadIdx.x;
        const int64_t v = (i < nblocks) ? block_sums[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int off = 1; off < SCAN_BLOCK; off <<= 1) {
            const int64_t t = (threadIdx.x >= off) ? sh[threadIdx.x - off] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nblocks) block_sums[i] = carry + sh[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == SCAN_BLOCK - 1) carry += sh[threadIdx.x];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void scan_add_kernel(int64_t m, int64_t *indptr, const int64_t *block_sums, const int64_t *total)
{
    const int64_t i = blockIdx.x * (int64_t)SCAN_BLOCK + threadIdx.x;
    if (i < m) indptr[i] += block_sums[blockIdx.x];
    if (i == 0) indptr[m] = *total;
}

__global__ void fill_kernel(int64_t m, int kk, const int32_t *idx, const double *val, const int32_t *cnt,
                            const int64_t *indptr, int32_t *cursor, int32_t *col, double *data, int mirror)
{
    const int64_t total = m * kk;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = e / kk;
        const int j = (int)(e % kk);
        if (j == 0) {                                       // diagonal placeholder in the last slot of row a
            const int64_t last = indptr[a + 1] - 1;
            col[last] = (int32_t)a;
            data[last] = 0.0;
        }
        if (j >= cnt[a]) continue;
        const int32_t b = idx[e];
        const double w = val[e];
        col[indptr[a] + j] = b;
        data[indptr[a] + j] = w;
        if (mirror && !list_contains(idx, kk, cnt, b, (int32_t)a)) {
            const int slot = atomicAdd(&cursor[b], 1);
            const int64_t pos = indptr[b] + cnt[b] + slot;
            col[pos] = (int32_t)a;
            data[pos] = w;
        }
    }
}

struct Ent { int32_t c; double w; };
__device__ __forceinline__ bool ent_less(const Ent &x, const Ent &y) { return x.c < y.c; }

// rows of length <= 64: one warp per row, two entries per lane, bitonic network through shuffles
__global__ void sort_rows_warp_kernel(int64_t m, const int64_t *indptr, int32_t *col, double *data, int64_t *long_rows,
                                      int32_t *long_count)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t a = warp; a < m; a += nwarps) {
        const int64_t beg = indptr[a];
        const int len = (int)(indptr[a + 1] - beg);
        if (len > 64) {
            if (lane == 0) long_rows[atomicAdd(long_count, 1)] = a;
            continue;
        }
        Ent e[2];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int i = lane + 32 * t;                       // element position i
            e[t].c = (i < len) ? col[beg + i] : 0x7fffffff;
            e[t].w = (i < len) ? data[beg + i] : 0.0;
        }
        // bitonic sort of 64 elements, element i = lane + 32*t
        for (int size = 2; size <= 64; size <<= 1) {
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                if (stride == 32) {
                    const bool asc = true;                     // size == 64: single ascending block
                    if (ent_less(e[1], e[0]) == asc) { Ent tmp = e[0]; e[0] = e[1]; e[1] = tmp; }
                } else {
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        const int i = lane + 32 * t;
                        Ent o;
                        o.c = __shfl_xor_sync(0xffffffffu, e[t].c, stride);
                        o.w = __shfl_xor_sync(0xffffffffu, e[t].w, stride);
                        const bool asc = ((i & size) == 0);
                        const bool lower = ((i & stride) == 0);
                        // lower keeps min when ascending, max when descending
                        const bool take_min = (lower == asc);
                        const bool o_less = ent_less(o, e[t]);
                        const bool e_less = ent_less(e[t], o);
                        if (take_min ? o_less : e_less) e[t] = o;
                    }
                }
            }
        }
        // degree: weights in ascending column order, diagonal excluded (its placeholder weight is 0)
        double deg = 0.0;
        for (int i = 0; i < len; ++i) {
            const double w = __shfl_sync(0xffffffffu, (i < 32) ? e[0].w : e[1].w, i & 31);
            deg += w;
        }
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int i = lane + 32 * t;
            if (i < len) {
                col[beg + i] = e[t].c;
                data[beg + i] = (e[t].c == (int32_t)a) ? deg : -e[t].w;
            }
        }
    }
}

// longer rows: one block per row, bitonic sort in global memory (rare: hub nodes)
__global__ void sort_rows_block_kernel(const int64_t *long_rows, const int32_t *long_count, const int64_t *indptr,
                                       int32_t *col, double *data, int32_t *scratch_col, double *scratch_w)
{
    const int nlong = *long_count;
    for (int r = blockIdx.x; r < nlong; r += gridDim.x) {
        const int64_t a = long_rows[r];
        const int64_t beg = indptr[a];
        const int64_t len = indptr[a + 1] - beg;
        int64_t p2 = 1;
        while (p2 < len) p2 <<= 1;
        int32_t *sc = scratch_col + 2 * beg;            // 2x row length is >= p2
        double *sw = scratch_w + 2 * beg;
        for (int64_t i = threadIdx.x; i < p2; i += blockDim.x) {
            sc[i] = (i < len) ? col[beg + i] : 0x7fffffff;
            sw[i] = (i < len) ? data[beg + i] : 0.0;
        }
        for (int64_t size = 2; size <= p2; size <<= 1)
            for (int64_t stride = size >> 1; stride > 0; stride >>= 1) {
                __syncthreads();
                for (int64_t i = threadIdx.x; i < p2 / 2; i += blockDim.x) {
                    const int64_t lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                    const bool asc = ((lo & size) == 0);
                    const int32_t ca = sc[lo], cb = sc[hi];
                    if (asc ? (cb < ca) : (ca < cb)) {
                        sc[lo] = cb; sc[hi] = ca;
                        const double t = sw[lo]; sw[lo] = sw[hi]; sw[hi] = t;
                    }
                }
            }
        __syncthreads();
        __shared__ double s_deg;
        if (threadIdx.x == 0) {
            double deg = 0.0;
            for (int64_t i = 0; i < len; ++i) deg += sw[i];
            s_deg = deg;
        }
        __syncthreads();
        for (int64_t i = threadIdx.x; i < len; i += blockDim.x) {
            col[beg + i] = sc[i];
            data[beg + i] = (sc[i] == (int32_t)a) ? s_deg : -sw[i];
        }
        __syncthreads();
    }
}

__global__ void extract_degree_kernel(int64_t m, const int64_t *indptr, const int32_t *col, const double *data, double *deg)
{
    for (int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; a < m; a += (int64_t)gridDim.x * blockDim.x)
        for (int64_t j = indptr[a]; j < indptr[a + 1]; ++j)
            if (col[j] == (int32_t)a) deg[a] = data[j];
}

// one warp per row: the row's entries are rewritten from the degrees of both endpoints (oracle.c normalise_laplacian)
__global__ void normalise_kernel(int64_t m, const int64_t *indptr, const int32_t *col, double *data, const double *deg, int mode)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t a = warp; a < m; a += nwarps) {
        const double da = deg[a];
        for (int64_t j = indptr[a] + lane; j < indptr[a + 1]; j += 32) {
            const int32_t b = col[j];
            if (b == (int32_t)a) { data[j] = da > 0.0 ? 1.0 : 0.0; continue; }
            const double w = -data[j], db = deg[b];
            double v = 0.0;
            if (mode == ASP_LAPLACIAN_SYM) { if (da > 0.0 && db > 0.0) v = -__ddiv_rn(w, __dsqrt_rn(__dmul_rn(da, db))); }
            else if (da > 0.0) v = -__ddiv_rn(w, da);
            data[j] = v;
        }
    }
}

}  // namespace

int asp_graph_host_mirror(asp_graph *g)
{
    if (!g->h_indptr.empty()) return ASP_OK;
    asp_ctx *ctx = g->ctx;
    g->h_indptr.resize(g->nnodes + 1);
    g->h_indices.resize(g->nnz);
    g->h_data.resize(g->nnz);
    ASP_CUDA(cudaMemcpyAsync(g->h_indptr.data(), g->d_indptr, sizeof(int64_t) * (g->nnodes + 1), cudaMemcpyDeviceToHost, ctx->stream));
    ASP_CUDA(cudaMemcpyAsync(g->h_indices.data(), g->d_indices, sizeof(int32_t) * g->nnz, cudaMemcpyDeviceToHost, ctx->stream));
    ASP_CUDA(cudaMemcpyAsync(g->h_data.data(), g->d_data, sizeof(double) * g->nnz, cudaMemcpyDeviceToHost, ctx->stream));
    ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ASP_OK;
}

int asp_assemble_laplacian(asp_ctx *ctx, const asp_knn_lists *lists, const asp_graph_params *gp, const asp_switches *sw,
                           asp_graph *g)
{
    const int64_t m = lists->m;
    const int kk = lists->kk;
    cudaStream_t st = ctx->stream;
    const int grid = ctx->num_sms * 8;
    const double sigma = gp->has_sigma ? gp->sigma : gp->eps * 0.5;     // src/helpers.rs:68-72

    weights_compact_kernel<<<grid, 256, 0, st>>>(m, kk, lists->idx, lists->dist, lists->cnt, sigma, gp->p, sw->kernel);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    if (sw->symmetrise == ASP_SYM_AVG || sw->symmetrise == ASP_SYM_MIN) {
        symmetrise_mark_kernel<<<grid, 256, 0, st>>>(m, kk, lists->idx, lists->dist, lists->cnt, sw->symmetrise);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
        if (sw->symmetrise == ASP_SYM_MIN) {
            drop_marked_kernel<<<grid, 256, 0, st>>>(m, kk, lists->idx, lists->dist, lists->cnt);
            ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
        }
    }
    const int mirror = (sw->symmetrise == ASP_SYM_NONE || sw->symmetrise == ASP_SYM_MIN) ? 0 : 1;

    asp_scratch sc(st);                                                   // temporaries; the g-> arrays belong to the graph
    int32_t *extra = nullptr, *cursor = nullptr, *long_count = nullptr;
    int64_t *block_sums = nullptr, *total = nullptr, *long_rows = nullptr;
    const int64_t nblocks = asp_ceil_div(m, SCAN_BLOCK);
    ASP_CHECK(sc.get(&extra, (size_t)m));
    ASP_CHECK(sc.get(&cursor, (size_t)m));
    ASP_CHECK(sc.get(&long_count, 1));
    ASP_CHECK(sc.get(&block_sums, (size_t)nblocks));
    ASP_CHECK(sc.get(&total, 1));
    ASP_CHECK(sc.get(&long_rows, (size_t)m));
    ASP_CUDA(cudaMemsetAsync(extra, 0, sizeof(int32_t) * m, st));
    ASP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int32_t) * m, st));
    ASP_CUDA(cudaMemsetAsync(long_count, 0, sizeof(int32_t), st));

    if (mirror) {
        count_mirror_kernel<<<grid, 256, 0, st>>>(m, kk, lists->idx, lists->cnt, extra);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    }

    ASP_CUDA(cudaMallocAsync(&g->d_indptr, sizeof(int64_t) * (m + 1), st));
    scan_blocks_kernel<<<(unsigned)nblocks, SCAN_BLOCK, 0, st>>>(m, lists->cnt, extra, g->d_indptr, block_sums);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    scan_sums_kernel<<<1, SCAN_BLOCK, 0, st>>>(nblocks, block_sums, total);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    scan_add_kernel<<<(unsigned)nblocks, SCAN_BLOCK, 0, st>>>(m, g->d_indptr, block_sums, total);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);

    int64_t nnz = 0;
    ASP_CUDA(cudaMemcpyAsync(&nnz, total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    g->nnodes = m;
    g->nnz = nnz;
    ASP_CUDA(cudaMallocAsync(&g->d_indices, sizeof(int32_t) * (nnz > 0 ? nnz : 1), st));
    ASP_CUDA(cudaMallocAsync(&g->d_data, sizeof(double) * (nnz > 0 ? nnz : 1), st));

    fill_kernel<<<grid, 256, 0, st>>>(m, kk, lists->idx, lists->dist, lists->cnt, g->d_indptr, cursor, g->d_indices,
                                      g->d_data, mirror);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);

    sort_rows_warp_kernel<<<grid, 256, 0, st>>>(m, g->d_indptr, g->d_indices, g->d_data, long_rows, long_count);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    int32_t *scratch_col = nullptr;
    double *scratch_w = nullptr;
    ASP_CHECK(sc.get(&scratch_col, 2 * (size_t)nnz));
    ASP_CHECK(sc.get(&scratch_w, 2 * (size_t)nnz));
    sort_rows_block_kernel<<<ctx->num_sms * 2, 256, 0, st>>>(long_rows, long_count, g->d_indptr, g->d_indices, g->d_data,
                                                             scratch_col, scratch_w);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);

    if (sw->laplacian != ASP_LAPLACIAN_COMBINATORIAL) {
        double *deg = nullptr;
        ASP_CHECK(sc.get(&deg, (size_t)m));
        extract_degree_kernel<<<grid, 256, 0, st>>>(m, g->d_indptr, g->d_indices, g->d_data, deg);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
        normalise_kernel<<<grid, 256, 0, st>>>(m, g->d_indptr, g->d_indices, g->d_data, deg, sw->laplacian);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    }
    return ASP_OK;
}
