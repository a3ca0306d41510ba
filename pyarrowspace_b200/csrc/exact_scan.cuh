// exact_scan.cuh -- the exact fallback of the search and of the item graph: rows whose candidate set could not be proven
// complete (ties around the k-th score, emission overflow, topk beyond the kept lists) are answered from the
// reference-order value of EVERY item.  All such rows of a call go through two launches:
//   scan_topk_kernel   block (x, y) = item range x of QPB query rows: a thread owns an item row at a time and carries the QPB
//                      ordered dot products together (the row is read once for all of them); the values of a chunk land in
//                      shared memory and one warp per query row folds them into that row's running top-k (k rounds of "best
//                      entry strictly after the previous winner": exact ties by index);
//   merge_kernel       one block per query row: the same k rounds over the ranges' top-k lists.
// What a value is (search score | negated graph distance, and which items are admissible) comes from a policy object.
#pragma once

#include <stdint.h>
#include <math.h>

namespace asp_xs {

constexpr int THREADS = 256, CHUNK = 1024, TOPK_MAX = 1024;
constexpr int64_t NONE = INT64_MAX;

// order (value desc, index asc): does (s, i) come strictly after (ps, pi) / strictly before (bs, bi)?
__device__ __forceinline__ bool after(double s, int64_t i, double ps, int64_t pi) { return (s < ps) || (s == ps && i > pi); }
__device__ __forceinline__ bool before(double s, int64_t i, double bs, int64_t bi) { return (s > bs) || (s == bs && i < bi); }

inline size_t scan_smem_bytes(int qpb, int f, int64_t topk) { return sizeof(double) * (size_t)qpb * f + (size_t)qpb * (2 * topk + CHUNK) * 16; }

// part_value / part_idx: [nslow][gridDim.x][topk]
template <int QPB, class Policy>
__global__ void __launch_bounds__(THREADS)
scan_topk_kernel(Policy pol, int first, int nslow, const double *__restrict__ items, int64_t n_local, int f, int pitch, int topk,
                 double *__restrict__ part_value, int64_t *__restrict__ part_idx)
{
    extern __shared__ __align__(128) unsigned char xs_smem[];
    double *qs = reinterpret_cast<double *>(xs_smem);                         // [QPB][f]
    double *sc = qs + (size_t)QPB * f;                                        // [QPB][topk | CHUNK | topk]: top, chunk, new top
    int64_t *ix = reinterpret_cast<int64_t *>(sc + (size_t)QPB * (2 * topk + CHUNK));
    const int stride = 2 * topk + CHUNK;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q0 = blockIdx.y * QPB;
    typename Policy::Row rowc[QPB];
    bool live[QPB];
#pragma unroll
    for (int u = 0; u < QPB; ++u) {
        live[u] = q0 + u < nslow;
        rowc[u] = pol.row(first + (live[u] ? q0 + u : 0));
    }
    for (int j = threadIdx.x; j < QPB * f; j += THREADS) {
        const int u = j / f, t = j - u * f;
        qs[j] = (q0 + u < nslow) ? pol.query(first + q0 + u)[t] : 0.0;
    }
    for (int j = threadIdx.x; j < QPB * topk; j += THREADS) {
        const int u = j / topk, t = j - u * topk;
        sc[u * stride + t] = -INFINITY;
        ix[u * stride + t] = NONE;
    }
    __syncthreads();
    const int64_t per = (n_local + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = blockIdx.x * per, r1 = (r0 + per < n_local) ? r0 + per : n_local;
    for (int64_t c0 = r0; c0 < r1; c0 += CHUNK) {
        const int len = (int)((r1 - c0 < CHUNK) ? r1 - c0 : CHUNK);
        for (int e = threadIdx.x; e < len; e += THREADS) {
            const int64_t it = c0 + e;
            const double *row = items + it * pitch;
            double d[QPB];
#pragma unroll
            for (int u = 0; u < QPB; ++u) d[u] = 0.0;
            int j = 0;
            for (; j + 2 <= f; j += 2) {                                      // one load of the row for the QPB ordered sums
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
            const typename Policy::Item ic = pol.item(it);
#pragma unroll
            for (int u = 0; u < QPB; ++u) {
                bool valid = true;
                const double v = pol.value(rowc[u], ic, d[u], it, valid);
                sc[u * stride + topk + e] = v;
                ix[u * stride + topk + e] = valid ? it : NONE;
            }
        }
        __syncthreads();
        if (warp < QPB && live[warp]) {                                       // warp u folds the chunk into row u's top-k
            double *s_u = sc + warp * stride;
            int64_t *i_u = ix + warp * stride;
            const int total = topk + len;
            double ps = INFINITY;
            int64_t pi = -1;
            for (int r = 0; r < topk; ++r) {
                double bs = -INFINITY;
                int64_t bi = NONE;
                for (int e = lane; e < total; e += 32) {
                    const double v = s_u[e];
                    const int64_t vi = i_u[e];
                    if (vi != NONE && after(v, vi, ps, pi) && before(v, vi, bs, bi)) { bs = v; bi = vi; }
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    const double os = __shfl_xor_sync(0xffffffffu, bs, off);
                    const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
                    if (oi != NONE && before(os, oi, bs, bi)) { bs = os; bi = oi; }
                }
                if (lane == 0) { s_u[topk + CHUNK + r] = bs; i_u[topk + CHUNK + r] = bi; }
                if (bi == NONE) { ps = -INFINITY; pi = NONE; } else { ps = bs; pi = bi; }
            }
            __syncwarp();
            for (int r = lane; r < topk; r += 32) { s_u[r] = s_u[topk + CHUNK + r]; i_u[r] = i_u[topk + CHUNK + r]; }
        }
        __syncthreads();
    }
    for (int j = threadIdx.x; j < QPB * topk; j += THREADS) {
        const int u = j / topk, t = j - u * topk;
        if (q0 + u < nslow) {
            const size_t o = ((size_t)(q0 + u) * gridDim.x + blockIdx.x) * topk + t;
            part_value[o] = sc[u * stride + t];
            part_idx[o] = ix[u * stride + t];
        }
    }
}

// one block per query row: top-k of its nparts x topk range winners, handed to the policy in order
template <class Policy>
__global__ void __launch_bounds__(THREADS)
merge_kernel(Policy pol, int first, const double *__restrict__ part_value, const int64_t *__restrict__ part_idx, int nparts, int topk)
{
    __shared__ double s_s[THREADS / 32];
    __shared__ int64_t s_i[THREADS / 32];
    __shared__ double prev_s;
    __shared__ int64_t prev_i;
    __shared__ int s_count;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t base = (size_t)blockIdx.x * nparts * topk;
    const int total = nparts * topk;
    if (threadIdx.x == 0) { prev_s = INFINITY; prev_i = -1; s_count = 0; }
    __syncthreads();
    for (int r = 0; r < topk; ++r) {
        const double ps = prev_s;
        const int64_t pi = prev_i;
        double bs = -INFINITY;
        int64_t bi = NONE;
        for (int e = threadIdx.x; e < total; e += THREADS) {
            const double v = part_value[base + e];
            const int64_t vi = part_idx[base + e];
            if (vi != NONE && after(v, vi, ps, pi) && before(v, vi, bs, bi)) { bs = v; bi = vi; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double os = __shfl_xor_sync(0xffffffffu, bs, off);
            const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (oi != NONE && before(os, oi, bs, bi)) { bs = os; bi = oi; }
        }
        if (lane == 0) { s_s[warp] = bs; s_i[warp] = bi; }
        __syncthreads();
        if (warp == 0) {
            bs = (lane < THREADS / 32) ? s_s[lane] : -INFINITY;
            bi = (lane < THREADS / 32) ? s_i[lane] : NONE;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double os = __shfl_xor_sync(0xffffffffu, bs, off);
                const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
                if (oi != NONE && before(os, oi, bs, bi)) { bs = os; bi = oi; }
            }
            if (lane == 0) {
                const bool ok = (bi != NONE);
                pol.emit(first + (int)blockIdx.x, r, ok, bs, bi);
                if (ok) s_count = r + 1;
                prev_s = ok ? bs : -INFINITY;
                prev_i = ok ? bi : NONE;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) pol.finish(first + (int)blockIdx.x, s_count);
}

// Host driver: `nslow` rows in groups (bounded scratch, grid.y <= 65535).  launched(n) is called once per kernel launch.
template <class Policy, class Launched>
int run(cudaStream_t st, int num_sms, const Policy &pol, int nslow, const double *items, int64_t n_local, int f, int pitch,
        int64_t topk, Launched launched)
{
    if (nslow <= 0 || topk <= 0) return 0;
    if (topk > TOPK_MAX) return 1;
    const int qpb = (scan_smem_bytes(4, f, topk) <= 200 * 1024) ? 4 : 1;
    const size_t smem = scan_smem_bytes(qpb, f, topk);
    if (smem > 220 * 1024) return 2;
    int64_t nparts = (n_local + CHUNK - 1) / CHUNK;
    if (nparts > (int64_t)num_sms * 2) nparts = (int64_t)num_sms * 2;
    if (nparts < 1) nparts = 1;
    const int64_t ngroups = (nslow + qpb - 1) / qpb;
    int64_t max_groups = (int64_t)(1u << 28) / (nparts * topk * 16 * qpb);
    if (max_groups > 65535) max_groups = 65535;
    if (max_groups < 1) max_groups = 1;
    const int64_t alloc_groups = ngroups < max_groups ? ngroups : max_groups;
    asp_scratch sc(st);
    double *part_value = nullptr;
    int64_t *part_idx = nullptr;
    if (sc.get(&part_value, (size_t)alloc_groups * qpb * nparts * topk) != ASP_OK) return 3;
    if (sc.get(&part_idx, (size_t)alloc_groups * qpb * nparts * topk) != ASP_OK) return 3;
    int rc = 0;
    if (qpb == 4) { if (cudaFuncSetAttribute(scan_topk_kernel<4, Policy>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) rc = 4; }
    else { if (cudaFuncSetAttribute(scan_topk_kernel<1, Policy>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) rc = 4; }
    for (int64_t g0 = 0; g0 < ngroups && rc == 0; g0 += max_groups) {
        const int64_t ng = (max_groups < ngroups - g0) ? max_groups : ngroups - g0;
        const int first = (int)(g0 * qpb);
        const int count = (int)((ng * qpb < nslow - first) ? ng * qpb : nslow - first);
        const dim3 grid((unsigned)nparts, (unsigned)ng);
        if (qpb == 4) scan_topk_kernel<4, Policy><<<grid, THREADS, smem, st>>>(pol, first, count, items, n_local, f, pitch, (int)topk, part_value, part_idx);
        else scan_topk_kernel<1, Policy><<<grid, THREADS, smem, st>>>(pol, first, count, items, n_local, f, pitch, (int)topk, part_value, part_idx);
        launched(1);
        merge_kernel<Policy><<<(unsigned)count, THREADS, 0, st>>>(pol, first, part_value, part_idx, (int)nparts, (int)topk);
        launched(1);
        if (cudaGetLastError() != cudaSuccess) rc = 4;
    }
    return rc;
}

}  // namespace asp_xs
