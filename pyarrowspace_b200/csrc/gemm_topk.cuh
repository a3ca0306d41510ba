// gemm_topk.cuh -- the FP64 DMMA "scores + per-row top-LIST" GEMM shared by the search (K4) and the
// item-graph (K1, item orientation) kernels.  See search.cu for the stage-1 / stage-2 contract.
//
// MODE 0 (search):     score = tau*cos(q,x) + (1-tau)/(1+|lambda_q - lambda_x|)
// MODE 1 (item graph): score = max(0, cos(x_i, x_j)), j != i, score >= smin (= 1 - eps - band)
// FILTER (MODE 0 only): a column whose bit in `allowed` is clear is treated like one beyond n_local -- it never enters a
// row's list, so it never raises the row's threshold.
#pragma once
#include "common.cuh"
#include "ptx.cuh"
#include "warp_sort.cuh"

#include <math.h>

namespace asp_gemm {

using asp::Cand;

constexpr int QT = 128;            // queries per CTA tile
constexpr int IT = 128;            // items per tile
constexpr int KSTEP = 16;          // features per pipeline stage (4 DMMA k-slabs)
constexpr int OPER_DOUBLES = (KSTEP / 4) * 128 * 4;       // 2048 doubles = 16 KB
constexpr int STAGE_DOUBLES_S = 2 * OPER_DOUBLES;
constexpr int MMA_WARPS = 8;

// ============================================================================ stage 1: GEMM

template <int LIST>
struct ListSmem {
    static constexpr int CAP = 2 * LIST;
    double sc[QT * CAP];
    int32_t ix[QT * CAP];
    int32_t cnt[QT];
    double theta[QT];
};

// Sort the CAP-slot buffer of `row`, keep the best LIST, refresh the threshold.  Whole warp.
template <int LIST>
__device__ __noinline__ void compact_row(ListSmem<LIST> *ls, int row, int lane)
{
    constexpr int CAP = 2 * LIST;
    constexpr int NPL = CAP / 32;
    const int cnt = ls->cnt[row];
    Cand e[NPL];
#pragma unroll
    for (int t = 0; t < NPL; ++t) {
        const int i = lane + 32 * t;
        if (i < cnt) { e[t].s = ls->sc[row * CAP + i]; e[t].i = ls->ix[row * CAP + i]; }
        else e[t] = asp::cand_empty();
    }
    asp::warp_sort_best_first<NPL>(e, lane);
#pragma unroll
    for (int t = 0; t < NPL; ++t) {
        const int i = lane + 32 * t;
        if (i < LIST) { ls->sc[row * CAP + i] = e[t].s; ls->ix[row * CAP + i] = e[t].i; }
    }
    // element LIST-1 lives in lane (LIST-1)%32, slot (LIST-1)/32
    const double last = __shfl_sync(0xffffffffu, e[(LIST - 1) / 32].s, (LIST - 1) & 31);
    if (lane == 0) {
        ls->cnt[row] = cnt < LIST ? cnt : LIST;
        ls->theta[row] = (cnt >= LIST) ? last : -INFINITY;
    }
    __syncwarp();
}

template <int LIST, int STAGES, bool USE_TMA, int MODE, bool FILTER = false>
__global__ void __launch_bounds__(MMA_WARPS * 32, 1)
search_gemm_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                   const double *__restrict__ q, const double *__restrict__ items, int64_t nq, int64_t n_local, int fp,
                   const double *__restrict__ inv_nx, const double *__restrict__ lam_x,
                   const double *__restrict__ inv_nq, const double *__restrict__ lam_q, double tau, double smin,
                   int nchunks, double *__restrict__ cand_score, int32_t *__restrict__ cand_idx,
                   const uint32_t *__restrict__ allowed)
{
    static_assert(!FILTER || MODE == 0, "only the search is filtered");
    constexpr int CAP = 2 * LIST;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *stages = reinterpret_cast<double *>(smem_raw);
    ListSmem<LIST> *ls = reinterpret_cast<ListSmem<LIST> *>(stages + STAGES * STAGE_DOUBLES_S);
    __shared__ __align__(8) uint64_t full_bar[STAGES];
    __shared__ __align__(8) uint64_t empty_bar[STAGES];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qb = blockIdx.x, chunk = blockIdx.y;
    const int64_t tiles_total = (n_local + IT - 1) / IT;
    const int64_t tile0 = (tiles_total * chunk) / nchunks;               // even split of the item tiles
    const int64_t ntiles = (tiles_total * (chunk + 1)) / nchunks - tile0;
    const int ksteps = (fp + KSTEP - 1) / KSTEP;
    const int64_t total_it = ntiles * ksteps;

    for (int i = threadIdx.x; i < QT; i += blockDim.x) { ls->cnt[i] = 0; ls->theta[i] = -INFINITY; }
    if (USE_TMA && threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            asp::mbar_init(&full_bar[s], 1);
            asp::mbar_init(&empty_bar[s], MMA_WARPS);
        }
        asp::fence_barrier_init();
    }
    __syncthreads();

    // TMA producer = thread 0, inline: it runs STAGES-1 iterations ahead of the DMMA loop.
    auto tma_issue = [&](int64_t it) {
        const int s = (int)(it % STAGES);
        if (it >= STAGES) asp::mbar_wait(&empty_bar[s], (uint32_t)(((it / STAGES) - 1) & 1));
        double *dst = stages + s * STAGE_DOUBLES_S;
        const int64_t jt = it / ksteps;
        const int kk = (int)(it % ksteps);
        asp::mbar_arrive_expect_tx(&full_bar[s], STAGE_DOUBLES_S * 8u);
        asp::tma_load_3d(dst, &tmap_q, &full_bar[s], 0, qb * QT, kk * (KSTEP / 4));
        asp::tma_load_3d(dst + OPER_DOUBLES, &tmap_x, &full_bar[s], 0, (int)((tile0 + jt) * IT), kk * (KSTEP / 4));
    };
    if (USE_TMA && threadIdx.x == 0) {
        asp::tma_prefetch_desc(&tmap_q);
        asp::tma_prefetch_desc(&tmap_x);
        for (int64_t it = 0; it < STAGES - 1 && it < total_it; ++it) tma_issue(it);
    }

    // ===== consumers: warp w owns query rows [16w, 16w+16) x all 128 item columns of the tile
    const int rowA = warp * 16 + (lane >> 2);       // + 8*mt
    const int a_off = (rowA * 4) + (lane & 3);      // + ks*512 + mt*32
    const int b_off = ((lane >> 2) * 4) + (lane & 3);   // + ks*512 + nt*32

    // per-row constants of this lane's two rows
    double rq[2], lq[2], theta[2];
    bool qvalid[2];
    int rows[2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        rows[mt] = rowA + 8 * mt;
        const int64_t gq = (int64_t)qb * QT + rows[mt];
        qvalid[mt] = gq < nq;
        rq[mt] = qvalid[mt] ? tau * inv_nq[gq] : 0.0;
        lq[mt] = (MODE == 0 && qvalid[mt]) ? lam_q[gq] : 0.0;
        theta[mt] = -INFINITY;
    }
    const double beta = 1.0 - tau;

    auto load_stage_cp_async = [&](int64_t it) {
        const int s = (int)(it % STAGES);
        double *dst = stages + s * STAGE_DOUBLES_S;
        const int64_t jt = it / ksteps;
        const int kk = (int)(it % ksteps);
        for (int op = 0; op < 2; ++op) {
            const double *base = op == 0 ? q : items;
            const int64_t row_base = op == 0 ? (int64_t)qb * QT : (tile0 + jt) * IT;
            const int64_t row_lim = op == 0 ? nq : n_local;
            for (int c = threadIdx.x; c < 128 * KSTEP / 2; c += MMA_WARPS * 32) {
                const int r = c / (KSTEP / 2);
                const int fl = (c % (KSTEP / 2)) * 2;         // feature inside the k-step
                const int fg = kk * KSTEP + fl;
                const bool valid = (row_base + r < row_lim) && (fg < fp);
                const double *src = valid ? base + (row_base + r) * fp + fg : base;
                asp::cp_async16(dst + op * OPER_DOUBLES + (((fl >> 2) * 128 + r) * 4 + (fl & 3)), src, valid);
            }
        }
    };
    if (!USE_TMA) {
        for (int64_t it = 0; it < STAGES - 1; ++it) {
            if (it < total_it) load_stage_cp_async(it);
            asp::cp_async_commit();
        }
    }

    for (int64_t jt = 0; jt < ntiles; ++jt) {
        double acc[2][16][2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

        for (int kk = 0; kk < ksteps; ++kk) {
            const int64_t it = jt * ksteps + kk;
            const int s = (int)(it % STAGES);
            if (USE_TMA) {
                if (threadIdx.x == 0 && it + STAGES - 1 < total_it) tma_issue(it + STAGES - 1);
                asp::mbar_wait(&full_bar[s], (uint32_t)((it / STAGES) & 1));
            } else {
                asp::cp_async_wait<STAGES - 2>();
                __syncthreads();
                if (it + STAGES - 1 < total_it) load_stage_cp_async(it + STAGES - 1);
                asp::cp_async_commit();
            }
            const double *A = stages + s * STAGE_DOUBLES_S;
            const double *B = A + OPER_DOUBLES;
#pragma unroll
            for (int ks = 0; ks < KSTEP / 4; ++ks) {
                double a[2];
                a[0] = A[a_off + ks * 512];
                a[1] = A[a_off + ks * 512 + 32];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    double b[8];
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) b[nt] = B[b_off + ks * 512 + (half * 8 + nt) * 32];
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) {
                        asp::dmma884(acc[0][half * 8 + nt][0], acc[0][half * 8 + nt][1], a[0], b[nt]);
                        asp::dmma884(acc[1][half * 8 + nt][0], acc[1][half * 8 + nt][1], a[1], b[nt]);
                    }
                }
            }
            if (USE_TMA) {
                __syncwarp();
                if (lane == 0) asp::mbar_arrive(&empty_bar[s]);
            }
        }

        // ----- fused epilogue: score, threshold, push, compact (warp local)
        const int64_t item_base = (tile0 + jt) * IT;
#pragma unroll
        for (int nt = 0; nt < 16; ++nt) {
            const int64_t c0 = item_base + nt * 8 + 2 * (lane & 3);
            double inx[2], lmx[2];
            bool cvalid[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                cvalid[e] = (c0 + e) < n_local;
                if (FILTER) cvalid[e] = cvalid[e] && asp_allowed(allowed, c0 + e);
                inx[e] = cvalid[e] ? inv_nx[c0 + e] : 0.0;
                lmx[e] = (MODE == 0 && cvalid[e]) ? lam_x[c0 + e] : 0.0;
            }
            bool pushed = false;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double dot = acc[mt][nt][e];
                    const double cs = rq[mt] * dot * inx[e];
                    if (MODE == 0) {
                        if (cvalid[e] && qvalid[mt] && (cs + beta > theta[mt])) {
                            const double sc = cs + beta / (1.0 + fabs(lq[mt] - lmx[e]));
                            if (sc > theta[mt]) {
                                const int slot = atomicAdd(&ls->cnt[rows[mt]], 1);
                                ls->sc[rows[mt] * CAP + slot] = sc;
                                ls->ix[rows[mt] * CAP + slot] = (int32_t)(c0 + e);
                                pushed = true;
                            }
                        }
                    } else {
                        const double sc = cs > 0.0 ? cs : 0.0;             // rectified cosine
                        const bool self = ((int64_t)qb * QT + rows[mt]) == (c0 + e);
                        if (cvalid[e] && qvalid[mt] && !self && sc >= smin && sc > theta[mt]) {
                            const int slot = atomicAdd(&ls->cnt[rows[mt]], 1);
                            ls->sc[rows[mt] * CAP + slot] = sc;
                            ls->ix[rows[mt] * CAP + slot] = (int32_t)(c0 + e);
                            pushed = true;
                        }
                    }
                }
            }
            if (__any_sync(0xffffffffu, pushed)) {
                __syncwarp();
                const int myrow = warp * 16 + (lane & 15);
                unsigned need = __ballot_sync(0xffffffffu, (lane < 16) && (ls->cnt[myrow] > CAP - 8));
                while (need) {
                    const int rr = __ffs(need) - 1;
                    need &= need - 1;
                    compact_row<LIST>(ls, warp * 16 + rr, lane);
                }
                __syncwarp();
                theta[0] = ls->theta[rows[0]];
                theta[1] = ls->theta[rows[1]];
            }
        }
    }

    // ----- flush: final compaction of the warp's 16 rows, best LIST out
    __syncwarp();
    for (int rr = 0; rr < 16; ++rr) {
        const int row = warp * 16 + rr;
        compact_row<LIST>(ls, row, lane);
        const int64_t gq = (int64_t)qb * QT + row;
        if (gq < nq) {
            const int cnt = ls->cnt[row];
            for (int i = lane; i < LIST; i += 32) {
                const size_t o = ((size_t)gq * nchunks + chunk) * LIST + i;
                cand_score[o] = (i < cnt) ? ls->sc[row * CAP + i] : -INFINITY;
                cand_idx[o] = (i < cnt) ? ls->ix[row * CAP + i] : -1;
            }
        }
    }
}


__device__ __forceinline__ double seq_dot_row(const double *__restrict__ qv, const double *__restrict__ row, int f)
{
    double d = 0.0;
    int j = 0;
    for (; j + 4 <= f; j += 4) {
        const double2 x0 = *reinterpret_cast<const double2 *>(row + j);
        const double2 x1 = *reinterpret_cast<const double2 *>(row + j + 2);
        d = __dadd_rn(d, __dmul_rn(qv[j], x0.x));
        d = __dadd_rn(d, __dmul_rn(qv[j + 1], x0.y));
        d = __dadd_rn(d, __dmul_rn(qv[j + 2], x1.x));
        d = __dadd_rn(d, __dmul_rn(qv[j + 3], x1.y));
    }
    for (; j < f; ++j) d = __dadd_rn(d, __dmul_rn(qv[j], row[j]));
    return d;
}

}  // namespace asp_gemm
