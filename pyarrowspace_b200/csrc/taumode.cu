// taumode.cu -- K3: per-vector taumode lambda (items at build time, queries at search time).
//   E = x^T L x / x^T x,  tau = max(median(x), 1e-9),  lambda = E / (E + tau)          (bounded form)
//   lambda = tau * E/(E+tau) + (1 - tau) * G(x),  G = clamp(sum e_ab^2 / (sum e_ab)^2)  (synthetic form, TAUMODE.md:8,26-27)
// (TAUMODE.md:18-19,24-27; SURVEY.md Appendix A8; replaces the lambda pass of ArrowSpaceBuilder::build and
// ArrowSpace::prepare_query_item, /root/reference/src/lib.rs:289,154).
//
// Formulation.  For ANY square L,  x^T L x = sum_a x_a (L_aa x_a - 2 sum_{b>a} c_ab x_b)  with  c_ab = -(L_ab + L_ba) / 2
// (the symmetrised quadratic form; c_ab = w_ab for the combinatorial Laplacian).  Only these strictly-upper coefficients
// are walked: half the gathers of a CSR SpMM, and the random-walk / unsymmetrised Laplacians of the unpinned switches
// need no second code path.
//
// ONE kernel, one pass over X (round 1 had a separate median kernel that read X a second time):
//   CTA = THR compute threads + 3 auxiliary warps + 1 producer warp, persistent over tiles of T = 16*R vectors.
//   compute warps   A. load the tile's rows (coalesced, two rows in flight per warp), store them transposed into shared
//                      memory xs[feature][item] (row stride T+1: conflict free both ways) and select the row's MEDIAN (tau)
//                      from the registers that still hold it: interpolation search on the empirical distribution
//                      (~8 passes of 12 compares + one warp reduction; exact, radix selection as fallback)
//                   B. walk the graph: a (part p = tid/16, lane group g = tid%16) pair owns items g+16r (r < R) and the row
//                      pieces p, p+NP, ... of the current graph chunk; per FOUR non-zeros: one 8-byte load of 4 columns, two
//                      16-byte loads of 4 coefficients (broadcasts), 4*R conflict-free 8-byte gathers of x
//                   C. partial energies: half-warp pairs by shuffle, warps through shared memory in warp order
//   auxiliary warps the left-to-right sums of squares (the norm the search divides by, the oracle's order; one thread per item)
//                      under the graph walk
//   producer warp   streams the graph, pre-cut into fixed-size chunks (cp.async.bulk + mbarrier, two buffers), and asks L2
//                      for the next tile's rows (cp.async.bulk.prefetch.L2) so that phase A finds them there
// Why the median sits in phase A: during the walk the LSU / MIO pipe is ~94 % busy with gathers (ncu), and every
// warp-collective instruction of a selection (redux, shuffles, shared-memory atomics) queues behind them -- medians on
// auxiliary warps next to the walk cost 1.9 - 3.7 ms per 1M items whatever the algorithm (profiles/k3_r02.md).
// Bound (SURVEY.md 8(d) K3): HBM 8*n*f bytes while nnz(L)/f is small; at k = 25 (nnz/f = 41) the 8-byte shared-memory
// gather per upper non-zero per item binds (128 B/clk/SM), see DESIGN.md section 4.
//
// Vectors longer than 1500 features do not fit a transposed tile: taumode_wide_kernel (one CTA per vector, the row in
// shared memory, block-wide selection) covers them up to 16384 features.
#include "common.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <math.h>
#include <stdlib.h>

namespace {

constexpr double TAU_FLOOR = 1e-9;

// ---- graph blob: row pieces of the upper coefficients in fixed-size chunks (one bulk copy each)
constexpr int TM_PIECE = 16;                                 // entries per row piece (multiple of 4)
constexpr int TM_CH_ENT = 512;                               // entries per chunk
constexpr int TM_CH_ROWS = 64;                               // pieces per chunk
constexpr int TM_OFF_W = 0;                                  // double  [TM_CH_ENT]   coefficient c_ab
constexpr int TM_OFF_COL = TM_OFF_W + TM_CH_ENT * 8;         // uint16  [TM_CH_ENT]   column b
constexpr int TM_OFF_DIAG = TM_OFF_COL + TM_CH_ENT * 2;      // double  [TM_CH_ROWS]  L_aa on the first piece of a row, else 0
constexpr int TM_OFF_PIECE = TM_OFF_DIAG + TM_CH_ROWS * 8;   // uint16x4[TM_CH_ROWS]  {row a, first entry (multiple of 4), end entry, 0}
constexpr int TM_OFF_HDR = TM_OFF_PIECE + TM_CH_ROWS * 8;    // int32   [4]           {pieces in this chunk, 0, 0, 0}
constexpr int TM_CHUNK_BYTES = TM_OFF_HDR + 16;
static_assert(TM_CHUNK_BYTES % 16 == 0 && TM_OFF_COL % 16 == 0 && TM_OFF_DIAG % 16 == 0, "bulk copies move 16-byte units");
constexpr int TM_AUX_WARPS = 3;                               // norm chains (one thread per item, T <= 64); + 1 producer warp = 4 warps

struct TmBlob {
    void *d_chunks = nullptr;
    int nchunks = 0;
    // plain upper CSR + diagonal of the same form, for taumode_wide_kernel
    int32_t *d_uptr = nullptr, *d_ucol = nullptr;
    double *d_uval = nullptr, *d_diag = nullptr;
};

// ---- order-preserving 64-bit keys
// key(x) is monotone in x for every non-NaN double (-0.0 is folded into +0.0 first); absent elements carry the largest key.
__device__ __forceinline__ unsigned long long f64_key(double x)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(x + 0.0);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(unsigned long long k)
{
    const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// identical leading bits of the n present keys (64: all equal); k0 = key of element 0
template <int FPL>
__device__ __forceinline__ int warp_common_lead(const unsigned long long (&k)[FPL], int n, int lane, unsigned long long *k0_out)
{
    uint32_t dhi = 0, dlo = 0;
    const unsigned long long k0 = __shfl_sync(0xffffffffu, k[0], 0);            // element 0 is always present
#pragma unroll
    for (int j = 0; j < FPL; ++j) {
        const bool present = (lane + 32 * j) < n;
        const unsigned long long d = present ? (k[j] ^ k0) : 0ull;
        dhi |= (uint32_t)(d >> 32);
        dlo |= (uint32_t)d;
    }
    dhi = __reduce_or_sync(0xffffffffu, dhi);
    dlo = __reduce_or_sync(0xffffffffu, dlo);
    *k0_out = k0;
    if ((dhi | dlo) == 0u) return 64;
    return dhi ? __clz(dhi) : 32 + __clz(dlo);
}

// the single key under (mask, prefix): fetched from the lane that holds it
template <int FPL>
__device__ __forceinline__ unsigned long long warp_fetch_unique(const unsigned long long (&k)[FPL], int n, int lane,
                                                                unsigned long long mask, unsigned long long prefix)
{
    unsigned long long mine = 0ull;
    bool have = false;
#pragma unroll
    for (int j = 0; j < FPL; ++j) {
        const bool act = ((lane + 32 * j) < n) && ((k[j] & mask) == prefix);
        if (act) { mine = k[j]; have = true; }
    }
    const int src = __ffs(__ballot_sync(0xffffffffu, have)) - 1;
    return __shfl_sync(0xffffffffu, mine, src);
}

// One MSB-first radix pass over the keys under (mask, prefix): which digit of `width` bits at `shift` holds the r-th of them.
// ALU form, NO shared memory: every lane counts its keys into sixteen 8-bit fields of two 64-bit registers, eight warp
// reductions (redux.sync) add the lanes, every lane scans the 16 totals.  width <= 4.
template <int FPL>
__device__ __forceinline__ void radix_pass_alu(const unsigned long long (&k)[FPL], int n, int lane, unsigned long long mask,
                                               unsigned long long prefix, int shift, int width, int r, uint32_t *digit,
                                               uint32_t *cnt, uint32_t *before)
{
    static_assert(FPL <= 255, "8-bit per-lane counters");
    unsigned long long ca = 0ull, cb = 0ull;                                     // bins 0-7 / 8-15, 8 bits each
    const uint32_t dmask = (1u << width) - 1u;
#pragma unroll
    for (int j = 0; j < FPL; ++j) {
        const bool act = ((lane + 32 * j) < n) && ((k[j] & mask) == prefix);
        const uint32_t d = (uint32_t)(k[j] >> shift) & dmask;
        const unsigned long long inc = act ? (1ull << (8 * (d & 7u))) : 0ull;
        if (d & 8u) cb += inc; else ca += inc;
    }
    uint32_t c[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t wa = (uint32_t)((ca >> (16 * i)) & 0xffull) | ((uint32_t)((ca >> (16 * i + 8)) & 0xffull) << 16);
        const uint32_t wb = (uint32_t)((cb >> (16 * i)) & 0xffull) | ((uint32_t)((cb >> (16 * i + 8)) & 0xffull) << 16);
        const uint32_t ta = __reduce_add_sync(0xffffffffu, wa), tb = __reduce_add_sync(0xffffffffu, wb);
        c[2 * i] = ta & 0xffffu; c[2 * i + 1] = ta >> 16;
        c[8 + 2 * i] = tb & 0xffffu; c[8 + 2 * i + 1] = tb >> 16;
    }
    uint32_t run = 0, dg = 0, cn = 0, bf = 0;
    bool found = false;
#pragma unroll
    for (int b = 0; b < 16; ++b) {
        const bool here = !found && (run + c[b] > (uint32_t)r);
        if (here) { dg = b; cn = c[b]; bf = run; found = true; }
        run += c[b];
    }
    *digit = dg; *cnt = cn; *before = bf;
}

// rank-th smallest key (0-based) of the n present keys held as k[j] of lane l = element l + 32 j.  MSB-first radix
// selection, 4 bits per pass; the bits all keys share are skipped and the walk stops as soon as the selected bin holds one
// key.  Exact for ANY input (ties, signed zeros, hundreds of binades): the fallback of the interpolation search below.
// *count_le = number of keys <= result.
template <int FPL>
__device__ unsigned long long warp_select(const unsigned long long (&k)[FPL], int n, int rank, int lane, int *count_le)
{
    unsigned long long k0;
    const int lead = warp_common_lead<FPL>(k, n, lane, &k0);
    if (lead == 64) { *count_le = n; return k0; }
    int remaining = 64 - lead;                                                   // low bits that may differ, >= 1
    unsigned long long prefix = (remaining == 64) ? 0ull : (k0 >> remaining) << remaining;
    unsigned long long mask = (remaining == 64) ? 0ull : ~0ull << remaining;
    int below = 0, r = rank;
    for (;;) {
        const int shift = remaining > 4 ? remaining - 4 : 0;
        const int width = remaining - shift;
        uint32_t digit, cnt, before;
        radix_pass_alu<FPL>(k, n, lane, mask, prefix, shift, width, r, &digit, &cnt, &before);
        below += (int)before;
        r -= (int)before;
        prefix |= (unsigned long long)digit << shift;
        mask |= (unsigned long long)((1u << width) - 1u) << shift;
        if (shift == 0) { *count_le = below + (int)cnt; return prefix; }         // cnt equal keys
        if (cnt == 1u) { *count_le = below + 1; return warp_fetch_unique<FPL>(k, n, lane, mask, prefix); }
        remaining = shift;
    }
}

// warp minimum / maximum of per-lane doubles through their order-preserving keys: four redux.sync, no shuffles
__device__ __forceinline__ double warp_min_f64(double v)
{
    const unsigned long long k = f64_key(v);
    const uint32_t hi = __reduce_min_sync(0xffffffffu, (uint32_t)(k >> 32));
    const uint32_t lo = __reduce_min_sync(0xffffffffu, ((uint32_t)(k >> 32) == hi) ? (uint32_t)k : 0xffffffffu);
    return key_f64(((unsigned long long)hi << 32) | lo);
}

// Exact selection by INTERPOLATION SEARCH on the empirical distribution, NV rows of one warp in lock step (NV = 2 gives the
// dependent chain of a pass -- compare, count, interpolate -- a second independent instance to overlap with).
// v[i][j] of lane l = element l + 32 j of row i (absent elements: NaN).  Per row: a bracket (lo, hi] that contains the wanted
// order statistic, c(lo) = #{v <= lo} <= rank < c(hi); the pivot is the linear interpolation of the rank inside the bracket;
// one pass counts #{v <= pivot} (12 compares per row at F = 384, the lane counts of both rows packed in one register and
// summed by a 5-step shuffle butterfly) and shrinks the bracket; a bracket that holds exactly one element ends the search
// and the element is fetched from the lane that owns it.  ~8 passes for embedding rows (C4 data: mean 8.2, p95 13) against
// ~2500 instructions for the radix selection.  ok[i] = false when row i was not isolated within MAX_PASSES (duplicates around
// the wanted rank, values spanning hundreds of binades, non-finite entries): the caller falls back to the radix selection.
template <int FPL, int NV>
__device__ void warp_select_interp(const double (&v)[NV][FPL], const bool (&want)[NV], int n, int rank, int lane,
                                   double (&result)[NV], int (&count_le)[NV], bool (&ok)[NV])
{
    constexpr int MAX_PASSES = 16;
    double lo[NV], hi[NV];
    int clo[NV], chi[NV];
    bool active[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        ok[i] = false;
        active[i] = want[i];
        // bracket from the high words of the extreme keys: lo strictly below every element, hi at or above every element
        double mn = INFINITY, mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < FPL; ++j) { mn = fmin(mn, v[i][j]); mx = fmax(mx, v[i][j]); }   // fmin / fmax skip the NaN of absent elements
        const uint32_t kmn = __reduce_min_sync(0xffffffffu, (uint32_t)(f64_key(mn) >> 32));
        const uint32_t kmx = __reduce_max_sync(0xffffffffu, (uint32_t)(f64_key(mx) >> 32));
        lo[i] = key_f64((((unsigned long long)kmn) << 32) - 1ull);
        hi[i] = key_f64((((unsigned long long)kmx) << 32) | 0xffffffffull);
        clo[i] = 0;
        chi[i] = n;
        if (!(hi[i] - lo[i] < INFINITY) || kmn == 0u) active[i] = false;         // non-finite entries / overflowing range: radix decides
    }
    for (int pass = 0; pass < MAX_PASSES; ++pass) {
        bool any = false;
        double p[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            p[i] = hi[i];
            if (!active[i]) continue;
            if (chi[i] - clo[i] == 1) {                                          // exactly one element in (lo, hi]: fetch it
                double mine = 0.0;
                bool have = false;
#pragma unroll
                for (int j = 0; j < FPL; ++j) { const bool in = (v[i][j] > lo[i]) && (v[i][j] <= hi[i]); if (in) { mine = v[i][j]; have = true; } }
                const int src = __ffs(__ballot_sync(0xffffffffu, have)) - 1;
                result[i] = __shfl_sync(0xffffffffu, mine, src) + 0.0;           // (-0.0 folded like the keys)
                count_le[i] = chi[i];
                ok[i] = true;
                active[i] = false;
                continue;
            }
            const float frac = __fdividef((float)(rank - clo[i]) + 0.5f, (float)(chi[i] - clo[i]));
            double q = fma(hi[i] - lo[i], (double)frac, lo[i]);
            if (!(q > lo[i] && q < hi[i])) q = lo[i] + 0.5 * (hi[i] - lo[i]);
            if (!(q > lo[i] && q < hi[i])) { active[i] = false; continue; }      // no double strictly inside: equal values, radix decides
            p[i] = q;
            any = true;
        }
        if (!any) return;
        uint32_t c = 0;                                                          // lane counts of the rows, 16 bits each
#pragma unroll
        for (int i = 0; i < NV; ++i)
#pragma unroll
            for (int j = 0; j < FPL; ++j) c += (v[i][j] <= p[i]) ? (1u << (16 * i)) : 0u;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            if (!active[i]) continue;
            const int ci = (int)((c >> (16 * i)) & 0xffffu);
            if (ci > rank) { hi[i] = p[i]; chi[i] = ci; } else { lo[i] = p[i]; clo[i] = ci; }
        }
    }
}

// medians of NV rows: the middle element, or the mean of the two middle ones (oracle.c median_of).  v[i][j] of lane l =
// element l + 32 j of row i (NaN when absent, already |.|-ed for median_abs).  use_interp: interpolation search first, radix
// selection as its fallback; else the radix selection only (A/B).
template <int FPL, int NV>
__device__ void warp_medians(const double (&v)[NV][FPL], const bool (&want)[NV], int n, int lane, int use_interp, double (&med)[NV])
{
    static_assert(NV <= 2 && FPL * 32 < 65536, "lane counts are packed 16 bits per row");
    const int r0 = (n & 1) ? n / 2 : n / 2 - 1;
    double vlo[NV];
    int cle[NV];
    bool ok[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) { ok[i] = false; vlo[i] = 0.0; cle[i] = 0; }
    if (use_interp) warp_select_interp<FPL, NV>(v, want, n, r0, lane, vlo, cle, ok);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        if (!want[i]) { med[i] = 1.0; continue; }
        if (!ok[i]) {
            unsigned long long k[FPL];
#pragma unroll
            for (int j = 0; j < FPL; ++j) k[j] = ((lane + 32 * j) < n) ? f64_key(v[i][j]) : ~0ull;
            vlo[i] = key_f64(warp_select<FPL>(k, n, r0, lane, &cle[i]));
        }
        double vhi = vlo[i];
        if (!(n & 1) && cle[i] < n / 2 + 1) {    // the next order statistic is the smallest value > vlo
            double m = INFINITY;
#pragma unroll
            for (int j = 0; j < FPL; ++j)
                if (v[i][j] > vlo[i]) m = fmin(m, v[i][j]);
            vhi = warp_min_f64(m) + 0.0;
        }
        med[i] = (n & 1) ? vlo[i] : 0.5 * (vlo[i] + vhi);
    }
}

__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(asp::smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(asp::smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *gmem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(gmem_src), "r"(bytes) : "memory");
}
template <int ID>
__device__ __forceinline__ void named_sync(int nthreads) { asm volatile("bar.sync %0, %1;\n" ::"n"(ID), "r"(nthreads) : "memory"); }
template <int ID>
__device__ __forceinline__ void named_arrive(int nthreads) { asm volatile("bar.arrive %0, %1;\n" ::"n"(ID), "r"(nthreads) : "memory"); }

template <int FPL, int R, int THR, bool SYN>
__global__ void __launch_bounds__(THR + 32 * TM_AUX_WARPS + 32, 1)
taumode_kernel(const double *__restrict__ x, int64_t n, int f, int pitch, const unsigned char *__restrict__ blob, int nchunks,
               int tau_mode, double tau_fixed, int use_interp, double *__restrict__ out_energy, double *__restrict__ out_tau,
               double *__restrict__ out_lambda, double *__restrict__ out_norm, double *__restrict__ out_inv_norm, int *zero_flag)
{
    constexpr int T = 16 * R;
    constexpr int XS = T + 1;
    constexpr int NW = THR / 32;                                       // compute warps
    constexpr int NP = THR / 16;                                       // parts: row pieces in flight
    constexpr int NAUX = 32 * TM_AUX_WARPS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *xs = reinterpret_cast<double *>(smem_raw);                                          // f * XS
    unsigned char *cbuf = smem_raw + (((size_t)f * XS * 8 + 15) & ~(size_t)15);               // 2 * TM_CHUNK_BYTES
    double *red = reinterpret_cast<double *>(cbuf + 2 * TM_CHUNK_BYTES);                        // NW * T
    double *s_tau = red + NW * T;                                                               // T
    double *s_n2 = s_tau + T;                                                                   // T
    __shared__ __align__(8) uint64_t full_bar[2], empty_bar[2];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool is_compute = threadIdx.x < THR;
    const bool is_aux = !is_compute && threadIdx.x < THR + NAUX;
    const int64_t ntiles = (n + T - 1) / T;
    if (threadIdx.x == 0) {
        for (int b = 0; b < 2; ++b) { asp::mbar_init(&full_bar[b], 1); asp::mbar_init(&empty_bar[b], NW); }
        asp::fence_barrier_init();
    }
    __syncthreads();

    if (!is_compute && !is_aux) {
        // ===================== producer warp: graph chunks + L2 prefetch of the next tile's rows =====================
        if (lane == 0) {
            int64_t it = 0;
            const bool can_prefetch = ((pitch & 1) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
            for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int64_t nxt = tile + gridDim.x;
                if (can_prefetch && nxt < ntiles) {
                    const int64_t i0 = nxt * T, i1 = (i0 + T < n) ? i0 + T : n;
                    bulk_prefetch_l2(x + i0 * pitch, (uint32_t)((i1 - i0) * pitch * 8));
                }
                for (int c = 0; c < nchunks; ++c, ++it) {
                    const int b = (int)(it & 1);
                    asp::mbar_wait(&empty_bar[b], (uint32_t)(((it >> 1) & 1) ^ 1));
                    asp::mbar_arrive_expect_tx(&full_bar[b], TM_CHUNK_BYTES);
                    bulk_g2s(cbuf + b * TM_CHUNK_BYTES, blob + (size_t)c * TM_CHUNK_BYTES, TM_CHUNK_BYTES, &full_bar[b]);
                }
            }
        }
        return;
    }

    const int g = threadIdx.x & 15, p = threadIdx.x >> 4;               // compute: lane group / part
    int64_t it = 0;                                                     // chunk sequence number (compute warps)
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t item0 = tile * T;
        if (is_aux) {
            named_sync<3>(THR + NAUX);                                 // the transposed tile is complete
            // ---- left-to-right sums (norm^2; mean), one thread per item
            const int ct = threadIdx.x - THR;
            if (ct < T) {
                double n2 = 0.0, sm = 0.0;
#pragma unroll 8
                for (int ff = 0; ff < f; ++ff) {                       // loads and products run ahead; only the adds are a chain
                    const double xv = xs[ff * XS + ct];
                    n2 = __dadd_rn(n2, __dmul_rn(xv, xv));
                    sm = __dadd_rn(sm, xv);
                }
                s_n2[ct] = n2;
                if (tau_mode == ASP_TAU_MEAN || tau_mode == ASP_TAU_FIXED) {     // (the medians come from the compute warps, phase A)
                    const double tau = (tau_mode == ASP_TAU_MEAN) ? sm / (double)f : tau_fixed;
                    s_tau[ct] = (tau > TAU_FLOOR) ? tau : TAU_FLOOR;
                }
            }
        } else {
            // ---- A: rows -> transposed tile, two rows in flight per warp (one when a row is more than 24 registers wide).
            // The per-vector median (tau) is selected HERE, from the registers that hold the row: in this phase the LSU /
            // MIO pipe is idle (the warps wait for L2), whereas during the graph walk every warp-collective instruction of
            // a selection (redux, shuffles, shared-memory atomics) queues behind the gathers -- measured: 64 medians on
            // auxiliary warps next to the walk cost 1.9 - 3.7 ms per 1M items whatever the selection algorithm.
            const bool want_median = (tau_mode == ASP_TAU_MEDIAN || tau_mode == ASP_TAU_MEDIAN_ABS);
            constexpr int NV = (FPL <= 24) ? 2 : 1;
            for (int t0 = warp; t0 < T; t0 += NV * NW) {
                double vv[NV][FPL];
                bool in[NV];
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const int t = t0 + i * NW;
                    in[i] = (t < T) && (item0 + t < n);
                    const double *row = x + (item0 + t) * pitch;
#pragma unroll
                    for (int j = 0; j < FPL; ++j) { const int ff = lane + 32 * j; vv[i][j] = (in[i] && ff < f) ? row[ff] : 0.0; }
                }
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const int t = t0 + i * NW;
                    if (t < T) {
#pragma unroll
                        for (int j = 0; j < FPL; ++j) { const int ff = lane + 32 * j; if (ff < f) xs[ff * XS + t] = vv[i][j]; }
                    }
                }
                if (want_median) {
                    const bool ab = tau_mode == ASP_TAU_MEDIAN_ABS;
#pragma unroll
                    for (int i = 0; i < NV; ++i)
#pragma unroll
                        for (int j = 0; j < FPL; ++j) { const int ff = lane + 32 * j; vv[i][j] = (ff < f) ? (ab ? fabs(vv[i][j]) : vv[i][j]) : NAN; }
                    double med[NV];
                    warp_medians<FPL, NV>(vv, in, f, lane, use_interp, med);
#pragma unroll
                    for (int i = 0; i < NV; ++i) {
                        const int t = t0 + i * NW;
                        if (lane == 0 && t < T) s_tau[t] = (med[i] > TAU_FLOOR) ? med[i] : TAU_FLOOR;
                    }
                }
            }
            named_sync<1>(THR);                                        // the tile is complete (compute warps)
            named_arrive<3>(THR + NAUX);                               // ... and the auxiliary warps may start

            // ---- B: x^T L x through the upper coefficients, chunk by chunk
            double en[R], tot[SYN ? R : 1], sq[SYN ? R : 1];
#pragma unroll
            for (int r = 0; r < R; ++r) en[r] = 0.0;
#pragma unroll
            for (int r = 0; r < (SYN ? R : 1); ++r) { tot[r] = 0.0; sq[r] = 0.0; }
            const double *xg = xs + g;
            for (int c = 0; c < nchunks; ++c, ++it) {
                const int b = (int)(it & 1);
                asp::mbar_wait(&full_bar[b], (uint32_t)((it >> 1) & 1));
                const unsigned char *cb = cbuf + b * TM_CHUNK_BYTES;
                const double *cw = reinterpret_cast<const double *>(cb + TM_OFF_W);
                const uint16_t *cc = reinterpret_cast<const uint16_t *>(cb + TM_OFF_COL);
                const double *cdiag = reinterpret_cast<const double *>(cb + TM_OFF_DIAG);
                const uint2 *cpiece = reinterpret_cast<const uint2 *>(cb + TM_OFF_PIECE);
                const int npieces = *reinterpret_cast<const int *>(cb + TM_OFF_HDR);
                for (int slot = p; slot < npieces; slot += NP) {
                    const uint2 pc = cpiece[slot];
                    const int a = (int)(pc.x & 0xffffu), jb = (int)(pc.x >> 16), je = (int)(pc.y & 0xffffu);
                    double xa[R], s[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) { xa[r] = xg[a * XS + 16 * r]; s[r] = 0.0; }
                    int j = jb;
                    for (; j + 4 <= je; j += 4) {
                        const uint2 c4 = *reinterpret_cast<const uint2 *>(cc + j);
                        const double2 w01 = *reinterpret_cast<const double2 *>(cw + j), w23 = *reinterpret_cast<const double2 *>(cw + j + 2);
                        const double *x0 = xg + (int)(c4.x & 0xffffu) * XS, *x1 = xg + (int)(c4.x >> 16) * XS;
                        const double *x2 = xg + (int)(c4.y & 0xffffu) * XS, *x3 = xg + (int)(c4.y >> 16) * XS;
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const double b0 = x0[16 * r], b1 = x1[16 * r], b2 = x2[16 * r], b3 = x3[16 * r];
                            s[r] = fma(w01.x, b0, s[r]);
                            s[r] = fma(w01.y, b1, s[r]);
                            s[r] = fma(w23.x, b2, s[r]);
                            s[r] = fma(w23.y, b3, s[r]);
                            if (SYN) {                                 // edgewise Dirichlet energies e = c (x_a - x_b)^2
                                const double d0 = xa[r] - b0, d1 = xa[r] - b1, d2 = xa[r] - b2, d3 = xa[r] - b3;
                                const double e0 = w01.x * d0 * d0, e1 = w01.y * d1 * d1, e2 = w23.x * d2 * d2, e3 = w23.y * d3 * d3;
                                tot[r] += (e0 + e1) + (e2 + e3);
                                sq[r] = fma(e0, e0, fma(e1, e1, fma(e2, e2, fma(e3, e3, sq[r]))));
                            }
                        }
                    }
                    for (; j < je; ++j) {                              // the 0-3 entries left of the piece, one at a time
                        const double w = cw[j];
                        const double *x0 = xg + (int)cc[j] * XS;
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const double b0 = x0[16 * r];
                            s[r] = fma(w, b0, s[r]);
                            if (SYN) { const double d0 = xa[r] - b0, e0 = w * d0 * d0; tot[r] += e0; sq[r] = fma(e0, e0, sq[r]); }
                        }
                    }
                    const double dg = cdiag[slot];
#pragma unroll
                    for (int r = 0; r < R; ++r) en[r] = fma(xa[r], fma(dg, xa[r], -2.0 * s[r]), en[r]);
                }
                __syncwarp();
                if (lane == 0) asp::mbar_arrive(&empty_bar[b]);
            }
            // ---- C: the two parts of a warp by shuffle, the warps through shared memory (summed in warp order below)
#pragma unroll
            for (int r = 0; r < R; ++r) {
                en[r] += __shfl_xor_sync(0xffffffffu, en[r], 16);
                if (lane < 16) red[warp * T + g + 16 * r] = en[r];
            }
            if (SYN) {
#pragma unroll
                for (int r = 0; r < R; ++r) { tot[r] += __shfl_xor_sync(0xffffffffu, tot[r], 16); sq[r] += __shfl_xor_sync(0xffffffffu, sq[r], 16); }
            }
            double num = 0.0, gt = 0.0, gs = 0.0;
            named_sync<2>(THR + NAUX);                                 // partial energies, norms and taus are in shared memory
            if (threadIdx.x < T) for (int q = 0; q < NW; ++q) num += red[q * T + threadIdx.x];
            if (SYN) {                                                 // two more rounds through the same buffer
                named_sync<1>(THR);
#pragma unroll
                for (int r = 0; r < R; ++r) if (lane < 16) red[warp * T + g + 16 * r] = tot[r];
                named_sync<1>(THR);
                if (threadIdx.x < T) for (int q = 0; q < NW; ++q) gt += red[q * T + threadIdx.x];
                named_sync<1>(THR);
#pragma unroll
                for (int r = 0; r < R; ++r) if (lane < 16) red[warp * T + g + 16 * r] = sq[r];
                named_sync<1>(THR);
                if (threadIdx.x < T) for (int q = 0; q < NW; ++q) gs += red[q * T + threadIdx.x];
            }
            if (threadIdx.x < T) {
                const int t = threadIdx.x;
                const int64_t item = item0 + t;
                if (item < n) {
                    const double n2 = s_n2[t];
                    const double tau = s_tau[t];
                    double e = NAN, lam = NAN;
                    if (n2 == 0.0) atomicExch(zero_flag, 1);             // TAUMODE.md:13
                    else {
                        e = num / n2;
                        lam = e / (e + tau);                             // TAUMODE.md:19,25
                        if (SYN) {                                       // TAUMODE.md:8,26-27
                            double gd = (gt == 0.0) ? 0.0 : gs / (gt * gt);
                            gd = gd < 0.0 ? 0.0 : (gd > 1.0 ? 1.0 : gd);
                            lam = tau * lam + (1.0 - tau) * gd;
                        }
                    }
                    if (out_energy) out_energy[item] = e;
                    if (out_tau) out_tau[item] = tau;
                    if (out_lambda) out_lambda[item] = lam;
                    const double nr = sqrt(n2);
                    if (out_norm) out_norm[item] = nr;
                    if (out_inv_norm) out_inv_norm[item] = (nr > 0.0) ? 1.0 / nr : 0.0;
                }
            }
        }
        if (is_aux) named_sync<2>(THR + NAUX);                         // (the compute warps passed theirs before the reduction)
        named_sync<4>(THR + NAUX);                                     // the tile is fully consumed: xs / s_tau / s_n2 / red reusable
    }
}

// ---- vectors of more than 1500 features: one CTA per vector, the row in shared memory
constexpr int TW_THREADS = 256;

__global__ void __launch_bounds__(TW_THREADS)
taumode_wide_kernel(const double *__restrict__ x, int64_t n, int f, int pitch, const int32_t *__restrict__ uptr,
                    const int32_t *__restrict__ ucol, const double *__restrict__ uval, const double *__restrict__ diag,
                    int tau_mode, double tau_fixed, int synthetic, double *__restrict__ out_energy, double *__restrict__ out_tau,
                    double *__restrict__ out_lambda, double *__restrict__ out_norm, double *__restrict__ out_inv_norm, int *zero_flag)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *xr = reinterpret_cast<double *>(smem_raw);                 // f
    __shared__ double s_part[3][TW_THREADS / 32];
    __shared__ uint32_t s_cnt[16];
    __shared__ double s_n2, s_mean;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int64_t item = blockIdx.x; item < n; item += gridDim.x) {
        __syncthreads();
        const double *row = x + item * pitch;
        for (int j = threadIdx.x; j < f; j += TW_THREADS) xr[j] = row[j];
        __syncthreads();
        // left-to-right sums on one thread (the oracle's order) while the other warps walk the graph
        if (threadIdx.x == 0) {
            double n2 = 0.0, sm = 0.0;
            for (int j = 0; j < f; ++j) { const double v = xr[j]; n2 = __dadd_rn(n2, __dmul_rn(v, v)); sm = __dadd_rn(sm, v); }
            s_n2 = n2; s_mean = sm / (double)f;
        }
        double en = 0.0, tot = 0.0, sq = 0.0;
        if (warp > 0) {
            for (int a = warp - 1; a < f; a += TW_THREADS / 32 - 1) {
                const double xa = xr[a];
                double s = 0.0;
                for (int j = uptr[a] + lane; j < uptr[a + 1]; j += 32) {
                    const double w = uval[j], xb = xr[ucol[j]];
                    s = fma(w, xb, s);
                    if (synthetic) { const double d = xa - xb, e = w * d * d; tot += e; sq = fma(e, e, sq); }
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
                en = fma(xa, fma(diag[a], xa, -2.0 * s), en);          // identical on every lane
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) { tot += __shfl_xor_sync(0xffffffffu, tot, off); sq += __shfl_xor_sync(0xffffffffu, sq, off); }
        if (lane == 0) { s_part[0][warp] = en; s_part[1][warp] = tot; s_part[2][warp] = sq; }
        // block-wide radix selection of the median (4 bits per pass over the keys in shared memory)
        double tau = tau_fixed;
        if (tau_mode == ASP_TAU_MEDIAN || tau_mode == ASP_TAU_MEDIAN_ABS) {
            const bool use_abs = tau_mode == ASP_TAU_MEDIAN_ABS;
            double med[2];
            const int ranks[2] = {(f & 1) ? f / 2 : f / 2 - 1, f / 2};
            for (int which = 0; which < ((f & 1) ? 1 : 2); ++which) {
                unsigned long long prefix = 0ull, mask = 0ull;
                int r = ranks[which];
                for (int shift = 60; shift >= 0; shift -= 4) {
                    __syncthreads();
                    if (threadIdx.x < 16) s_cnt[threadIdx.x] = 0u;
                    __syncthreads();
                    uint32_t loc[16];
#pragma unroll
                    for (int b = 0; b < 16; ++b) loc[b] = 0u;
                    for (int j = threadIdx.x; j < f; j += TW_THREADS) {
                        const unsigned long long key = f64_key(use_abs ? fabs(xr[j]) : xr[j]);
                        if ((key & mask) == prefix) {
                            const uint32_t d = (uint32_t)(key >> shift) & 15u;
#pragma unroll
                            for (int b = 0; b < 16; ++b) loc[b] += (d == (uint32_t)b) ? 1u : 0u;
                        }
                    }
#pragma unroll
                    for (int b = 0; b < 16; ++b) {
                        const uint32_t t = __reduce_add_sync(0xffffffffu, loc[b]);
                        if (lane == 0 && t) atomicAdd(&s_cnt[b], t);
                    }
                    __syncthreads();
                    uint32_t run = 0, digit = 0;
                    bool found = false;
                    for (int b = 0; b < 16; ++b) {
                        const uint32_t cbin = s_cnt[b];
                        if (!found && run + cbin > (uint32_t)r) { digit = b; r -= (int)run; found = true; }
                        run += cbin;
                    }
                    prefix |= (unsigned long long)digit << shift;
                    mask |= 15ull << shift;
                }
                med[which] = key_f64(prefix);
            }
            tau = (f & 1) ? med[0] : 0.5 * (med[0] + med[1]);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            if (tau_mode == ASP_TAU_MEAN) tau = s_mean;
            tau = (tau > TAU_FLOOR) ? tau : TAU_FLOOR;
            double num = 0.0, gt = 0.0, gs = 0.0;
            for (int w = 0; w < TW_THREADS / 32; ++w) { num += s_part[0][w]; gt += s_part[1][w]; gs += s_part[2][w]; }
            const double n2 = s_n2;
            double e = NAN, lam = NAN;
            if (n2 == 0.0) atomicExch(zero_flag, 1);
            else {
                e = num / n2;
                lam = e / (e + tau);
                if (synthetic) {
                    double gd = (gt == 0.0) ? 0.0 : gs / (gt * gt);
                    gd = gd < 0.0 ? 0.0 : (gd > 1.0 ? 1.0 : gd);
                    lam = tau * lam + (1.0 - tau) * gd;
                }
            }
            if (out_energy) out_energy[item] = e;
            if (out_tau) out_tau[item] = tau;
            if (out_lambda) out_lambda[item] = lam;
            const double nr = sqrt(n2);
            if (out_norm) out_norm[item] = nr;
            if (out_inv_norm) out_inv_norm[item] = (nr > 0.0) ? 1.0 / nr : 0.0;
        }
    }
}

template <int FPL, int R, int THR>
int launch_tm(asp_ctx *ctx, const TmBlob *blob, const asp_switches *sw, const double *x, int64_t n, int f, int pitch,
              double *oe, double *ot, double *ol, double *on, double *oi, int *zero_flag)
{
    constexpr int T = 16 * R;
    constexpr int NTHREADS = THR + 32 * TM_AUX_WARPS + 32;
    // median selection (A/B knob ASP_TM_MEDIAN = interp | alu): interpolation search with the ALU radix selection as its
    // fallback, or the radix selection alone; both select the same element, so the knob cannot change a result.
    int use_interp = 1;
    if (const char *menv = getenv("ASP_TM_MEDIAN")) { if (menv[0] == 'a') use_interp = 0; }
    const bool syn = sw->lambda_form == ASP_LAMBDA_SYNTHETIC;
    const size_t smem = (((size_t)f * (T + 1) * 8 + 15) & ~(size_t)15) + 2 * (size_t)TM_CHUNK_BYTES + (size_t)(THR / 32) * T * 8 +
                        (size_t)T * 16;
    if (smem > 227 * 1024) ASP_FAIL(ASP_ERR_UNSUPPORTED, "taumode kernel: %d features do not fit in shared memory", f);
    auto kern = syn ? taumode_kernel<FPL, R, THR, true> : taumode_kernel<FPL, R, THR, false>;
    ASP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;                                                       // resident CTAs per SM: their load / gather phases overlap
    ASP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NTHREADS, smem));
    if (occ < 1) occ = 1;
    const int64_t ntiles = (n + T - 1) / T;
    const int64_t slots = (int64_t)ctx->num_sms * occ;
    const int grid = (int)(ntiles < slots ? ntiles : slots);
    kern<<<grid, NTHREADS, smem, ctx->stream>>>(x, n, f, pitch, static_cast<const unsigned char *>(blob->d_chunks), blob->nchunks,
                                                  sw->tau_mode, sw->tau_fixed, use_interp, oe, ot, ol, on, oi, zero_flag);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}

// Symmetrised quadratic form of the host CSR, cut into pieces and chunks (see the top of the file).
int build_tm_blob(asp_ctx *ctx, const asp_graph *g, TmBlob *out)
{
    const int64_t m = g->nnodes;
    if (m > 65535) ASP_FAIL(ASP_ERR_UNSUPPORTED, "the lambda pass supports at most 65535 graph nodes (got %lld)", (long long)m);
    std::vector<std::vector<std::pair<int32_t, double>>> up(m);
    std::vector<double> diag(m, 0.0);
    for (int64_t a = 0; a < m; ++a)
        for (int64_t j = g->h_indptr[a]; j < g->h_indptr[a + 1]; ++j) {
            const int32_t c = g->h_indices[j];
            if (c == a) { diag[a] += g->h_data[j]; continue; }
            const int64_t lo = c < a ? c : a;
            const int32_t hi = c < a ? (int32_t)a : c;
            up[lo].push_back({hi, -0.5 * g->h_data[j]});               // c_ab = -(L_ab + L_ba) / 2
        }
    std::vector<int32_t> uptr(m + 1, 0), ucol;
    std::vector<double> uval;
    for (int64_t a = 0; a < m; ++a) {
        auto &v = up[a];
        std::stable_sort(v.begin(), v.end(), [](const std::pair<int32_t, double> &x, const std::pair<int32_t, double> &y) { return x.first < y.first; });
        size_t o = 0;
        for (size_t i = 0; i < v.size(); ++i) {
            if (o > 0 && v[o - 1].first == v[i].first) v[o - 1].second += v[i].second;    // row a's entry first, then row b's
            else v[o++] = v[i];
        }
        v.resize(o);
        for (auto &e : v) { ucol.push_back(e.first); uval.push_back(e.second); }
        uptr[a + 1] = (int32_t)ucol.size();
    }
    // pieces, longest first (equal lengths inside a chunk balance the parts)
    struct Piece { int32_t row, beg, len; double diag; };
    std::vector<Piece> pieces;
    for (int64_t a = 0; a < m; ++a) {
        const int32_t len = uptr[a + 1] - uptr[a];
        if (len == 0) { if (diag[a] != 0.0) pieces.push_back({(int32_t)a, uptr[a], 0, diag[a]}); continue; }
        for (int32_t o = 0; o < len; o += TM_PIECE)
            pieces.push_back({(int32_t)a, uptr[a] + o, std::min<int32_t>(TM_PIECE, len - o), o == 0 ? diag[a] : 0.0});
    }
    std::stable_sort(pieces.begin(), pieces.end(), [](const Piece &x, const Piece &y) { return x.len > y.len; });
    std::vector<unsigned char> blob;
    int nchunks = 0;
    size_t i = 0;
    while (i < pieces.size() || nchunks == 0) {
        blob.resize((size_t)(nchunks + 1) * TM_CHUNK_BYTES, 0);
        unsigned char *cb = blob.data() + (size_t)nchunks * TM_CHUNK_BYTES;
        double *cw = reinterpret_cast<double *>(cb + TM_OFF_W);
        uint16_t *cc = reinterpret_cast<uint16_t *>(cb + TM_OFF_COL);
        double *cd = reinterpret_cast<double *>(cb + TM_OFF_DIAG);
        uint16_t *cp = reinterpret_cast<uint16_t *>(cb + TM_OFF_PIECE);
        int np = 0, ne = 0;
        while (i < pieces.size() && np < TM_CH_ROWS) {
            const Piece &pc = pieces[i];
            const int padded = (pc.len + 3) & ~3;
            if (ne + padded > TM_CH_ENT) break;
            cp[4 * np + 0] = (uint16_t)pc.row; cp[4 * np + 1] = (uint16_t)ne; cp[4 * np + 2] = (uint16_t)(ne + pc.len); cp[4 * np + 3] = 0;
            cd[np] = pc.diag;
            for (int e = 0; e < padded; ++e) {
                cw[ne + e] = e < pc.len ? uval[pc.beg + e] : 0.0;      // storage padding (pieces start on 4-entry boundaries), never walked
                cc[ne + e] = (uint16_t)(e < pc.len ? ucol[pc.beg + e] : pc.row);
            }
            ne += padded; ++np; ++i;
        }
        *reinterpret_cast<int32_t *>(cb + TM_OFF_HDR) = np;
        ++nchunks;
    }
    cudaStream_t st = ctx->stream;
    const size_t un = ucol.empty() ? 1 : ucol.size();
    ASP_CUDA(cudaMallocAsync(&out->d_chunks, blob.size(), st));
    ASP_CUDA(cudaMallocAsync(&out->d_uptr, sizeof(int32_t) * (m + 1), st));
    ASP_CUDA(cudaMallocAsync(&out->d_ucol, sizeof(int32_t) * un, st));
    ASP_CUDA(cudaMallocAsync(&out->d_uval, sizeof(double) * un, st));
    ASP_CUDA(cudaMallocAsync(&out->d_diag, sizeof(double) * m, st));
    ASP_CUDA(cudaMemcpyAsync(out->d_chunks, blob.data(), blob.size(), cudaMemcpyHostToDevice, st));
    ASP_CUDA(cudaMemcpyAsync(out->d_uptr, uptr.data(), sizeof(int32_t) * (m + 1), cudaMemcpyHostToDevice, st));
    if (!ucol.empty()) {
        ASP_CUDA(cudaMemcpyAsync(out->d_ucol, ucol.data(), sizeof(int32_t) * ucol.size(), cudaMemcpyHostToDevice, st));
        ASP_CUDA(cudaMemcpyAsync(out->d_uval, uval.data(), sizeof(double) * uval.size(), cudaMemcpyHostToDevice, st));
    }
    ASP_CUDA(cudaMemcpyAsync(out->d_diag, diag.data(), sizeof(double) * m, cudaMemcpyHostToDevice, st));
    ASP_CUDA(cudaStreamSynchronize(st));                               // the host vectors go out of scope
    out->nchunks = nchunks;
    return ASP_OK;
}

}  // namespace

// Called once per feature graph (asp_graph_from_gram): the graph-only inputs of the lambda pass.  A per-call upload would
// queue behind the query uploads of a pipelined search.
int asp_graph_upload_upper(asp_graph *g)
{
    ASP_CHECK(asp_graph_host_mirror(g));
    TmBlob *b = new TmBlob();
    g->tm_blob = b;                                                    // a partly built blob is freed like a complete one
    const int rc = build_tm_blob(g->ctx, g, b);
    if (rc != ASP_OK) asp_graph_free_upper(g);
    return rc;
}

void asp_graph_free_upper(asp_graph *g)
{
    if (!g->tm_blob) return;
    TmBlob *b = static_cast<TmBlob *>(g->tm_blob);
    cudaStream_t st = g->ctx->stream;
    void *bufs[] = {b->d_chunks, b->d_uptr, b->d_ucol, b->d_uval, b->d_diag};
    for (void *p : bufs)
        if (p) cudaFreeAsync(p, st);
    delete b;
    g->tm_blob = nullptr;
}

int asp_launch_taumode(asp_ctx *ctx, const asp_graph *g, const asp_switches *sw, const double *x_dev, int64_t n,
                       int32_t f, int32_t pitch, double *out_energy, double *out_tau, double *out_lambda,
                       double *out_norm, double *out_inv_norm, int *zero_flag_dev)
{
    if (n == 0) return ASP_OK;
    if (f != g->nnodes) ASP_FAIL(ASP_ERR_ARG, "vector length %d must equal the graph's node count %lld", f, (long long)g->nnodes);
    if (!g->tm_blob) ASP_FAIL(ASP_ERR_ARG, "graph has no upper adjacency (not a feature graph)");
    const TmBlob *b = static_cast<const TmBlob *>(g->tm_blob);
    if (f <= 128)  return launch_tm<4, 4, 256>(ctx, b, sw, x_dev, n, f, pitch, out_energy, out_tau, out_lambda, out_norm, out_inv_norm, zero_flag_dev);
    if (f <= 384)  return launch_tm<12, 4, 512>(ctx, b, sw, x_dev, n, f, pitch, out_energy, out_tau, out_lambda, out_norm, out_inv_norm, zero_flag_dev);
    if (f <= 768)  return launch_tm<24, 2, 256>(ctx, b, sw, x_dev, n, f, pitch, out_energy, out_tau, out_lambda, out_norm, out_inv_norm, zero_flag_dev);
    if (f <= 1024) return launch_tm<32, 1, 256>(ctx, b, sw, x_dev, n, f, pitch, out_energy, out_tau, out_lambda, out_norm, out_inv_norm, zero_flag_dev);
    if (f <= 1500) return launch_tm<47, 1, 128>(ctx, b, sw, x_dev, n, f, pitch, out_energy, out_tau, out_lambda, out_norm, out_inv_norm, zero_flag_dev);
    if (f > 16384) ASP_FAIL(ASP_ERR_UNSUPPORTED, "the lambda pass supports at most 16384 features (got %d)", f);
    const size_t smem = (size_t)f * 8;
    ASP_CUDA(cudaFuncSetAttribute(taumode_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t want = (int64_t)ctx->num_sms * 4;
    taumode_wide_kernel<<<(unsigned)(n < want ? n : want), TW_THREADS, smem, ctx->stream>>>(
        x_dev, n, f, pitch, b->d_uptr, b->d_ucol, b->d_uval, b->d_diag, sw->tau_mode, sw->tau_fixed,
        sw->lambda_form == ASP_LAMBDA_SYNTHETIC ? 1 : 0, out_energy, out_tau, out_lambda, out_norm, out_inv_norm, zero_flag_dev);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}
