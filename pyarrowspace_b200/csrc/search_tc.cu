// search_tc.cu -- K4 (batches) and K4' (small batches on large shards): stage 1 of the lambda-aware search on the 5th-generation tensor
// cores (tcgen05.mma, accumulators in TMEM, operands by TMA), stage 2 exact.
// (replaces ArrowSpace::search_lambda_aware, /root/reference/src/lib.rs:173; score TAUMODE.md:33.)
//
// Why: the f64 score GEMM is bound by the FP64 tensor pipe (35 TFLOP/s measured); 2*Q*N*F = 1.26e13 FLOP per
// 16k-query step at C4 cannot go below ~360 ms there.  tcgen05 has no f64 kind, but the ANSWER only needs f64 on a
// few candidates per query: stage 1 computes every cosine from a two-term fp16 split of the UNIT vectors
//     128 x^ = hi + lo + r,  |r| <= 2^-22 |128 x^|     q^.x^ ~ (q_lo.x_hi + q_hi.x_lo + q_hi.x_hi) 2^-14   (3 MMAs, f32 accumulate)
// with the band  |cos~ - cos| <= DELTA_COS(kp)  (split truncation 3*2^-22 + one f32 rounding per K=16 MMA step, x4
// margin; checked against f64 in tests/test_gpu_parity.py::test_tc_dot_error_band), and EMITS every item whose
// approximate score could still be in the top-k:  s~ >= theta_k - 2 DELTA, theta_k = running k-th best.
//
// Items are visited in LAMBDA ORDER (a bucket sort of the shard by lambda when the cache is built; `perm` maps back).
// A 256-item tile then spans a tiny lambda interval [lo, hi], so the proximity term of a (query, tile) pair is known
// up to ~1e-5 BEFORE looking at the accumulators:  s <= tau*cos + beta/(1 + dist(lambda_q, [lo, hi])).  That turns the
// per-element epilogue into ONE compare of the raw accumulator against a per-(row, tile) threshold (a max tree over
// 32 TMEM columns + 1 branch); the exact score expression runs only for the few elements that pass.  The running
// thresholds are shared between the column quarters of a row (shared memory) and between the CTAs that scan
// different item chunks for the same query (global atomicMax), so late chunks start with a warm threshold.
//
// Stage 2 (tc_rescore_kernel<WPQ>), one warp per query for batches, a whole CTA per query for small batches (the
// reference's one query per call: the per-query work is a chain of dependent global loads, so it is spread over
// 8 or 32 warps and the per-warp lists are merged pairwise): (A) every survivor of the final cut is re-scored in f64 with a
// warp-cooperative coalesced dot product (error <= EPS ~ 1e-13), the best 32 kept; (B) the candidates within 2 EPS of
// the k-th best are re-scored in the reference order (sequential, __dmul_rn/__dadd_rn: exactly the oracle's
// expression) and sorted by (score desc, index asc).  More than 32 candidates inside that band, or a full emission
// buffer, send the query to the exact scan.  The result is bit-identical to the FP64 path's (tests assert it).
//
// Per-call k of 32 .. 64 (asp_search_batch_k and the hybrid _k entry points only; their `wide` flag): stage 1 runs with
// 64-entry running lists (ceil(k / 4) <= 16 scores per column-quarter thread, so every threshold is still a lower bound of
// the k-th best score) and a larger emission capacity; stage 2 is tc_rescore_wide_kernel, one CTA per query, which keeps
// every survivor of the cut (up to asp_lk::SURV_CAP) instead of 32 per warp: large_k.cuh.  The graph-topk entry points never
// set the flag, so a graph topk >= 32 still takes the exact scan there; moving them onto this route needs its own B200
// measurements and a deliberate change of the test that pins their route.
//
// Completeness.  Let t_k be the exact k-th best score.  Any running threshold theta is the k-th best APPROXIMATE score
// of some k distinct items, whose exact scores are >= theta - DELTA, so t_k >= theta - DELTA.  An item of the true top-k
// has s >= t_k, hence s~ >= s - DELTA >= theta - 2 DELTA: it passes every emission test and the final cut.  The same
// argument with EPS in place of DELTA covers (A) -> (B).
//
// Filtered search (FILTER instantiations): a per-call bitmask in VISITING order, vbits[pos] = allowed[perm[pos]], gives the
// 32 columns of one TMEM load in one word.  The rare path drops the columns that are not allowed before anything else, so no
// such item is emitted, enters a quarter list or raises theta_k / s_theta / theta_glob: every threshold stays the k-th best
// approximate score of k distinct allowed items and the argument above holds over the allowed set.  The common path is
// unchanged.  A query with fewer allowed items than topk never gets a finite threshold; stage 2 sees fewer than k
// candidates in the band and sends it to the exact scan (search_slow_queries), which skips the rows that are not allowed.
//
// Kernel (one CTA per SM, 64 + 512 threads):
//   warp 0     TMA producer: 4-stage ring of {128 queries x 64 k, 256 items x 64 k} fp16 tiles, SWIZZLE_128B
//   warp 1     allocates TMEM (512 columns = 2 accumulators of 128 x 256 f32), issues tcgen05.mma (one lane),
//              tcgen05.commit -> frees the smem stage / publishes the accumulator
//   warps 2-17 epilogue: tcgen05.ld 32 lanes x 32 columns; thread <-> (query row, 64-column quarter of the tile)
// Bound: fp16 tensor pipe, 3 * 2*Q*N*Fp FLOP executed for 2*Q*N*F algorithmic.
#include "common.cuh"
#include "ptx.cuh"
#include "warp_sort.cuh"
#include "l2_bound.cuh"
#include "large_k.cuh"
#include "sweep_bound.cuh"

#include <cuda_fp16.h>
#include <algorithm>
#include <math.h>
#include <memory>
#include <stdlib.h>

namespace {

using asp::Cand;

constexpr int TQ = 128;            // queries per CTA (UMMA M)
constexpr int TN = 256;            // items per tile (UMMA N)
constexpr int TKB = 64;            // fp16 per smem row = 128 B = one swizzle atom
constexpr int TC_STAGES = 4;
constexpr int A_BYTES = TQ * TKB * 2;          // 16 KB
constexpr int B_BYTES = TN * TKB * 2;          // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int TK_LIST_MAX = 32;    // running top list per (query row, column quarter): 16 or 32 registers (topk <= 32)
constexpr int EPI_WARPS = 16;      // 4 per TMEM lane group: each thread owns one query row x 64 of the 256 tile columns
constexpr int EPI_SPLIT = EPI_WARPS / 4;
constexpr int EPI_COLS = TN / EPI_SPLIT;
constexpr int TC_THREADS = 64 + EPI_WARPS * 32;
constexpr double OPERAND_SCALE = 128.0;                                  // unit vectors are stored as fp16(128 x^): lo stays normal
constexpr float ACC_SCALE = (float)(OPERAND_SCALE * OPERAND_SCALE);      // accumulator = 2^14 cos
constexpr int LAM_BUCKETS = 1 << 16;

// order-preserving float <-> uint32 (thresholds are shared with atomicMax); 0 = "none yet", below every float
__device__ __forceinline__ uint32_t f2o(float f) { const uint32_t b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float o2f(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }

// ------------------------------------------------------------------ cache construction: lambda order, fp16 split
__global__ void minmax_kernel(const double *__restrict__ a, int64_t n, double *__restrict__ out /* [grid][2] */)
{
    double lo = INFINITY, hi = -INFINITY;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = a[i];
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
    __shared__ double s_lo[256], s_hi[256];
    s_lo[threadIdx.x] = lo;
    s_hi[threadIdx.x] = hi;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) {
            s_lo[threadIdx.x] = fmin(s_lo[threadIdx.x], s_lo[threadIdx.x + off]);
            s_hi[threadIdx.x] = fmax(s_hi[threadIdx.x], s_hi[threadIdx.x + off]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[2 * blockIdx.x] = s_lo[0]; out[2 * blockIdx.x + 1] = s_hi[0]; }
}

// [lo, 1/bucket width] of the keys from the per-block partials of minmax_kernel (one warp)
__global__ void range_finalize_kernel(const double *__restrict__ partials, int nblocks, double *__restrict__ range)
{
    double lo = INFINITY, hi = -INFINITY;
    for (int i = threadIdx.x; i < nblocks; i += 32) { lo = fmin(lo, partials[2 * i]); hi = fmax(hi, partials[2 * i + 1]); }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, off));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, off));
    }
    if (threadIdx.x == 0) {
        const double width = (hi > lo) ? (hi - lo) / LAM_BUCKETS : 1.0;
        range[0] = lo;
        range[1] = 1.0 / width;
    }
}

__device__ __forceinline__ int lam_bucket(double v, double lo, double inv_width)
{
    const double t = (v - lo) * inv_width;
    int b = (t > 0.0) ? (int)t : 0;                                      // NaN -> 0
    return b < LAM_BUCKETS ? b : LAM_BUCKETS - 1;
}

__global__ void bucket_hist_kernel(const double *__restrict__ lam, int64_t n, const double *__restrict__ range, uint32_t *__restrict__ hist)
{
    const double lo = range[0], inv_width = range[1];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&hist[lam_bucket(lam[i], lo, inv_width)], 1u);
}

// exclusive scan of LAM_BUCKETS counters by one CTA of 1024 threads (64 counters per thread, held in registers: all 16
// 16-byte loads of a thread are in flight together)
__global__ void __launch_bounds__(1024) bucket_scan_kernel(uint32_t *__restrict__ hist /* in: counts, out: cursors */)
{
    constexpr int PER = LAM_BUCKETS / 1024;
    static_assert(PER % 4 == 0, "vector loads");
    __shared__ uint32_t s_warp[32];
    uint4 *mine = reinterpret_cast<uint4 *>(hist + threadIdx.x * PER);
    uint4 v[PER / 4];
#pragma unroll
    for (int j = 0; j < PER / 4; ++j) v[j] = mine[j];
    uint32_t tot = 0;
#pragma unroll
    for (int j = 0; j < PER / 4; ++j) tot += v[j].x + v[j].y + v[j].z + v[j].w;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = tot;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = s_warp[lane], wi = w;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, wi, off);
            if (lane >= off) wi += t;
        }
        s_warp[lane] = wi - w;                                           // exclusive prefix of the warp totals
    }
    __syncthreads();
    uint32_t run = s_warp[warp] + incl - tot;
#pragma unroll
    for (int j = 0; j < PER / 4; ++j) {
        uint4 o;
        o.x = run; run += v[j].x;
        o.y = run; run += v[j].y;
        o.z = run; run += v[j].z;
        o.w = run; run += v[j].w;
        mine[j] = o;
    }
}

__global__ void bucket_scatter_kernel(const double *__restrict__ lam, int64_t n, const double *__restrict__ range,
                                      uint32_t *__restrict__ cursor, int32_t *__restrict__ perm)
{
    const double lo = range[0], inv_width = range[1];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        perm[atomicAdd(&cursor[lam_bucket(lam[i], lo, inv_width)], 1u)] = (int32_t)i;
}

// visiting order: for every query block, the tile whose lambda interval is nearest to the block's median lambda_q
// (tiles are in ascending lambda order: last tile whose lower end is <= the median)
__global__ void block_center_kernel(const float *__restrict__ lam_q_sorted, int64_t nq, const float *__restrict__ tile_lo,
                                    int ntiles, int32_t *__restrict__ center)
{
    const int qb = blockIdx.x * blockDim.x + threadIdx.x;
    if ((int64_t)qb * TQ >= nq) return;
    const int64_t r0 = (int64_t)qb * TQ, r1 = (r0 + TQ < nq) ? r0 + TQ : nq;
    const float med = lam_q_sorted[(r0 + r1) / 2];
    int lo = 0, hi = ntiles;                                                // first tile with tile_lo > med
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tile_lo[mid] > med) hi = mid; else lo = mid + 1;
    }
    center[qb] = lo > 0 ? lo - 1 : 0;
}

__global__ void gather_f32_kernel(const double *__restrict__ a, const int32_t *__restrict__ perm, int64_t n, float *__restrict__ fa)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        fa[i] = (float)a[perm ? perm[i] : i];
}

// filtered search: vbits[pos] = allowed[perm[pos]] for the nwords * 32 visiting positions (0 from n on)
__global__ void visit_bits_kernel(const uint32_t *__restrict__ allowed, const int32_t *__restrict__ perm, int64_t n, int64_t nwords,
                                  uint32_t *__restrict__ vbits)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp; w < nwords; w += nwarps) {
        const int64_t pos = w * 32 + lane;
        const unsigned word = __ballot_sync(0xffffffffu, pos < n && asp_allowed(allowed, perm[pos]));
        if (lane == 0) vbits[w] = word;
    }
}

// ---- mean direction of the unit vectors (any unit vector keeps the identity below exact; the mean makes the residuals small)
constexpr int MD_BLOCKS = 296;
__global__ void colsum_unit_kernel(const double *__restrict__ x, int64_t n, int f, int pitch, const double *__restrict__ row_scale,
                                   double *__restrict__ partials /* [MD_BLOCKS][f] */)
{
    for (int c = threadIdx.x; c < f; c += blockDim.x) {
        double acc = 0.0;
        for (int64_t r = blockIdx.x; r < n; r += gridDim.x) acc += x[r * pitch + c] * row_scale[r];
        partials[(size_t)blockIdx.x * f + c] = acc;
    }
}

__global__ void mean_dir_kernel(const double *__restrict__ partials, int nblocks, int f, double *__restrict__ mdir)
{
    __shared__ double s_red[256];
    double n2 = 0.0;
    for (int c = threadIdx.x; c < f; c += blockDim.x) {
        double acc = 0.0;
        for (int b = 0; b < nblocks; ++b) acc += partials[(size_t)b * f + c];
        mdir[c] = acc;
        n2 += acc * acc;
    }
    s_red[threadIdx.x] = n2;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) s_red[threadIdx.x] += s_red[threadIdx.x + off];
        __syncthreads();
    }
    const double nrm = sqrt(s_red[0]);
    const double inv = (nrm > 1e-200) ? 1.0 / nrm : 0.0;                 // centred data: m = 0, the residual is the vector itself
    for (int c = threadIdx.x; c < f; c += blockDim.x) mdir[c] *= inv;
}

// One warp per row.  With x^ = x / |x| and the unit vector m:
//     x^ = alpha m + v,  alpha = m.x^,  v orthogonal to m      =>      q^.x^ = beta_q alpha_x + u_q.v_x      (exactly)
// The operand row holds fp16(128 v) in columns [0, f) (its remainder in `lo`, if wanted) and three rank-1 columns at
// [f, f+3): items {a_hi, a_hi, a_lo}, queries {b_hi, b_lo, b_hi} (128 alpha = a_hi + a_lo + O(2^-22)), so that ONE K-major
// contraction over [0, f+3) yields 2^14 (u.v + alpha beta): the rank-1 term to ~2^-21, the residual term to 2^-10 |u||v|
// from a single fp16 term (or 3 2^-22 |u||v| from the two-term split).  rho = |v| feeds the error band.
__global__ void __launch_bounds__(256)
project_split_kernel(const double *__restrict__ x, int64_t n, int f, int pitch, int kp, const double *__restrict__ row_scale,
                     const int32_t *__restrict__ perm, const double *__restrict__ mdir, int is_query,
                     __half *__restrict__ hi, __half *__restrict__ lo, double *__restrict__ rho)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n; r += nwarps) {
        const int64_t src = perm ? (int64_t)perm[r] : r;
        const double sc = row_scale[src];
        const double *row = x + src * pitch;
        double al = 0.0;
        for (int c = lane; c < f; c += 32) al = fma(mdir[c], row[c] * sc, al);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) al += __shfl_xor_sync(0xffffffffu, al, off);
        double r2 = 0.0;
        __half *ph = hi + (size_t)r * kp, *pl = lo ? lo + (size_t)r * kp : nullptr;
        for (int c = lane; c < kp; c += 32) {
            double v = 0.0;
            if (c < f) { v = row[c] * sc - al * mdir[c]; r2 = fma(v, v, r2); }
            const double vs = v * OPERAND_SCALE;
            __half h = __double2half(vs);
            __half l = __double2half(vs - (double)__half2float(h));
            if (c >= f && c < f + 3) {
                const double as = al * OPERAND_SCALE;
                const __half a_hi = __double2half(as);
                const __half a_lo = __double2half(as - (double)__half2float(a_hi));
                const int k = c - f;
                h = is_query ? (k == 1 ? a_lo : a_hi) : (k == 2 ? a_lo : a_hi);
                l = __double2half(0.0);
            }
            ph[c] = h;
            if (pl) pl[c] = l;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) r2 += __shfl_xor_sync(0xffffffffu, r2, off);
        if (lane == 0) rho[r] = sqrt(r2) * (1.0 + 1e-12);
    }
}

// per-row band of the approximate SCORE (f32, visiting order) from the row's residual norm
__global__ void row_delta_kernel(const double *__restrict__ rho_q, int64_t nq, double c_main, double c_fixed, double tau_abs,
                                 double score_slack, float *__restrict__ delta)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nq; i += (int64_t)gridDim.x * blockDim.x)
        delta[i] = __double2float_ru(tau_abs * (rho_q[i] * c_main + c_fixed) + score_slack);
}

// per-row band of the approximate l2 score -d^2~ (f32, visiting order): 2 A B_max |cos~ - cos| plus the f32 roundings of
// the score expression and of the two norms (< 1e-6 (A + B)^2, x2 margin), A = the row's norm
__global__ void row_delta_l2_kernel(const double *__restrict__ rho_q, const double *__restrict__ qnorm, const int32_t *__restrict__ qperm,
                                    int64_t nq, double c_main, double c_fixed, double b_max, float *__restrict__ delta)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nq; i += (int64_t)gridDim.x * blockDim.x) {
        const double a = qnorm[qperm ? qperm[i] : i];
        delta[i] = __double2float_ru(2.0 * a * b_max * (rho_q[i] * c_main + c_fixed) + 2e-6 * (a + b_max) * (a + b_max) + 1e-36);
    }
}

// f32 copies of the lambdas in visiting order + per-tile [min, max] rounded outwards
__global__ void __launch_bounds__(TN) tile_lambda_kernel(const double *__restrict__ lam, const int32_t *__restrict__ perm,
                                                         int64_t n, float *__restrict__ lam32, float *__restrict__ tile_lo,
                                                         float *__restrict__ tile_hi)
{
    const int64_t i = (int64_t)blockIdx.x * TN + threadIdx.x;
    double v = NAN;
    if (i < n) { v = lam[perm[i]]; lam32[i] = (float)v; }
    __shared__ double s_lo[TN], s_hi[TN];
    s_lo[threadIdx.x] = (i < n) ? v : INFINITY;
    s_hi[threadIdx.x] = (i < n) ? v : -INFINITY;
    __syncthreads();
    for (int off = TN / 2; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) {
            s_lo[threadIdx.x] = fmin(s_lo[threadIdx.x], s_lo[threadIdx.x + off]);
            s_hi[threadIdx.x] = fmax(s_hi[threadIdx.x], s_hi[threadIdx.x + off]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { tile_lo[blockIdx.x] = __double2float_rd(s_lo[0]); tile_hi[blockIdx.x] = __double2float_ru(s_hi[0]); }
}

// ------------------------------------------------------------------ descriptors
// K-major operand tile in shared memory, rows of 128 bytes, SWIZZLE_128B (what TMA wrote):
// 8-row groups are 1024 B apart (SBO), LBO unused (1), descriptor version 1 (sm_100).
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// The same for a NARROW K-major tile: rows of `row_bytes` = 32 or 64 bytes (16 / 32 halves, what TMA wrote with
// SWIZZLE_32B / SWIZZLE_64B), 8-row groups 8 * row_bytes apart, layout type 6 / 4 (cute/arch/mma_sm100_desc.hpp).
__device__ __forceinline__ uint64_t make_kmajor_narrow_desc(uint32_t smem_addr, int row_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * row_bytes) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(row_bytes == 32 ? 6 : 4) << 61;
    return d;
}

// kind::f16: D f32 (bit 4), A f16 (bits 7-9 = 0), B f16 (bits 10-12 = 0), both K-major, N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t IDESC_F16_128x256 = (1u << 4) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TQ >> 4) << 24);
constexpr uint32_t IDESC_F16_256x256 = (1u << 4) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)((2 * TQ) >> 4) << 24);   // cta_group::2

// r[j] for a run-time j without local memory.  Called from the rare path, where usually ONE lane of the warp is active.
#ifdef ASP_PICK_SWITCH
#define ASP_PICK_CASE(i) case i: v = r[i]; break;
__device__ __forceinline__ float pick32(const uint32_t (&r)[32], int j)
{
    uint32_t v = 0;
    switch (j) {
        ASP_PICK_CASE(0) ASP_PICK_CASE(1) ASP_PICK_CASE(2) ASP_PICK_CASE(3) ASP_PICK_CASE(4) ASP_PICK_CASE(5) ASP_PICK_CASE(6)
        ASP_PICK_CASE(7) ASP_PICK_CASE(8) ASP_PICK_CASE(9) ASP_PICK_CASE(10) ASP_PICK_CASE(11) ASP_PICK_CASE(12) ASP_PICK_CASE(13)
        ASP_PICK_CASE(14) ASP_PICK_CASE(15) ASP_PICK_CASE(16) ASP_PICK_CASE(17) ASP_PICK_CASE(18) ASP_PICK_CASE(19) ASP_PICK_CASE(20)
        ASP_PICK_CASE(21) ASP_PICK_CASE(22) ASP_PICK_CASE(23) ASP_PICK_CASE(24) ASP_PICK_CASE(25) ASP_PICK_CASE(26) ASP_PICK_CASE(27)
        ASP_PICK_CASE(28) ASP_PICK_CASE(29) ASP_PICK_CASE(30) ASP_PICK_CASE(31)
    }
    return __uint_as_float(v);
}
#undef ASP_PICK_CASE
#else
// a 5-level select tree (31 SEL)
__device__ __forceinline__ float pick32(const uint32_t (&r)[32], int j)
{
    uint32_t a[16], b[8], c[4], d[2];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (j & 16) ? r[i + 16] : r[i];
#pragma unroll
    for (int i = 0; i < 8; ++i) b[i] = (j & 8) ? a[i + 8] : a[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) c[i] = (j & 4) ? b[i + 4] : b[i];
#pragma unroll
    for (int i = 0; i < 2; ++i) d[i] = (j & 2) ? c[i + 2] : c[i];
    return __uint_as_float((j & 1) ? d[1] : d[0]);
}
#endif

struct TcParams {
    int64_t nq, n_local;
    int kp;                       // padded feature count (multiple of 64)
    int nchunks;
    int capb;                     // emission capacity per (query, chunk)
    int topk;
    float tau, beta;              // tau > 0, beta = 1 - tau >= 0
    float score_floor;            // candidates below it are never emitted (kNN: 1 - eps - band; search: -inf)
    const float *delta_q;         // [nq] band of one approximate score of the row (visiting order)
    int nterms;                   // 1: single fp16 term of the residuals; 3: two-term split (lo.hi, hi.lo, hi.hi)
    int kb_lo, kb_hi;             // 64-wide k blocks of the lo terms (residual columns only) / of hi.hi (all columns)
    int sub_lo_last, sub_hi_last; // K=16 MMA steps in the last block of each
    int nw_hi;                    // > 0: the last hi.hi block (it holds the 3 rank-1 columns: 16 useful columns of 64 at F = 384) is
                                  // loaded as a NARROW box of nw_hi = 16 | 32 halves (SWIZZLE_32B | 64B): -11 % operand bytes per tile
    const float *lam_x, *lam_q;   // lam_x in visiting (lambda) order
    const float *tile_lo, *tile_hi;
    const int32_t *perm;          // visiting position -> local item index
    const int32_t *center;        // [query blocks] tile nearest to the block's lambda_q (nullptr: 0)
    uint32_t *theta_glob;         // [nq] ordered bits of the best k-th approximate score any CTA has seen
    float *emit_sc;
    int32_t *emit_ix;
    int32_t *emit_cnt;
    float *dump;                  // DUMP mode: approximate cosines [nq][n_local], local item order
    const uint32_t *vbits;        // FILTER: item mask in visiting order, zero beyond n_local (whole tiles)
    // NT > 1 (tau sweep): ntau (2 .. NT) taus from one pass; tau t reads plane t of delta_q / theta_glob ([nq] each) and
    // writes plane t of emit_sc (`plane` floats each) and of emit_cnt ([nq][nchunks] each); slots t >= ntau hold tau 1, beta 0
// and are never read
    int ntau;
    float taus[asp_sweep::NT_MAX], betas[asp_sweep::NT_MAX], inv_taus[asp_sweep::NT_MAX];
    size_t plane;
};

// ARES (1-term mode, <= 7 k blocks): the query operand (128 x kp fp16, <= 112 KB) is loaded ONCE and stays resident in
// shared memory; only the 32 KB item tiles stream through a 3-stage ring -- a third less L2 -> SM traffic, which is what
// bounds the kernel once the executed FLOP are down to one term.
// PAIR (with ARES): clusters of two CTAs (two query blocks of the same chunk) on the two SMs of a TPC run ONE
// tcgen05.mma.cta_group::2 of M = 256: each CTA keeps its own 128 query rows resident and loads only HALF of every item
// tile (128 of the 256 rows, 16 KB per stage, 6 stages); the leader CTA issues the MMAs, which read both halves and write
// each CTA's rows into its own TMEM.  Half the L2 -> SM item traffic and shared-memory operand reads per SM, twice the
// pipeline depth.  Barriers: TMA loads of both CTAs complete on the LEADER's full barrier; tcgen05.commit multicasts the
// "stage free" / "accumulator ready" arrivals to both CTAs; the peer's epilogue warps arrive remotely on the leader's
// "accumulator drained" barrier.
// L2 (score kind of the Euclidean item graph): the score is -d^2~ (l2_bound.cuh) instead of tau cos~ + beta prox; lam_x /
// lam_q / tile_lo / tile_hi then hold the f32 norms (items in norm order) and the per-(row, tile) raw-accumulator threshold
// comes from asp_l2::threshold instead of the proximity bound.  The MMAs and the pipeline are the same.
// NT > 1: a tau sweep (search only, LISTN 16): the epilogue serves p.ntau <= NT taus from the one set of accumulators.
template <bool DUMP, int VARIANT, bool ARES, bool PAIR, int LISTN, bool L2 = false, bool FILTER = false, int NT = 1>   // LISTN (>= topk): the four column-quarter threads of a query row keep LISTN / 4 scores each; VARIANT (profiling only): 0 normal, 2 epilogue does no work, 3 no MMA issued, 4 epilogue loads TMEM only
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap map_q_hi, const __grid_constant__ CUtensorMap map_q_lo,
               const __grid_constant__ CUtensorMap map_x_hi, const __grid_constant__ CUtensorMap map_x_lo,
               const __grid_constant__ CUtensorMap map_q_nw, const __grid_constant__ CUtensorMap map_x_nw, const TcParams p)
{
    static_assert(!PAIR || ARES, "the CTA-pair kernel keeps the query operand resident");
    static_assert(!L2 || (!DUMP && VARIANT == 0), "the l2 score kind has no dump or profiling variants");
    static_assert(!FILTER || (!L2 && !DUMP && VARIANT == 0), "only the search is filtered");
    static_assert(NT == 1 || (!L2 && !DUMP && VARIANT == 0 && LISTN == 16 && NT <= asp_sweep::NT_MAX), "the tau sweep is a search of k <= 16");
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // SWIZZLE_128B tiles must start on 1024-byte boundaries
    constexpr int NST = PAIR ? 6 : ARES ? 3 : TC_STAGES;                         // ring depth
    constexpr int STB = PAIR ? B_BYTES / 2 : ARES ? B_BYTES : STAGE_BYTES;       // bytes per ring stage
    constexpr int MAXST = 6;
    unsigned char *a_res = smem_raw + ((1024u - (asp::smem_u32(smem_raw) & 1023u)) & 1023u);     // ARES: kb_hi * A_BYTES
    unsigned char *stages = a_res + (ARES ? (size_t)p.kb_hi * A_BYTES : 0);      // NST * STB
    float *s_const = reinterpret_cast<float *>(stages + NST * STB);              // [2][TN]: item lambdas per accumulator
    __shared__ __align__(8) uint64_t full_bar[MAXST], empty_bar[MAXST], tmem_full[2], tmem_empty[2], a_full;
    __shared__ uint32_t s_tmem_base;
    __shared__ uint32_t s_theta[NT * TQ];     // per query row: best k-th score seen by its threads / other CTAs (ordered bits)
    __shared__ int s_cnt[TQ];                 // per query row: emission cursor shared by its column-quarter threads
    __shared__ float s_part[NT * TQ * 4];     // per query row and column quarter: that quarter's ceil(topk/4)-th best score

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qb = blockIdx.x, chunk = blockIdx.y;
    // visiting order of the query block: centre-out from the tile nearest to its lambda_q (descending proximity
    // bound, so the thresholds tighten early); the chunk CTAs of a block take interleaved ranks of that order
    const int tiles_total = (int)((p.n_local + TN - 1) / TN);
    const uint32_t cta_rank = PAIR ? asp::cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const int center = p.center ? p.center[PAIR ? (qb & ~1) : qb] : 0;           // a pair walks ONE tile sequence
    const int side_min = min(center, tiles_total - 1 - center);
    const bool more_below = center > tiles_total - 1 - center;
    const int ntiles = (tiles_total - chunk + p.nchunks - 1) / p.nchunks;        // ranks chunk, chunk + nchunks, ...
    auto tile_of = [&](int t) {
        const int rank = chunk + t * p.nchunks;
        if (rank <= 2 * side_min) { const int j = (rank + 1) >> 1; return (rank & 1) ? center + j : center - j; }
        const int rest = rank - 2 * side_min;
        return more_below ? center - (side_min + rest) : center + (side_min + rest);
    };
    const int klo = (p.nterms == 3) ? p.kb_lo : 0;
    const int kiters = 2 * klo + p.kb_hi;                                        // small terms first, the rank-1 columns last

    if (threadIdx.x == 0) {
        for (int s = 0; s < MAXST; ++s) { asp::mbar_init(&full_bar[s], 1); asp::mbar_init(&empty_bar[s], 1); }
        asp::mbar_init(&a_full, 1);
        for (int a = 0; a < 2; ++a) { asp::mbar_init(&tmem_full[a], 1); asp::mbar_init(&tmem_empty[a], PAIR ? 2 * EPI_WARPS : EPI_WARPS); }
        asp::fence_barrier_init();
    }
    if constexpr (NT == 1) {
        if (threadIdx.x < TQ) { s_theta[threadIdx.x] = 0u; s_cnt[threadIdx.x] = 0; }
        if (threadIdx.x < TQ * 4) s_part[threadIdx.x] = -INFINITY;
    } else {                                                                     // one s_theta / s_part slot per tau
        if (threadIdx.x < TQ) s_cnt[threadIdx.x] = 0;
        for (int i = threadIdx.x; i < NT * TQ; i += TC_THREADS) s_theta[i] = 0u;
        for (int i = threadIdx.x; i < NT * TQ * 4; i += TC_THREADS) s_part[i] = -INFINITY;
    }
    if (warp == 1) { if (PAIR) asp::tmem_alloc_pair(&s_tmem_base, 512); else asp::tmem_alloc(&s_tmem_base, 512); }
    asp::tc_fence_before();
    __syncthreads();
    if (PAIR) asp::cluster_sync_all();                                           // both CTAs' barriers initialised
    asp::tc_fence_after();
    const uint32_t tmem_base = s_tmem_base;

    // Both single-thread roles run as WARP-UNIFORM loops (all 32 lanes walk the tiles and wait on the barriers); only the
    // asynchronous instructions themselves sit under one elected lane.  With the whole role under `if (lane == 0)` the
    // compiler wraps every uniform-datapath instruction (UTMALDG, UTCHMMA, UTCBAR) in an ELECT / BRA.U.ANY loop and the
    // issuing thread needs ~100 instructions per k block -- as long as the 4 MMAs it feeds (ncu: tensor pipe 56 % active,
    // the issuer never waiting for operands).
    if (warp == 0) {
        // ===================== TMA producer =====================
        const bool el = asp::elect_one();
        if (el) {
            asp::tma_prefetch_desc(&map_q_hi); asp::tma_prefetch_desc(&map_q_lo);
            asp::tma_prefetch_desc(&map_x_hi); asp::tma_prefetch_desc(&map_x_lo);
            if (PAIR) {
                // completions of BOTH CTAs' loads are credited to the leader's barriers (only its MMA thread waits)
                const uint32_t a_bar = asp::mapa_shared(asp::smem_u32(&a_full), 0);
                if (leader) asp::mbar_arrive_expect_tx(&a_full, (uint32_t)(2 * p.kb_hi * A_BYTES));
                for (int kb = 0; kb < p.kb_hi; ++kb) asp::tma_load_2d_pair(a_res + (size_t)kb * A_BYTES, &map_q_hi, a_bar, kb * TKB, qb * TQ);
            } else if (ARES) {
                const int a_last = p.nw_hi ? TQ * p.nw_hi * 2 : A_BYTES;             // bytes of the last (maybe narrow) block
                asp::mbar_arrive_expect_tx(&a_full, (uint32_t)((p.kb_hi - 1) * A_BYTES + a_last));
                for (int kb = 0; kb < p.kb_hi; ++kb)
                    asp::tma_load_2d(a_res + (size_t)kb * A_BYTES, (p.nw_hi && kb == p.kb_hi - 1) ? &map_q_nw : &map_q_hi, &a_full, kb * TKB, qb * TQ);
            }
        }
        int s = 0;
        uint32_t ph = 1;                                                         // parity of the "stage free" wait (first round passes)
        for (int t = 0; t < ntiles; ++t) {
            const int item0 = tile_of(t) * TN;
            for (int ki = 0; ki < kiters; ++ki) {
                asp::mbar_wait_suspend(&empty_bar[s], ph, 4000);
                if (el) {
                    const int seg = (ki < klo) ? 0 : (ki < 2 * klo) ? 1 : 2;
                    const int kc = (ki - seg * klo) * TKB;
                    // small terms first: (q_lo, x_hi), (q_hi, x_lo), then (q_hi, x_hi)
                    const CUtensorMap *ma = (seg == 0) ? &map_q_lo : &map_q_hi;
                    const CUtensorMap *mb = (seg == 1) ? &map_x_lo : &map_x_hi;
                    unsigned char *dst = stages + (size_t)s * STB;
                    if (PAIR) {                                                  // this CTA's half of the item tile (map_x_lo = half-box map)
                        if (leader) asp::mbar_arrive_expect_tx(&full_bar[s], 2 * STB);
                        asp::tma_load_2d_pair(dst, &map_x_lo, asp::mapa_shared(asp::smem_u32(&full_bar[s]), 0), kc, item0 + (int)cta_rank * (TN / 2));
                    } else if (p.nw_hi && ki == kiters - 1) {                    // narrow last block of hi.hi
                        asp::mbar_arrive_expect_tx(&full_bar[s], (uint32_t)((ARES ? 0 : TQ * p.nw_hi * 2) + TN * p.nw_hi * 2));
                        if (!ARES) asp::tma_load_2d(dst, &map_q_nw, &full_bar[s], kc, qb * TQ);
                        asp::tma_load_2d(dst + (ARES ? 0 : A_BYTES), &map_x_nw, &full_bar[s], kc, item0);
                    } else {
                        asp::mbar_arrive_expect_tx(&full_bar[s], STB);
                        if (!ARES) asp::tma_load_2d(dst, ma, &full_bar[s], kc, qb * TQ);
                        asp::tma_load_2d(dst + (ARES ? 0 : A_BYTES), mb, &full_bar[s], kc, item0);
                    }
                }
                if (++s == NST) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (PAIR: the leader CTA only) =====================
        if (leader) {
            const bool el = asp::elect_one();
            if (ARES) { asp::mbar_wait(&a_full, 0); asp::tc_fence_after(); }
            int s = 0;
            uint32_t ph = 0;                                                     // parity of the "stage full" wait
            for (int t = 0; t < ntiles; ++t) {
                const int acc = (int)(t & 1);
                asp::mbar_wait(&tmem_empty[acc], (uint32_t)((((t >> 1) & 1)) ^ 1));
                asp::tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * TN);
                for (int ki = 0; ki < kiters; ++ki) {
                    asp::mbar_wait(&full_bar[s], ph);
                    asp::tc_fence_after();
                    if (el) {
                        const uint32_t st_addr = asp::smem_u32(stages + (size_t)s * STB);
                        const uint32_t a_addr = ARES ? asp::smem_u32(a_res + (size_t)ki * A_BYTES) : st_addr;
                        const uint32_t b_addr = ARES ? st_addr : st_addr + A_BYTES;
                        const bool narrow = !PAIR && p.nw_hi && ki == kiters - 1;
                        const uint64_t da = narrow ? make_kmajor_narrow_desc(a_addr, 2 * p.nw_hi) : make_kmajor_sw128_desc(a_addr);
                        const uint64_t db = narrow ? make_kmajor_narrow_desc(b_addr, 2 * p.nw_hi) : make_kmajor_sw128_desc(b_addr);
                        // K = 16 halves per MMA = 32 B = +2 in the address field; the last block of a term may be short
                        const int nsub = (ki == klo - 1 || ki == 2 * klo - 1) ? p.sub_lo_last : (ki == kiters - 1) ? p.sub_hi_last : TKB / 16;
                        if (VARIANT != 3) {
#pragma unroll
                            for (int k = 0; k < TKB / 16; ++k)
                                if (k < nsub) {
                                    if (PAIR) asp::umma_f16_pair(tmem_d, da + 2 * k, db + 2 * k, IDESC_F16_256x256, (ki > 0 || k > 0) ? 1u : 0u);
                                    else asp::umma_f16(tmem_d, da + 2 * k, db + 2 * k, IDESC_F16_128x256, (ki > 0 || k > 0) ? 1u : 0u);
                                }
                        }
                        if (PAIR) asp::umma_commit_pair(&empty_bar[s]); else asp::umma_commit(&empty_bar[s]);   // stage reusable when these MMAs retire
                        if (ki == kiters - 1) { if (PAIR) asp::umma_commit_pair(&tmem_full[acc]); else asp::umma_commit(&tmem_full[acc]); }   // accumulator complete
                    }
                    __syncwarp();
                    if (++s == NST) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if constexpr (NT > 1) {
        // ===================== tau-sweep epilogue: warps 2..17, thread <-> (query row, column quarter) =====================
        // Per tau u, the state of the single-tau epilogue below (running list, theta_k, theta_emit, beta_ub, its s_theta /
        // s_part / theta_glob slot), every update as there.  The common path compares the max tree against the SMALLEST of
        // the taus' raw-accumulator thresholds (sweep_bound.cuh); a column that passes gets its score at every tau, is emitted
        // once if it reaches some tau's theta_emit (index in emit_ix, score u in plane u of emit_sc) and enters every tau's
        // list it beats.  Slots u >= p.ntau start at +inf and never move.  DESIGN §2 item 8.
        const int lg = warp & 3;
        const int part = (warp - 2) >> 2;
        const int row = lg * 32 + lane;
        const int64_t gq = (int64_t)qb * TQ + row;
        const bool qvalid = gq < p.nq;
        const float lq = qvalid ? p.lam_q[gq] : 0.f;
        const int et = threadIdx.x - 64;
        constexpr int PL = LISTN / 4;
        const int rr = (p.topk + 3) >> 2;
        __shared__ float s_delta2[NT * TQ];                                    // 2 x the row's band per tau (needed when theta_k moves)
        __shared__ int s_lost[TQ];                                             // per row: bit u = a record tau u admitted found the buffer full
        if (part == 0) s_lost[row] = 0;
        float theta_k[NT], theta_emit[NT], lst[NT][PL];
        uint32_t nx_go[NT];
#pragma unroll
        for (int u = 0; u < NT; ++u) {
            const bool used = u < p.ntau;
            if (part == 0) s_delta2[u * TQ + row] = (qvalid && used) ? 2.0f * p.delta_q[u * p.nq + gq] : 0.f;
            theta_k[u] = used ? -INFINITY : INFINITY;
            theta_emit[u] = theta_k[u];
            nx_go[u] = 0u;
#pragma unroll
            for (int i = 0; i < PL; ++i) lst[u][i] = (!used || i < PL - rr) ? INFINITY : -INFINITY;
        }
        const size_t ebase = ((size_t)gq * p.nchunks + chunk) * (size_t)p.capb;
        float nx_lam = 0.f, nx_tl = 0.f, nx_th = 0.f;
        auto prefetch = [&](int t) {
            if (t >= ntiles) return;
            const int tile = tile_of(t);
            if (et < TN) { const int64_t n = (int64_t)tile * TN + et; nx_lam = (n < p.n_local) ? p.lam_x[n] : 0.f; }
            nx_tl = p.tile_lo[tile];
            nx_th = p.tile_hi[tile];
            if (part == 0 && qvalid) {
#pragma unroll
                for (int u = 0; u < NT; ++u)
                    if (u < p.ntau) nx_go[u] = p.theta_glob[u * p.nq + gq];
            }
        };
        prefetch(0);
        for (int t = 0; t < ntiles; ++t) {
            const int acc = (int)(t & 1);
            const int tile = tile_of(t);
            const int64_t item0 = (int64_t)tile * TN;
            float *c_lam = s_const + acc * TN;
            if (et < TN) c_lam[et] = nx_lam;
            const float tl = nx_tl, th = nx_th;
            if (part == 0 && qvalid) {
#pragma unroll
                for (int u = 0; u < NT; ++u)
                    if (nx_go[u] > s_theta[u * TQ + row]) atomicMax(&s_theta[u * TQ + row], nx_go[u]);
            }
            asm volatile("bar.sync 1, %0;\n" ::"n"(EPI_WARPS * 32) : "memory");    // epilogue warps only
            prefetch(t + 1);
            float theta_acc = INFINITY;
            const float pb = asp_sweep::prox_bound(lq, tl, th);
            if (qvalid) {
#pragma unroll
                for (int u = 0; u < NT; ++u) {
                    const uint32_t so = s_theta[u * TQ + row];
                    if (so != 0u) {
                        const float sh = o2f(so);
                        if (sh > theta_k[u]) { theta_k[u] = sh; theta_emit[u] = theta_k[u] - s_delta2[u * TQ + row]; }
                    }
                }
                theta_acc = asp_sweep::combined_threshold(theta_emit, p.betas, p.inv_taus, pb, NT);
            }
            asp::mbar_wait_suspend(&tmem_full[acc], (uint32_t)((t >> 1) & 1), 8000);
            asp::tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < EPI_COLS / 32; ++c) {
                const int col0 = part * EPI_COLS + c * 32;
                uint32_t r[32];
                asp::tmem_ld_32x32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(acc * TN + col0), r);
                asp::tmem_ld_wait();
                float m[16];                                                     // common path: a max tree and one compare
#pragma unroll
                for (int j = 0; j < 16; ++j) m[j] = fmaxf(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
#pragma unroll
                for (int w = 8; w > 0; w >>= 1)
#pragma unroll
                    for (int j = 0; j < w; ++j) m[j] = fmaxf(m[j], m[j + w]);
                if (m[0] < theta_acc) continue;
                uint32_t mask = 0;
#pragma unroll
                for (int j = 0; j < 32; ++j) mask |= (__uint_as_float(r[j]) >= theta_acc) ? (1u << j) : 0u;
                if constexpr (FILTER) mask &= p.vbits[(item0 + col0) >> 5];
                while (mask) {
                    const int j = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const float a = pick32(r, j);
                    if (a < theta_acc) continue;                                 // the threshold rose inside this loop
                    const int col = col0 + j;
                    const int64_t n = item0 + col;
                    if (n >= p.n_local) continue;
                    const float px = asp_sweep::prox(lq, c_lam[col]);
                    float sc[NT];
                    uint32_t adm = 0;                                            // the taus whose threshold admits the column
#pragma unroll
                    for (int u = 0; u < NT; ++u) {
                        sc[u] = asp_sweep::score(p.taus[u], p.betas[u], px, a);
                        adm |= (sc[u] >= theta_emit[u]) ? (1u << u) : 0u;
                    }
                    if (!adm) continue;
                    const int pos = atomicAdd(&s_cnt[row], 1);
                    if (pos < p.capb) {
                        p.emit_ix[ebase + pos] = p.perm[n];
#pragma unroll
                        for (int u = 0; u < NT; ++u)
                            if (u < p.ntau) p.emit_sc[u * p.plane + ebase + pos] = sc[u];
                    } else {
                        atomicOr(&s_lost[row], (int)adm);
                    }
                    bool raised = false;
#pragma unroll
                    for (int u = 0; u < NT; ++u) {
                        if (!(sc[u] > lst[u][PL - 1])) continue;
                        float v = sc[u];                                         // sorted insertion
#pragma unroll
                        for (int i = 0; i < PL; ++i) {
                            const float o = lst[u][i];
                            const bool sw = v > o;
                            lst[u][i] = sw ? v : o;
                            v = sw ? o : v;
                        }
                        volatile float *my_part = s_part + (u * TQ + row) * 4;
                        my_part[part] = lst[u][PL - 1];                          // a stale (lower) value read by the others is still valid
                        const float kth = fminf(fminf(my_part[0], my_part[1]), fminf(my_part[2], my_part[3]));
                        if (kth > theta_k[u]) {
                            theta_k[u] = kth;
                            theta_emit[u] = theta_k[u] - s_delta2[u * TQ + row];
                            raised = true;
                            const uint32_t ko = f2o(kth);
                            atomicMax(&s_theta[u * TQ + row], ko);
                            atomicMax(&p.theta_glob[u * p.nq + gq], ko);
                        }
                    }
                    if (raised) theta_acc = asp_sweep::combined_threshold(theta_emit, p.betas, p.inv_taus, pb, NT);
                }
            }
            asp::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (PAIR) asp::mbar_arrive_cluster(asp::mapa_shared(asp::smem_u32(&tmem_empty[acc]), 0));   // the leader's MMA thread waits
                else asp::mbar_arrive(&tmem_empty[acc]);
            }
        }
        asm volatile("bar.sync 1, %0;\n" ::"n"(EPI_WARPS * 32) : "memory");
        if (qvalid && part == 0) {
            // one count plane per tau: the overflow (count > capb) only for a tau that lost a record it admitted; the other
            // taus keep every record their own thresholds asked for, and stage 2 reads the capb that were written
            const int cnt = s_cnt[row], lost = s_lost[row];
#pragma unroll
            for (int u = 0; u < NT; ++u)
                if (u < p.ntau) p.emit_cnt[(u * p.nq + gq) * p.nchunks + chunk] = ((lost >> u) & 1) ? cnt : min(cnt, p.capb);
        }
    } else {
        // ===================== epilogue: warps 2..17, thread <-> (query row, column quarter) =====================
        const int lg = warp & 3;                                                 // TMEM lane group this warp may touch
        const int part = (warp - 2) >> 2;                                        // which EPI_COLS columns of the tile
        const int row = lg * 32 + lane;
        const int64_t gq = (int64_t)qb * TQ + row;
        const bool qvalid = gq < p.nq;
        const float lq = qvalid ? p.lam_q[gq] : 0.f;
        const int et = threadIdx.x - 64;                                         // 0 .. EPI_WARPS*32-1
        const float inv_tau = 1.0f / p.tau;
        const float delta2 = (qvalid && !DUMP) ? 2.0f * p.delta_q[gq] : 0.f;
        // Running threshold of a query row: its four threads (column quarters) each keep the best rr = ceil(topk / 4) scores of
        // THEIR columns; 4 rr >= topk distinct items score at least m = min over the quarters of the rr-th best, so m is a valid
        // lower bound of the row's topk-th best -- about the (topk + 4)-th best overall, where a full list per quarter would
        // only give the 4 topk-th.  lst[PL-1] is the rr-th best (the slots in front of the real ones hold +inf and never move).
        constexpr int PL = LISTN / 4;
        const int rr = (p.topk + 3) >> 2;
        float lst[PL];
#pragma unroll
        for (int i = 0; i < PL; ++i) lst[i] = (i < PL - rr) ? INFINITY : -INFINITY;
        volatile float *my_part = s_part + row * 4;
        const float floor_row = p.score_floor - 0.5f * delta2;                    // exact-score floor minus the row's band (-inf: none)
        float theta_k = -INFINITY, theta_emit = floor_row;
        const size_t ebase = ((size_t)gq * p.nchunks + chunk) * (size_t)p.capb;

        // per-tile inputs are fetched one tile AHEAD (registers), so their global-memory latency hides behind the previous
        // tile's accumulator wait and processing instead of delaying the release of the accumulator
        float nx_lam = 0.f, nx_tl = 0.f, nx_th = 0.f;
        uint32_t nx_go = 0u;
        auto prefetch = [&](int t) {
            if (t >= ntiles) return;
            const int tile = tile_of(t);
            if (et < TN) { const int64_t n = (int64_t)tile * TN + et; nx_lam = (n < p.n_local) ? p.lam_x[n] : 0.f; }
            if (!DUMP) {
                nx_tl = p.tile_lo[tile];
                nx_th = p.tile_hi[tile];
                if (part == 0 && qvalid) nx_go = p.theta_glob[gq];
            }
        };
        prefetch(0);
        for (int t = 0; t < ntiles; ++t) {
            const int acc = (int)(t & 1);
            const int tile = tile_of(t);
            const int64_t item0 = (int64_t)tile * TN;
            float *c_lam = s_const + acc * TN;
            if (et < TN) c_lam[et] = nx_lam;
            const float tl = nx_tl, th = nx_th;
            if (!DUMP && part == 0 && qvalid && nx_go > s_theta[row]) atomicMax(&s_theta[row], nx_go);   // other chunks' thresholds
            asm volatile("bar.sync 1, %0;\n" ::"n"(EPI_WARPS * 32) : "memory");    // epilogue warps only
            prefetch(t + 1);
            float theta_acc = qvalid ? -INFINITY : INFINITY;                     // raw-accumulator filter of this (row, tile)
            float beta_ub = p.beta;
            if (!DUMP && qvalid) {
                const uint32_t so = s_theta[row];
                if (so != 0u) {
                    const float sh = o2f(so);
                    if (sh > theta_k) { theta_k = sh; theta_emit = fmaxf(theta_k - delta2, floor_row); }
                }
                if constexpr (L2) {
                    // lq = the row's norm, [tl, th] = the tile's norm interval: the smallest cos~ a column needs to reach
                    // theta_emit (l2_bound.cuh).  It is not refreshed when theta_emit rises inside the tile (stale = lower = safe).
                    theta_acc = asp_l2::threshold(lq, tl, th, theta_emit);
                } else {
                // s <= tau*cos + beta*prox_ub, prox_ub = 1/(1 + distance of lambda_q to the tile's lambda interval);
                // the 2.5e-7 / 1.000001 keep the bound safe against the f32 roundings of lambda_q and the interval
                const float gap = fmaxf(0.f, fmaxf(lq - th, tl - lq) - 2.5e-7f);
                beta_ub = p.beta * __fdividef(1.0f, 1.0f + gap) * 1.000001f;
                theta_acc = ((theta_emit - beta_ub) * inv_tau - 1e-6f) * ACC_SCALE;
                }
            }
            asp::mbar_wait_suspend(&tmem_full[acc], (uint32_t)((t >> 1) & 1), 8000);
            asp::tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < ((VARIANT == 2 || VARIANT == 3) ? 0 : EPI_COLS / 32); ++c) {
                const int col0 = part * EPI_COLS + c * 32;
                uint32_t r[32];
                asp::tmem_ld_32x32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(acc * TN + col0), r);
                asp::tmem_ld_wait();
                if (VARIANT == 4) continue;
                if (DUMP) {
                    if (qvalid) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int64_t n = item0 + col0 + j;
                            if (n < p.n_local) p.dump[gq * p.n_local + p.perm[n]] = __uint_as_float(r[j]) * (1.0f / ACC_SCALE);
                        }
                    }
                } else {
                    // common path: a max tree and one compare
                    float m[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) m[j] = fmaxf(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
#pragma unroll
                    for (int w = 8; w > 0; w >>= 1)
#pragma unroll
                        for (int j = 0; j < w; ++j) m[j] = fmaxf(m[j], m[j + w]);
                    if (m[0] >= theta_acc) {
                        // rare path: the columns that pass, one at a time (registers cannot be indexed: select tree)
                        uint32_t mask = 0;
#pragma unroll
                        for (int j = 0; j < 32; ++j) mask |= (__uint_as_float(r[j]) >= theta_acc) ? (1u << j) : 0u;
                        if constexpr (FILTER) mask &= p.vbits[(item0 + col0) >> 5];       // col0 % 32 == 0: one word
                        while (mask) {
                            const int j = __ffs(mask) - 1;
                            mask &= mask - 1;
                            const float a = pick32(r, j);
                            if (a < theta_acc) continue;                         // the threshold rose inside this loop
                            const int col = col0 + j;
                            const int64_t n = item0 + col;
                            const float sc = L2 ? asp_l2::score(lq, c_lam[col], a)
                                                : fmaf(p.beta, __fdividef(1.0f, 1.0f + fabsf(lq - c_lam[col])), p.tau * (a * (1.0f / ACC_SCALE)));
                            if (sc >= theta_emit && n < p.n_local) {
                                const int pos = atomicAdd(&s_cnt[row], 1);
                                if (pos < p.capb) { p.emit_sc[ebase + pos] = sc; p.emit_ix[ebase + pos] = p.perm[n]; }
                                if (sc > lst[PL - 1]) {
                                    float v = sc;                                // sorted insertion
#pragma unroll
                                    for (int i = 0; i < PL; ++i) {
                                        const float o = lst[i];
                                        const bool sw = v > o;
                                        lst[i] = sw ? v : o;
                                        v = sw ? o : v;
                                    }
                                    my_part[part] = lst[PL - 1];                 // a stale (lower) value read by the others is still valid
                                    const float kth = fminf(fminf(my_part[0], my_part[1]), fminf(my_part[2], my_part[3]));
                                    if (kth > theta_k) {
                                        theta_k = kth;
                                        theta_emit = fmaxf(theta_k - delta2, floor_row);
                                        if constexpr (!L2) theta_acc = ((theta_emit - beta_ub) * inv_tau - 1e-6f) * ACC_SCALE;
                                        const uint32_t ko = f2o(kth);
                                        atomicMax(&s_theta[row], ko);
                                        atomicMax(&p.theta_glob[gq], ko);
                                    }
                                }
                            }
                        }
                    }
                }
            }
            asp::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (PAIR) asp::mbar_arrive_cluster(asp::mapa_shared(asp::smem_u32(&tmem_empty[acc]), 0));   // the leader's MMA thread waits
                else asp::mbar_arrive(&tmem_empty[acc]);
            }
        }
        asm volatile("bar.sync 1, %0;\n" ::"n"(EPI_WARPS * 32) : "memory");
        if (!DUMP && qvalid && part == 0) p.emit_cnt[gq * p.nchunks + chunk] = s_cnt[row];
    }
    asp::tc_fence_before();
    __syncthreads();
    if (PAIR) asp::cluster_sync_all();                                           // the leader's MMAs read the peer's shared memory
    if (warp == 1) { if (PAIR) asp::tmem_dealloc_pair(tmem_base, 512); else asp::tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------ stage 2
__device__ __forceinline__ double exact_score_tc(double dot, double nq, double nx, double tau, double lq, double lx)
{
    const double den = __dmul_rn(nq, nx);
    const double c = (den == 0.0) ? 0.0 : __ddiv_rn(dot, den);
    const double prox = __ddiv_rn(1.0, __dadd_rn(1.0, fabs(__dsub_rn(lq, lx))));
    return __dadd_rn(__dmul_rn(tau, c), __dmul_rn(__dsub_rn(1.0, tau), prox));
}

__device__ __forceinline__ double seq_dot_row_tc(const double *__restrict__ qv, const double *__restrict__ row, int f)
{
    double d = 0.0;
    int j = 0;
    for (; j + 16 <= f; j += 16) {                                               // 8 loads in flight, then the ordered sum
        double2 x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) x[u] = *reinterpret_cast<const double2 *>(row + j + 2 * u);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            d = __dadd_rn(d, __dmul_rn(qv[j + 2 * u], x[u].x));
            d = __dadd_rn(d, __dmul_rn(qv[j + 2 * u + 1], x[u].y));
        }
    }
    for (; j < f; ++j) d = __dadd_rn(d, __dmul_rn(qv[j], row[j]));
    return d;
}

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

constexpr int TR_WARPS = 4;
constexpr int TR_MIN_CTAS = 8;    // throughput shape: 32 resident warps per SM (64 registers per thread)
constexpr int TR_QUEUE = 96;       // survivor queue per warp (flushed in batches of 32)

// WPQ warps per query.  See the header: (A) coalesced f64 re-scoring of every survivor, best 32 kept;
// (B) reference-order re-scoring of the candidates within 2*eps_fast of the k-th best; sort; emit.
// WPQ == 1 (throughput shape): TR_WARPS independent queries per CTA.  WPQ > 1 (latency shape, small batches such as the
// reference's one-query-per-call `search`): one CTA per query, warp w takes the emission streams w, w + WPQ, ...; the
// per-warp top lists are merged pairwise through shared memory.  Every quantity that decides the result (cut-off, fast
// scores, the 32 kept, the band) is a function of the SET of emitted candidates, so all WPQ give bit-identical output.
template <int WPQ, int MINB = 1>   // MINB: resident CTAs per SM the register allocation must allow
__global__ void __launch_bounds__((WPQ == 1 ? TR_WARPS : WPQ) * 32, MINB)
tc_rescore_kernel(const double *__restrict__ q, int qpitch, int64_t nq, const double *__restrict__ items, int64_t n_local,
                  int f, int pitch, int64_t row0, const double *__restrict__ norm_x, const double *__restrict__ lam_x,
                  const double *__restrict__ norm_q, const double *__restrict__ lam_q, double tau, int topk, int nstreams,
                  int capb, const float *__restrict__ delta_q, double eps_fast, const float *__restrict__ emit_sc,
                  const int32_t *__restrict__ emit_ix, const int32_t *__restrict__ emit_cnt,
                  const uint32_t *__restrict__ theta_glob, const int32_t *__restrict__ qperm,
                  int64_t *__restrict__ out_idx, double *__restrict__ out_score,
                  int32_t *slow_list, int32_t *slow_count, unsigned long long *survivor_total, unsigned long long *exact_total)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    constexpr int NWARPS = (WPQ == 1) ? TR_WARPS : WPQ;
    constexpr int QCOPIES = (WPQ == 1) ? TR_WARPS : 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wq = (WPQ == 1) ? 0 : warp;                                        // this warp's rank within its query
    double *qs = reinterpret_cast<double *>(smem_raw) + (size_t)((WPQ == 1) ? warp : 0) * pitch;   // zero padded to the item pitch
    int32_t *queue = reinterpret_cast<int32_t *>(reinterpret_cast<double *>(smem_raw) + (size_t)QCOPIES * pitch) + warp * TR_QUEUE;
    // merge areas of the latency shape (unused when WPQ == 1)
    double *x_s = reinterpret_cast<double *>(smem_raw) + (size_t)QCOPIES * pitch + (size_t)(NWARPS * TR_QUEUE) / 2;
    int32_t *x_i = reinterpret_cast<int32_t *>(x_s + NWARPS * 32);
    float *x_f = reinterpret_cast<float *>(x_i + NWARPS * 32);
    __shared__ float s_cutoff;
    __shared__ unsigned long long s_nsurv;
    const int64_t qi = (WPQ == 1) ? (int64_t)blockIdx.x * TR_WARPS + warp : (int64_t)blockIdx.x;   // position in lambda_q order
    if (qi >= nq) return;
    const int64_t oq = qperm ? (int64_t)qperm[qi] : qi;                          // the caller's query index
    if (WPQ == 1) {
        for (int j = lane; j < pitch; j += 32) qs[j] = (j < f) ? q[oq * qpitch + j] : 0.0;
    } else {
        for (int j = threadIdx.x; j < pitch; j += NWARPS * 32) qs[j] = (j < f) ? q[oq * qpitch + j] : 0.0;
        if (threadIdx.x == 0) s_nsurv = 0ull;
    }

    bool overflow = false;
    if (WPQ == 1) {
        for (int c = lane; c < nstreams; c += 32) overflow |= emit_cnt[qi * nstreams + c] > capb;
        overflow = __any_sync(0xffffffffu, overflow);
    } else {
        for (int c = threadIdx.x; c < nstreams; c += NWARPS * 32) overflow |= emit_cnt[qi * nstreams + c] > capb;
        overflow = __syncthreads_or(overflow ? 1 : 0) != 0;                      // also publishes qs / s_nsurv
    }
    if (overflow) {                                                              // uniform over the query's warps
        if (lane == 0 && wq == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)oq;
        return;
    }
    // final cut: the k-th largest approximate score over ALL emitted candidates of the query (distinct items, so it is
    // a valid threshold, and the tightest one: the in-kernel thresholds only see one thread's share of the items)
    const int kk = topk < n_local ? topk : (int)n_local;
    float cutoff;
    {
        float top[2] = {-INFINITY, -INFINITY};                                   // best 32 in top[0], sorted descending by lane
        float floor32 = -INFINITY;                                               // 32nd best so far
        for (int c = wq; c < nstreams; c += WPQ) {
            const int cnt = emit_cnt[qi * nstreams + c];
            const size_t base = ((size_t)qi * nstreams + c) * (size_t)capb;
            for (int e0 = 0; e0 < cnt; e0 += 128) {                              // four loads in flight per lane
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { const int e = e0 + 32 * u + lane; v[u] = (e < cnt) ? emit_sc[base + e] : -INFINITY; }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (!__any_sync(0xffffffffu, v[u] > floor32)) continue;
                    top[1] = v[u];
                    asp::warp_sort_desc_f32x2(top, lane);
                    floor32 = __shfl_sync(0xffffffffu, top[0], 31);
                }
            }
        }
        if (WPQ > 1) {                                                           // pairwise merge of the warps' sorted lists
            x_f[warp * 32 + lane] = top[0];
            __syncthreads();
#pragma unroll 1
            for (int step = 1; step < WPQ; step <<= 1) {
                if ((warp & (2 * step - 1)) == 0 && warp + step < WPQ) {
                    top[1] = x_f[(warp + step) * 32 + lane];
                    asp::warp_sort_desc_f32x2(top, lane);
                    x_f[warp * 32 + lane] = top[0];
                }
                __syncthreads();
            }
            if (warp == 0) {
                const float kth = __shfl_sync(0xffffffffu, top[0], kk - 1);
                if (lane == 0) s_cutoff = kth - 2.0f * delta_q[qi];
            }
            __syncthreads();
            cutoff = s_cutoff;
        } else {
            const float kth = __shfl_sync(0xffffffffu, top[0], kk - 1);          // -inf when fewer than kk were emitted
            cutoff = kth - 2.0f * delta_q[qi];
        }
    }
    (void)theta_glob;
    const double nqv = norm_q[oq], lqv = lam_q[oq];
    __syncwarp();

    Cand best[2];
    best[0] = asp::cand_empty();
    best[1] = asp::cand_empty();
    int qn = 0;                                                                  // queued survivors (warp uniform)
    unsigned long long nsurv = 0;
    // (A): `count` queued survivors, four rows at a time, every lane a slice of the features (coalesced 16 B loads)
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
                const double2 qq = *reinterpret_cast<const double2 *>(qs + j);
                double2 a[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) a[u] = *reinterpret_cast<const double2 *>(rr[u] + j);
#pragma unroll
                for (int u = 0; u < 4; ++u) { d[u] = fma(qq.x, a[u].x, d[u]); d[u] = fma(qq.y, a[u].y, d[u]); }
            }
            const double tot = warp_sum4_transposed(d, lane);                    // lanes 8u .. 8u+7: the dot of row s0 + u
            const int u_mine = lane - s0;                                        // lanes s0 .. s0+3 keep one result each
            const double dd = __shfl_sync(0xffffffffu, tot, 8 * (u_mine & 3));
            if (u_mine >= 0 && u_mine < 4 && lane < count) {
                my_dot = dd;
                my_item = (u_mine == 0) ? ii[0] : (u_mine == 1) ? ii[1] : (u_mine == 2) ? ii[2] : ii[3];
            }
        }
        if (my_item >= 0) {                                                      // one score per lane, all lanes at once
            mine.s = exact_score_tc(my_dot, nqv, norm_x[my_item], tau, lqv, lam_x[my_item]);
            mine.i = my_item;
        }
        best[1] = mine;
        asp::warp_sort_best_first<2>(best, lane);
    };
    for (int c = wq; c < nstreams; c += WPQ) {
        const int cnt = emit_cnt[qi * nstreams + c];
        const size_t base = ((size_t)qi * nstreams + c) * (size_t)capb;
        for (int e0 = 0; e0 < cnt; e0 += 128) {                                  // four loads in flight per lane
            float sc4[4];
            int32_t ix4[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + 32 * u + lane;
                sc4[u] = (e < cnt) ? emit_sc[base + e] : -INFINITY;
                ix4[u] = (e < cnt) ? emit_ix[base + e] : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + 32 * u + lane;
                const bool keep = (e < cnt) && (sc4[u] >= cutoff);
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                if (m == 0u) continue;
                if (keep) queue[qn + __popc(m & ((1u << lane) - 1))] = ix4[u];
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
    }
    if (qn > 0) { flush(qn); nsurv += qn; }

    if (WPQ > 1) {                                                               // pairwise merge of the warps' best-32 lists
        x_s[warp * 32 + lane] = best[0].s;
        x_i[warp * 32 + lane] = best[0].i;
        if (lane == 0) atomicAdd(&s_nsurv, nsurv);
        __syncthreads();
#pragma unroll 1
        for (int step = 1; step < WPQ; step <<= 1) {
            if ((warp & (2 * step - 1)) == 0 && warp + step < WPQ) {
                best[1].s = x_s[(warp + step) * 32 + lane];
                best[1].i = x_i[(warp + step) * 32 + lane];
                asp::warp_sort_best_first<2>(best, lane);
                x_s[warp * 32 + lane] = best[0].s;
                x_i[warp * 32 + lane] = best[0].i;
            }
            __syncthreads();
        }
        if (warp != 0) return;
        nsurv = s_nsurv;
    }

    // (B): candidates whose fast score is within 2 eps of the k-th best fast score
    const double kth = __shfl_sync(0xffffffffu, best[0].s, kk - 1);              // -inf when fewer than kk survivors
    const bool valid = best[0].i != 0x7fffffff;
    const bool in_band = valid && (best[0].s >= kth - 2.0 * eps_fast);
    const unsigned band = __ballot_sync(0xffffffffu, in_band);
    if (band == 0xffffffffu || __popc(band) < kk) {
        // the band may extend beyond the 32 kept (long runs of ties), or the emission was short: exact scan
        if (lane == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)oq;
        return;
    }
    Cand fin[1];
    fin[0] = asp::cand_empty();
    if (in_band) {
        const int64_t it = best[0].i;
        const double d = seq_dot_row_tc(qs, items + it * pitch, f);
        fin[0].s = exact_score_tc(d, nqv, norm_x[it], tau, lqv, lam_x[it]);
        fin[0].i = (int32_t)it;
    }
    asp::warp_sort_best_first<1>(fin, lane);
    if (lane == 0) { atomicAdd(survivor_total, nsurv); atomicAdd(exact_total, (unsigned long long)__popc(band)); }
    if (lane < topk) {
        const bool ok = (lane < kk) && fin[0].i != 0x7fffffff;
        out_idx[oq * topk + lane] = ok ? row0 + fin[0].i : -1;
        out_score[oq * topk + lane] = ok ? fin[0].s : NAN;
    }
}

constexpr int TW_THREADS = 256;
static_assert(TW_THREADS == 256, "one thread per radix digit");

// block-wide bitonic sort of n (a power of two) (key, index) pairs in shared memory
__device__ __forceinline__ void block_bitonic(uint64_t *key, int32_t *ix, int n)
{
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < n / 2; t += TW_THREADS) asp_lk::bitonic_cx(key, ix, t, size, stride);
            __syncthreads();
        }
}

// Wide stage 2 (k = 32 .. 128, the _k entry points): one CTA per query, every survivor of the cut kept in shared memory.
// The phases and their reasons are in large_k.cuh.  Dynamic shared memory: the query row (pitch doubles), then SURV_CAP
// sort keys and SURV_CAP item indices.
__global__ void __launch_bounds__(TW_THREADS)
tc_rescore_wide_kernel(const double *__restrict__ q, int qpitch, const double *__restrict__ items, int64_t n_local, int f,
                       int pitch, int64_t row0, const double *__restrict__ norm_x, const double *__restrict__ lam_x,
                       const double *__restrict__ norm_q, const double *__restrict__ lam_q, double tau, int topk, int nstreams,
                       int capb, const float *__restrict__ delta_q, double eps_fast, const float *__restrict__ emit_sc,
                       const int32_t *__restrict__ emit_ix, const int32_t *__restrict__ emit_cnt, const int32_t *__restrict__ qperm,
                       int64_t *__restrict__ out_idx, double *__restrict__ out_score, int32_t *slow_list, int32_t *slow_count,
                       unsigned long long *survivor_total, unsigned long long *exact_total)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    double *qs = reinterpret_cast<double *>(smem_raw);
    uint64_t *key = reinterpret_cast<uint64_t *>(qs + pitch);
    int32_t *ix = reinterpret_cast<int32_t *>(key + asp_lk::SURV_CAP);
    __shared__ int s_hist[256];
    __shared__ int s_krem, s_nsurv;
    __shared__ uint32_t s_prefix;
    __shared__ unsigned long long s_emitted;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t qi = blockIdx.x;                                               // position in lambda_q order
    const int64_t oq = qperm ? (int64_t)qperm[qi] : qi;
    const int kk = topk < n_local ? topk : (int)n_local;
    for (int j = tid; j < pitch; j += TW_THREADS) qs[j] = (j < f) ? q[oq * qpitch + j] : 0.0;
    if (tid == 0) { s_emitted = 0ull; s_nsurv = 0; s_prefix = 0u; s_krem = kk; }
    bool overflow = false;
    unsigned long long mine = 0;
    for (int c = tid; c < nstreams; c += TW_THREADS) {
        const int cnt = emit_cnt[qi * nstreams + c];
        overflow |= cnt > capb;
        mine += (unsigned long long)cnt;
    }
    overflow = __syncthreads_or(overflow ? 1 : 0) != 0;
    if (overflow) {
        if (tid == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)oq;
        return;
    }
    if (mine) atomicAdd(&s_emitted, mine);
    __syncthreads();
    const int64_t emitted = (int64_t)s_emitted;

    // (1) cut: radix select of the kk-th largest approximate score over every emitted candidate
    float cutoff = -INFINITY;
    if (emitted >= kk) {
        for (int pass = 0; pass < 4; ++pass) {
            s_hist[tid] = 0;                                                     // TW_THREADS == 256 digits
            __syncthreads();
            const uint32_t prefix = s_prefix;
            for (int c = 0; c < nstreams; ++c) {
                const int cnt = emit_cnt[qi * nstreams + c];
                const float *sc = emit_sc + ((size_t)qi * nstreams + c) * (size_t)capb;
                for (int e = tid; e < cnt; e += TW_THREADS) {
                    const uint32_t k = asp_lk::f32_key(sc[e]);
                    if (asp_lk::prefix_match(k, prefix, pass)) atomicAdd(&s_hist[asp_lk::digit(k, pass)], 1);
                }
            }
            __syncthreads();
            if (tid == 0) {
                int kr = s_krem;
                const int d = asp_lk::select_digit(s_hist, &kr);
                s_krem = kr;
                s_prefix = prefix | ((uint32_t)d << (24 - 8 * pass));
            }
            __syncthreads();
        }
        cutoff = asp_lk::survivor_cutoff(s_prefix, delta_q[qi]);
    }

    // (2) survivors of the cut (their order here depends on the schedule; the sorts below make it irrelevant)
    for (int c = 0; c < nstreams; ++c) {
        const int cnt = emit_cnt[qi * nstreams + c];
        const size_t base = ((size_t)qi * nstreams + c) * (size_t)capb;
        for (int e = tid; e < cnt; e += TW_THREADS)
            if (emit_sc[base + e] >= cutoff) {
                const int pos = atomicAdd(&s_nsurv, 1);
                if (pos < asp_lk::SURV_CAP) ix[pos] = emit_ix[base + e];
            }
    }
    __syncthreads();
    const int nsurv = s_nsurv;
    if (asp_lk::route(false, emitted, nsurv, kk) != asp_lk::ROUTE_OK) {
        if (tid == 0) slow_list[atomicAdd(slow_count, 1)] = (int32_t)oq;
        return;
    }

    // (3) f64 re-score of every survivor (one warp per survivor, coalesced 16 B loads), sort by (fast desc, index asc)
    const double nqv = norm_q[oq], lqv = lam_q[oq];
    for (int s = warp; s < nsurv; s += TW_THREADS / 32) {
        const int it = ix[s];
        const double *row = items + (int64_t)it * pitch;
        double d = 0.0;
        for (int j = 2 * lane; j < pitch; j += 64) {
            const double2 qq = *reinterpret_cast<const double2 *>(qs + j);
            const double2 a = *reinterpret_cast<const double2 *>(row + j);
            d = fma(qq.x, a.x, d);
            d = fma(qq.y, a.y, d);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
        if (lane == 0) key[s] = asp_range::desc_key(exact_score_tc(d, nqv, norm_x[it], tau, lqv, lam_x[it]));
    }
    const int n2 = asp_lk::next_pow2(nsurv);
    for (int s = nsurv + tid; s < n2; s += TW_THREADS) { key[s] = ~0ull; ix[s] = 0x7fffffff; }
    __syncthreads();
    block_bitonic(key, ix, n2);

    // (4) the band of the kk-th best fast score (a prefix of the sorted survivors), in the reference order
    int nb = 0;
    for (int i0 = 0; i0 < nsurv; i0 += TW_THREADS) {
        const int i = i0 + tid;
        const int cnt = __syncthreads_count(i < nsurv && asp_lk::in_band(key, i, kk, eps_fast));
        nb += cnt;
        if (cnt < TW_THREADS) break;
    }
    __syncthreads();                                                             // every thread has read the fast keys
    const int n3 = asp_lk::next_pow2(nb);
    for (int i = tid; i < n3; i += TW_THREADS) {
        if (i < nb) {
            const int it = ix[i];
            const double d = seq_dot_row_tc(qs, items + (int64_t)it * pitch, f);
            key[i] = asp_range::desc_key(exact_score_tc(d, nqv, norm_x[it], tau, lqv, lam_x[it]));
        } else {
            key[i] = ~0ull;
            ix[i] = 0x7fffffff;
        }
    }
    __syncthreads();
    block_bitonic(key, ix, n3);
    for (int j = tid; j < topk; j += TW_THREADS) asp_lk::emit_slot(j, kk, key, ix, row0, out_idx + oq * topk, out_score + oq * topk);
    if (tid == 0) { atomicAdd(survivor_total, (unsigned long long)nsurv); atomicAdd(exact_total, (unsigned long long)nb); }
}

}  // namespace

// ------------------------------------------------------------------ host side
struct asp_tc_cache {               // per-space fp16 operands in lambda order, built on the first tensor-core search
    __half *hi = nullptr, *lo = nullptr;      // lo (remainder of the residual columns) only once a 3-term search needs it
    float *lam32 = nullptr, *tile_lo = nullptr, *tile_hi = nullptr;   // the order key (lambda | norm) per item and tile
    int32_t *perm = nullptr;
    int order = ASP_TC_ORDER_IDENTITY;   // visiting order of the items: lambda (search), norm (l2 item graph) or identity
                                         // (cosine item graph before the lambdas exist)
    double norm_max = 0.0;          // ASP_TC_ORDER_NORM: the shard's largest norm
    double *mdir = nullptr;         // [f] unit mean direction of the shard's unit vectors
    double rho_max = 1.0;           // largest residual norm |x^ - (m.x^) m| of the shard
    int kp = 0;                     // operand row: f residual columns + 3 rank-1 columns, padded to a multiple of 64
    CUtensorMap map_hi, map_lo, map_hi_half;      // boxes of 256 item rows; 128 for the CTA-pair kernel
    CUtensorMap map_hi_nw;                        // narrow box (16 | 32 halves) over the last k block, see TcParams::nw_hi
    int nw = 0;
    asp_scratch mem;                // owns hi, lo, lam32, tile_lo, tile_hi, perm, mdir
};

int asp_device_max(asp_ctx *ctx, const double *v_dev, int64_t n, double *out)
{
    cudaStream_t st = ctx->stream;
    asp_scratch sc(st);
    double *d_mm = nullptr;
    std::vector<double> h_mm(512);
    ASP_CHECK(sc.get(&d_mm, 512));
    minmax_kernel<<<256, 256, 0, st>>>(v_dev, n, d_mm);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaMemcpyAsync(h_mm.data(), d_mm, sizeof(double) * 512, cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    double hi = 0.0;
    for (int i = 0; i < 256; ++i) hi = fmax(hi, h_mm[2 * i + 1]);
    *out = hi;
    return ASP_OK;
}

// ascending bucket order of n f64 keys (65536 buckets over [min, max]); the order inside a bucket is whatever the
// atomics produce -- callers only rely on the bucket order.  No host synchronisation.
static int bucket_order(asp_ctx *ctx, const double *keys_dev, int64_t n, int32_t *perm_dev)
{
    cudaStream_t st = ctx->stream;
    asp_scratch sc(st);
    double *scratch = nullptr;                                              // [256][2] partials + [2] range
    uint32_t *cursor = nullptr;
    ASP_CHECK(sc.get(&scratch, 514));
    ASP_CHECK(sc.get(&cursor, LAM_BUCKETS));
    ASP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(uint32_t) * LAM_BUCKETS, st));
    const int grid = (int)(asp_ceil_div(n, 256) < ctx->num_sms * 4 ? asp_ceil_div(n, 256) : ctx->num_sms * 4);
    minmax_kernel<<<256, 256, 0, st>>>(keys_dev, n, scratch);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    range_finalize_kernel<<<1, 32, 0, st>>>(scratch, 256, scratch + 512);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    bucket_hist_kernel<<<grid, 256, 0, st>>>(keys_dev, n, scratch + 512, cursor);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    bucket_scan_kernel<<<1, 1024, 0, st>>>(cursor);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    bucket_scatter_kernel<<<grid, 256, 0, st>>>(keys_dev, n, scratch + 512, cursor, perm_dev);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    return ASP_OK;
}

__global__ void iota_kernel(int32_t *__restrict__ p, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = (int32_t)i;
}

// by_norm: the l2 item graph's cache (items in norm order).  Otherwise the cosine one: lambda order once the space has
// lambdas, identity order before.  A cache of the other kind is rebuilt, so a search sees the same operands whatever graph
// was built before it.
static int ensure_tc_cache(const asp_space *s, bool by_norm, asp_tc_cache **out)
{
    asp_space *ms = const_cast<asp_space *>(s);
    if (ms->tc_cache) {
        asp_tc_cache *have = static_cast<asp_tc_cache *>(ms->tc_cache);
        const bool ok = by_norm ? have->order == ASP_TC_ORDER_NORM
                                : have->order == ASP_TC_ORDER_LAMBDA || (have->order == ASP_TC_ORDER_IDENTITY && !s->have_lambdas);
        if (ok) { *out = have; return ASP_OK; }
        asp_free_tc_cache(ms);                                          // other order (or built before the lambdas existed): rebuild
    }
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    std::unique_ptr<asp_tc_cache> c(new asp_tc_cache());           // the space holds it once it is complete
    c->mem = asp_scratch(st);
    c->kp = (s->f + 3 + TKB - 1) / TKB * TKB;
    const int64_t n = s->n_local;
    const size_t ne = (size_t)n * c->kp;
    const int64_t ntile = asp_ceil_div(n, TN);
    asp_scratch tmp(st);
    double *partials = nullptr, *rho = nullptr;
    ASP_CHECK(c->mem.get(&c->hi, ne));
    ASP_CHECK(c->mem.get(&c->lam32, (size_t)n));
    ASP_CHECK(c->mem.get(&c->perm, (size_t)n));
    ASP_CHECK(c->mem.get(&c->tile_lo, (size_t)ntile));
    ASP_CHECK(c->mem.get(&c->tile_hi, (size_t)ntile));
    ASP_CHECK(c->mem.get(&c->mdir, (size_t)s->f));
    ASP_CHECK(tmp.get(&partials, (size_t)MD_BLOCKS * s->f));
    ASP_CHECK(tmp.get(&rho, (size_t)n));
    // visiting order: bucket sort of the shard by lambda (identity while the space has no lambdas: item graph), or by norm
    c->order = by_norm ? ASP_TC_ORDER_NORM : s->have_lambdas ? ASP_TC_ORDER_LAMBDA : ASP_TC_ORDER_IDENTITY;
    if (c->order != ASP_TC_ORDER_IDENTITY) ASP_CHECK(bucket_order(ctx, by_norm ? s->norms : s->lambdas, n, c->perm));
    else { iota_kernel<<<ctx->num_sms * 4, 256, 0, st>>>(c->perm, n); ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx); }
    // mean direction, projection, fp16 operands
    colsum_unit_kernel<<<MD_BLOCKS, 256, 0, st>>>(s->items, n, s->f, s->fp, s->inv_norms, partials);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    mean_dir_kernel<<<1, 256, 0, st>>>(partials, MD_BLOCKS, s->f, c->mdir);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    project_split_kernel<<<ctx->num_sms * 8, 256, 0, st>>>(s->items, n, s->f, s->fp, c->kp, s->inv_norms, c->perm, c->mdir, 0,
                                                          c->hi, nullptr, rho);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    ASP_CHECK(asp_device_max(ctx, rho, n, &c->rho_max));
    if (c->order != ASP_TC_ORDER_IDENTITY) {
        tile_lambda_kernel<<<(unsigned)ntile, TN, 0, st>>>(by_norm ? s->norms : s->lambdas, c->perm, n, c->lam32, c->tile_lo, c->tile_hi);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
        if (by_norm) ASP_CHECK(asp_device_max(ctx, s->norms, n, &c->norm_max));
    } else {
        ASP_CUDA(cudaMemsetAsync(c->lam32, 0, sizeof(float) * n, st));
        ASP_CUDA(cudaMemsetAsync(c->tile_lo, 0, sizeof(float) * ntile, st));
        ASP_CUDA(cudaMemsetAsync(c->tile_hi, 0, sizeof(float) * ntile, st));
    }
    ASP_CHECK(asp_make_f16_tmap(&c->map_hi, c->hi, n, c->kp, TN));
    ASP_CHECK(asp_make_f16_tmap(&c->map_hi_half, c->hi, n, c->kp, TN / 2));
    c->map_lo = c->map_hi;
    {   // the last k block holds (f + 3) - 64 * (kp / 64 - 1) useful columns: 16 or 32 of them travel as a narrow box
        const int used = s->f + 3 - (c->kp / TKB - 1) * TKB;
        c->nw = (used <= 16) ? 16 : (used <= 32) ? 32 : 0;
        if (const char *e = getenv("ASP_TC_NARROW")) { if (atoi(e) == 0) c->nw = 0; }     // A/B knob (same results either way)
        c->map_hi_nw = c->map_hi;
        if (c->nw) ASP_CHECK(asp_make_f16_tmap_narrow(&c->map_hi_nw, c->hi, n, c->kp, TN, c->nw));
    }
    *out = c.release();
    ms->tc_cache = *out;
    return ASP_OK;
}

// the remainders of the residual columns, for the two-term split (3 MMA terms): built when first needed
static int ensure_tc_lo(const asp_space *s, asp_tc_cache *c)
{
    if (c->lo) return ASP_OK;
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    asp_scratch tmp(st);
    double *rho = nullptr;
    ASP_CHECK(c->mem.get(&c->lo, (size_t)s->n_local * c->kp));
    ASP_CHECK(tmp.get(&rho, (size_t)s->n_local));
    project_split_kernel<<<ctx->num_sms * 8, 256, 0, st>>>(s->items, s->n_local, s->f, s->fp, c->kp, s->inv_norms, c->perm, c->mdir, 0,
                                                          c->hi, c->lo, rho);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    ASP_CHECK(asp_make_f16_tmap(&c->map_lo, c->lo, s->n_local, c->kp, TN));
    return ASP_OK;
}

void asp_free_tc_cache(asp_space *s)
{
    delete static_cast<asp_tc_cache *>(s->tc_cache);
    s->tc_cache = nullptr;
}

bool asp_search_tc_supported(const asp_space *s, int64_t nq, int64_t topk, double tau, bool wide)
{
    return topk >= 1 && topk <= (wide ? asp_lk::KMAX : TK_LIST_MAX) && nq >= 1 && s->n_local >= 1 && s->n_local < 2147483647LL && tau > 1e-3 &&
           tau <= 1.0 && s->fp <= 6144;   // beta = 1 - tau >= 0: the proximity term is bounded from above by prox_ub
}

// ------------------------------------------------------------------ stage 1 for one batch of query vectors
// Prepares the query operands (lambda_q order when lambdas are given, projection, per-row bands), runs tc_gemm_kernel and
// leaves the emission lists in `b` for the caller's stage 2 (search: tc_rescore_kernel; item graph: knn.cu).
// lambda_q_dev == nullptr: no lambda term (cosine kNN): identity query order.  dump_dev != nullptr: approximate cosines
// [nq][n_local] f32 (tests), no emission.  l2 (Euclidean item graph): score -d^2~, items in norm order, queries visited in
// the order of their norms (qnorm_dev is the key; lambda_q_dev and tau are unused).  ntau > 1 (tau sweep, search of
// topk <= 16): the pass serves sweep_taus[0 .. ntau), `tau` is unused, and delta_q, theta_glob and emit_sc hold one plane
// per tau ([nq] / [nq] / [nq][nsub][capb]), and so does emit_cnt ([nq][nsub]).
int asp_tc_stage1(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                  const double *qnorm_dev, double tau, int64_t topk, double score_floor, int force_terms, int capb_override,
                  float *dump_dev, asp_tc_batch *b, bool l2, const uint32_t *allowed_dev, const double *sweep_taus, int ntau)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const double t_stage1 = asp_now_us();
    asp_tc_cache *c = nullptr;
    if (l2 && dump_dev) ASP_FAIL(ASP_ERR_ARG, "asp_tc_stage1: no dump of the l2 score");
    if (allowed_dev && (l2 || dump_dev)) ASP_FAIL(ASP_ERR_ARG, "asp_tc_stage1: only the search is filtered");
    const bool sweep = ntau > 1;
    if (sweep && (l2 || dump_dev || topk > 16 || ntau > asp_sweep::NT_MAX || score_floor > -1e300))
        ASP_FAIL(ASP_ERR_ARG, "asp_tc_stage1: a tau sweep is a search of k <= 16 over at most %d taus", asp_sweep::NT_MAX);
    const int planes = sweep ? ntau : 1;
    ASP_CHECK(ensure_tc_cache(s, l2, &c));
    if (l2) { lambda_q_dev = qnorm_dev; tau = 1.0; }
    const int kp = c->kp;
    *b = asp_tc_batch();
    b->mem = asp_scratch(st);
    b->nq = nq;

    __half *q_hi = nullptr, *q_lo = nullptr;
    const int64_t qblocks = asp_ceil_div(nq, TQ);
    ASP_CHECK(b->mem.get(&q_hi, (size_t)nq * kp));
    ASP_CHECK(b->mem.get(&q_lo, (size_t)nq * kp));
    b->q_hi = q_hi; b->q_lo = q_lo;
    ASP_CHECK(b->mem.get(&b->lam_q32, (size_t)nq));
    ASP_CHECK(b->mem.get(&b->inv_nq, (size_t)nq));
    ASP_CHECK(b->mem.get(&b->rho_q, (size_t)nq));
    ASP_CHECK(b->mem.get(&b->delta_q, (size_t)nq * planes));
    ASP_CHECK(asp_launch_reciprocal(ctx, qnorm_dev, nq, b->inv_nq));
    const bool by_lambda = !dump_dev && lambda_q_dev && c->order != ASP_TC_ORDER_IDENTITY;   // (l2: by the query norms)
    if (by_lambda) {
        // queries visited in lambda_q order: coherent blocks -> one visiting order per block
        ASP_CHECK(b->mem.get(&b->qperm, (size_t)nq));
        ASP_CHECK(b->mem.get(&b->center, (size_t)qblocks));
        if (nq > TQ) ASP_CHECK(bucket_order(ctx, lambda_q_dev, nq, b->qperm));
        else {              // one query block: its visiting order starts at one of its own lambdas whatever the query order
            iota_kernel<<<1, 128, 0, st>>>(b->qperm, nq);
            ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
        }
    }
    project_split_kernel<<<ctx->num_sms * 4, 256, 0, st>>>(q_dev, nq, s->f, qpitch, kp, b->inv_nq, b->qperm, c->mdir, 1, q_hi, q_lo, b->rho_q);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    // error band of one approximate cosine, |cos~ - cos| <= rho_q rho_x c_main + c_fixed (margin x2 on a worst-case
    // model: fp16 roundings of both residuals, round-toward-zero f32 accumulation, truncated rank-1 split)
    double rho_q_max = 1.0;
    ASP_CHECK(asp_device_max(ctx, b->rho_q, nq, &rho_q_max));
    ctx->stats["search_host_prep_us"] = asp_now_us() - t_stage1;
    const double steps = (double)((s->f + 15) / 16);
    const double c_main1 = 2.0 * c->rho_max * (ldexp(1.0, -10) * (1.0 + ldexp(1.0, -11)) + steps * ldexp(1.0, -23));
    const double c_main3 = 2.0 * c->rho_max * (3.0 * ldexp(1.0, -22) + 3.0 * steps * ldexp(1.0, -23));
    const double c_fixed = 2.0 * (3.0 * ldexp(1.0, -22) + 4.0 * ldexp(1.0, -23) + 1e-12);
    int nterms = (rho_q_max * c_main1 + c_fixed <= 2.5e-4) ? 1 : 3;
    if (const char *e = getenv("ASP_TC_TERMS")) { const int v = atoi(e); if (v == 1 || v == 3) nterms = v; }
    if (force_terms == 1 || force_terms == 3) nterms = force_terms;
    if (nterms == 3) ASP_CHECK(ensure_tc_lo(s, c));
    const double c_main = (nterms == 1) ? c_main1 : c_main3;
    if (l2) row_delta_l2_kernel<<<64, 256, 0, st>>>(b->rho_q, qnorm_dev, b->qperm, nq, c_main, c_fixed, c->norm_max, b->delta_q);
    else
        for (int u = 0; u < planes; ++u) {
            const double tu = sweep ? sweep_taus[u] : tau;
            row_delta_kernel<<<64, 256, 0, st>>>(b->rho_q, nq, c_main, c_fixed, fabs(tu), (fabs(tu) + fabs(1.0 - tu)) * 2e-6,
                                                 b->delta_q + (size_t)u * nq);
            if (u + 1 < planes) { ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx); }
        }
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    b->nterms = nterms;
    b->delta_cos_max = rho_q_max * c_main + c_fixed;
    ctx->stats["search_terms"] = nterms;
    ctx->stats["search_delta_cos_max"] = b->delta_cos_max;
    ctx->stats["search_rho_q_max"] = rho_q_max;
    ctx->stats["search_rho_x_max"] = c->rho_max;
    if (lambda_q_dev) {
        gather_f32_kernel<<<64, 256, 0, st>>>(lambda_q_dev, b->qperm, nq, b->lam_q32);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    } else {
        ASP_CUDA(cudaMemsetAsync(b->lam_q32, 0, sizeof(float) * nq, st));
    }
    if (by_lambda) {
        block_center_kernel<<<(unsigned)asp_ceil_div(qblocks, 128), 128, 0, st>>>(b->lam_q32, nq, c->tile_lo,
                                                                               (int)asp_ceil_div(s->n_local, TN), b->center);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    }
    CUtensorMap map_q_hi, map_q_lo, map_q_nw;
    ASP_CHECK(asp_make_f16_tmap(&map_q_hi, q_hi, nq, kp, TQ));
    ASP_CHECK(asp_make_f16_tmap(&map_q_lo, q_lo, nq, kp, TQ));
    map_q_nw = map_q_hi;
    if (c->nw) ASP_CHECK(asp_make_f16_tmap_narrow(&map_q_nw, q_hi, nq, kp, TQ, c->nw));

    // grid: query blocks x item chunks, whole waves of SMs
    const int64_t tiles_total = asp_ceil_div(s->n_local, TN);
    int64_t best_chunks = 1;
    double best_eff = 0.0;
    for (int w = 1; w <= 16; ++w) {
        int64_t cc = ((int64_t)w * ctx->num_sms) / qblocks;
        if (cc < 1) continue;
        if (cc > tiles_total) cc = tiles_total;
        const int64_t ctas = cc * qblocks;
        const double eff = (double)ctas / (double)(asp_ceil_div(ctas, ctx->num_sms) * ctx->num_sms);
        if (eff > best_eff + 1e-9) { best_eff = eff; best_chunks = cc; }
        if (eff >= 0.97 || cc == tiles_total) break;
    }
    int nchunks = (int)best_chunks;
    if (const char *e = getenv("ASP_TC_CHUNKS")) {                   // tuning knob (same results for any split)
        const long v = atol(e);
        if (v >= 1 && v <= tiles_total) nchunks = (int)v;
    }
    int capb = dump_dev ? 1 : (capb_override > 0 ? capb_override : 1024);   // per (query, chunk)
    if (const char *e = getenv("ASP_TC_CAPB")) {                     // test knob: shrink the emission buffers
        const int v = atoi(e);
        if (!dump_dev && v >= 8 && v <= 65536) capb = v;
    }
    b->nsub = nchunks; b->capb = capb;

    TcParams p;
    p.nq = nq; p.n_local = s->n_local; p.kp = kp; p.nchunks = nchunks; p.capb = capb; p.topk = (int)topk;
    p.tau = (float)tau; p.beta = (float)(1.0 - tau);
    p.score_floor = (score_floor > -1e300) ? nextafterf((float)score_floor, -INFINITY) : -INFINITY;
    p.delta_q = b->delta_q; p.nterms = nterms;
    p.kb_lo = (s->f + TKB - 1) / TKB; p.kb_hi = kp / TKB;
    p.sub_lo_last = (s->f - (p.kb_lo - 1) * TKB + 15) / 16;
    p.sub_hi_last = (s->f + 3 - (p.kb_hi - 1) * TKB + 15) / 16;
    p.nw_hi = c->nw;
    p.lam_x = c->lam32; p.lam_q = b->lam_q32; p.tile_lo = c->tile_lo; p.tile_hi = c->tile_hi; p.perm = c->perm; p.center = b->center;
    p.theta_glob = nullptr; p.emit_sc = nullptr; p.emit_ix = nullptr; p.emit_cnt = nullptr; p.dump = dump_dev; p.vbits = nullptr;
    p.ntau = planes; p.plane = (size_t)nq * nchunks * capb;
    for (int u = 0; u < asp_sweep::NT_MAX; ++u) {                 // unused slots: tau 1, beta 0 (never read)
        const float tu = (sweep && u < ntau) ? (float)sweep_taus[u] : 1.0f;
        p.taus[u] = tu; p.betas[u] = (sweep && u < ntau) ? (float)(1.0 - sweep_taus[u]) : 0.0f; p.inv_taus[u] = 1.0f / tu;
    }
    if (allowed_dev) {                                            // from the cache's current order (it may have been rebuilt)
        const int64_t nwords = tiles_total * (TN / 32);
        ASP_CHECK(b->mem.get(&b->vbits, (size_t)nwords));
        visit_bits_kernel<<<(unsigned)std::min<int64_t>(asp_ceil_div(nwords, 8), (int64_t)ctx->num_sms * 8), 256, 0, st>>>(
            allowed_dev, c->perm, s->n_local, nwords, b->vbits);
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
        p.vbits = b->vbits;
    }
    if (!dump_dev) {
        ASP_CHECK(b->mem.get(&b->emit_sc, (size_t)nq * nchunks * capb * planes));
        ASP_CHECK(b->mem.get(&b->emit_ix, (size_t)nq * nchunks * capb));
        ASP_CHECK(b->mem.get(&b->emit_cnt, (size_t)nq * nchunks * planes));
        ASP_CHECK(b->mem.get(&b->theta_glob, (size_t)nq * planes));
        ASP_CUDA(cudaMemsetAsync(b->theta_glob, 0, sizeof(uint32_t) * (size_t)nq * planes, st));
        p.emit_sc = b->emit_sc; p.emit_ix = b->emit_ix; p.emit_cnt = b->emit_cnt; p.theta_glob = b->theta_glob;
    }

    // 1-term mode with a query operand of <= 7 k blocks: keep it resident (ARES), stream only the item tiles
    bool ares = (nterms == 1) && (p.kb_hi <= 7);
    if (const char *e = getenv("ASP_TC_ARES")) ares = ares && atoi(e) != 0;
    const bool wide = topk > 16;                                  // 32-entry running lists
    const int listn = topk > 32 ? 64 : 0;                         // k = 33 .. 64 (the _k entry points): 64-entry lists
    // CTA pairs (cta_group::2: two query blocks share one M = 256 MMA, each SM loads half of every item tile) whenever there
    // are two query blocks to pair: -18 % stage-1 time at C4 / 64k queries (ASP_TC_PAIR=0: the 1-SM kernel, same bits)
    bool pair = ares && !dump_dev && qblocks >= 2;
    if (const char *e = getenv("ASP_TC_PAIR")) pair = pair && atoi(e) != 0;
    const size_t smem = (ares ? (size_t)p.kb_hi * A_BYTES + 3 * (size_t)B_BYTES : (size_t)TC_STAGES * STAGE_BYTES) +
                        2 * TN * sizeof(float) + 1024;
    const int64_t grid_x = pair ? (qblocks + 1) / 2 * 2 : qblocks;
    dim3 grid((unsigned)grid_x, nchunks);
    // Profiling variants (epilogue / MMA switched off: the results are WRONG) exist only in builds with -DASP_PROFILING
    // (python -m pyarrowspace_b200.build --profiling); the shipped library has no knob that changes a result.
#ifdef ASP_PROFILING
    const char *var = getenv("ASP_TC_VARIANT");
    int v = (var && !dump_dev && !wide) ? atoi(var) : 0;
#else
    int v = 0;
#endif
    if (pair) p.nw_hi = 0;                                        // (the CTA-pair kernel keeps full boxes)
    if (l2 || allowed_dev || listn) v = 0;
    void (*k)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, TcParams) =
        dump_dev ? (ares ? tc_gemm_kernel<true, 0, true, false, 16> : tc_gemm_kernel<true, 0, false, false, 16>)
        : wide ? (pair ? tc_gemm_kernel<false, 0, true, true, 32> : ares ? tc_gemm_kernel<false, 0, true, false, 32> : tc_gemm_kernel<false, 0, false, false, 32>)
#ifdef ASP_PROFILING
        : pair ? ((v == 2) ? tc_gemm_kernel<false, 2, true, true, 16> : (v == 3) ? tc_gemm_kernel<false, 3, true, true, 16>
                  : (v == 4) ? tc_gemm_kernel<false, 4, true, true, 16> : tc_gemm_kernel<false, 0, true, true, 16>)
        : (v == 4 && ares) ? tc_gemm_kernel<false, 4, true, false, 16>
        : (v == 2) ? (ares ? tc_gemm_kernel<false, 2, true, false, 16> : tc_gemm_kernel<false, 2, false, false, 16>)
        : (v == 3) ? (ares ? tc_gemm_kernel<false, 3, true, false, 16> : tc_gemm_kernel<false, 3, false, false, 16>)
#else
        : pair ? tc_gemm_kernel<false, 0, true, true, 16>
#endif
        : (ares ? tc_gemm_kernel<false, 0, true, false, 16> : tc_gemm_kernel<false, 0, false, false, 16>);
    if (allowed_dev)
        k = wide ? (pair ? tc_gemm_kernel<false, 0, true, true, 32, false, true> : ares ? tc_gemm_kernel<false, 0, true, false, 32, false, true>
                         : tc_gemm_kernel<false, 0, false, false, 32, false, true>)
                 : (pair ? tc_gemm_kernel<false, 0, true, true, 16, false, true> : ares ? tc_gemm_kernel<false, 0, true, false, 16, false, true>
                         : tc_gemm_kernel<false, 0, false, false, 16, false, true>);
    if (listn == 64)
        k = allowed_dev ? (pair ? tc_gemm_kernel<false, 0, true, true, 64, false, true> : ares ? tc_gemm_kernel<false, 0, true, false, 64, false, true>
                                : tc_gemm_kernel<false, 0, false, false, 64, false, true>)
                        : (pair ? tc_gemm_kernel<false, 0, true, true, 64> : ares ? tc_gemm_kernel<false, 0, true, false, 64>
                                : tc_gemm_kernel<false, 0, false, false, 64>);
    if (l2)
        k = wide ? (pair ? tc_gemm_kernel<false, 0, true, true, 32, true> : ares ? tc_gemm_kernel<false, 0, true, false, 32, true>
                         : tc_gemm_kernel<false, 0, false, false, 32, true>)
                 : (pair ? tc_gemm_kernel<false, 0, true, true, 16, true> : ares ? tc_gemm_kernel<false, 0, true, false, 16, true>
                         : tc_gemm_kernel<false, 0, false, false, 16, true>);
    constexpr int NTS = asp_sweep::NT_MAX;
    if (sweep)
        k = allowed_dev ? (pair ? tc_gemm_kernel<false, 0, true, true, 16, false, true, NTS> : ares ? tc_gemm_kernel<false, 0, true, false, 16, false, true, NTS>
                                : tc_gemm_kernel<false, 0, false, false, 16, false, true, NTS>)
                        : (pair ? tc_gemm_kernel<false, 0, true, true, 16, false, false, NTS> : ares ? tc_gemm_kernel<false, 0, true, false, 16, false, false, NTS>
                                : tc_gemm_kernel<false, 0, false, false, 16, false, false, NTS>);
    ASP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ASP_CUDA(cudaEventRecord(ctx->ev0, st));
    if (pair) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        ASP_CUDA(cudaLaunchKernelEx(&cfg, k, map_q_hi, map_q_lo, c->map_hi, c->map_hi_half, map_q_nw, c->map_hi_nw, p));
    } else {
        k<<<grid, TC_THREADS, smem, st>>>(map_q_hi, map_q_lo, c->map_hi, c->map_lo, map_q_nw, c->map_hi_nw, p);
    }
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaEventRecord(ctx->ev1, st));
    ctx->stats["search_host_stage1_launched_us"] = asp_now_us() - t_stage1;
    b->variant = v;
    ctx->stats["search_cta_pair"] = pair ? 1.0 : 0.0;
    ctx->stats["search_a_resident"] = ares ? 1.0 : 0.0;
    return ASP_OK;
}

namespace {
__global__ void gather_queries_kernel(const double *__restrict__ q, int qpitch, const double *__restrict__ lam, const double *__restrict__ nrm,
                                      const int32_t *__restrict__ list, int count, double *__restrict__ q2, double *__restrict__ lam2,
                                      double *__restrict__ nrm2)
{
    const int i = blockIdx.x;
    if (i >= count) return;
    const int64_t src = list[i];
    for (int j = threadIdx.x; j < qpitch; j += blockDim.x) q2[(size_t)i * qpitch + j] = q[src * qpitch + j];
    if (threadIdx.x == 0) { lam2[i] = lam[src]; nrm2[i] = nrm[src]; }
}
__global__ void scatter_results_kernel(const int64_t *__restrict__ idx2, const double *__restrict__ sc2, const int32_t *__restrict__ list,
                                       int count, int topk, int64_t *__restrict__ idx, double *__restrict__ sc)
{
    const int i = blockIdx.x;
    if (i >= count) return;
    const int64_t dst = list[i];
    for (int j = threadIdx.x; j < topk; j += blockDim.x) { idx[dst * topk + j] = idx2[(size_t)i * topk + j]; sc[dst * topk + j] = sc2[(size_t)i * topk + j]; }
}
}  // namespace

// f64 band of stage 2's fast re-score at tau
static double stage2_eps_fast(const asp_space *s, double tau)
{
    const double u = 1.1102230246251565e-16;
    return (4.0 * s->f + 64.0) * u * (fabs(tau) + fabs(1.0 - tau) + 1.0);
}

// Stage 2 of topk <= 32 (tc_rescore_kernel) on the emission lists of b, with the scores, counts and bands of one tau (emit_sc,
// emit_cnt, delta_q: b's own, or one plane of a tau sweep).
static int launch_stage2(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                         const double *qnorm_dev, double tau, int64_t topk, const asp_tc_batch &b, const float *delta_q,
                         const float *emit_sc, const int32_t *emit_cnt, int64_t *out_idx_dev, double *out_score_dev, int32_t *slow_list,
                         int32_t *slow_count, unsigned long long *counters)
{
    cudaStream_t st = s->ctx->stream;
    const double eps_fast = stage2_eps_fast(s, tau);
    // small batches (the reference's one query per call, latency bound): a whole CTA per query
    const int wpq = (nq <= 64) ? 32 : (nq <= 1024) ? 8 : 1;
    auto launch_rescore = [&](auto kern, int nwarps, int qcopies, unsigned grid) -> int {
        const size_t rsmem = (size_t)qcopies * s->fp * 8 + (size_t)nwarps * TR_QUEUE * 4 + (size_t)nwarps * 32 * 16;
        ASP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem));
        kern<<<grid, nwarps * 32, rsmem, st>>>(
            q_dev, qpitch, nq, s->items, s->n_local, s->f, s->fp, s->row0, s->norms, s->lambdas, qnorm_dev, lambda_q_dev, tau,
            (int)topk, b.nsub, b.capb, delta_q, eps_fast, emit_sc, b.emit_ix, emit_cnt, b.theta_glob, b.qperm, out_idx_dev,
            out_score_dev, slow_list, slow_count, counters, counters + 1);
        return ASP_OK;
    };
    if (wpq == 32) return launch_rescore(tc_rescore_kernel<32>, 32, 1, (unsigned)nq);
    if (wpq == 8) return launch_rescore(tc_rescore_kernel<8>, 8, 1, (unsigned)nq);
    if (getenv("ASP_TC_RESCORE_OCC6")) return launch_rescore(tc_rescore_kernel<1>, TR_WARPS, TR_WARPS, (unsigned)asp_ceil_div(nq, TR_WARPS));
    return launch_rescore(tc_rescore_kernel<1, TR_MIN_CTAS>, TR_WARPS, TR_WARPS, (unsigned)asp_ceil_div(nq, TR_WARPS));
}

// One attempt with a given number of MMA terms.  The search always tries ONE fp16 term first: its band is wide when the
// residual norms are large (mean-zero embeddings: 2e-3 in cosine against 2e-5 for the three-term split), but a wide band only
// costs survivors in stage 2 -- measured on the mean-zero C4 regime: 22.9 survivors per query instead of 10.1, 37 ms per 64k
// queries instead of 114 ms, same answers.  Queries whose emission buffers overflow under the wide band are redone with the
// three-term split (retry), and what is still undecided (exact ties around the k-th score) takes the exact scan.
static int search_tc_attempt(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                             const double *qnorm_dev, double tau, int64_t topk, int64_t *out_idx_dev, double *out_score_dev,
                             float *dump_dev, int force_terms, bool may_retry, const uint32_t *allowed_dev, bool wide);

// The retry of the slow queries (slow_list, device) of a single-term attempt with the three-term split; their results are
// scattered into the caller's rows.  Synchronises the stream.
static int retry_three_terms(const asp_space *s, const double *q_dev, int32_t qpitch, const double *lambda_q_dev,
                             const double *qnorm_dev, double tau, int64_t topk, const int32_t *slow_list, int nslow,
                             int64_t *out_idx_dev, double *out_score_dev, const uint32_t *allowed_dev, bool wide)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    asp_scratch retry(st);
    double *q2 = nullptr, *lam2 = nullptr, *nrm2 = nullptr, *sc2 = nullptr;
    int64_t *idx2 = nullptr;
    ASP_CHECK(retry.get(&q2, (size_t)nslow * qpitch));
    ASP_CHECK(retry.get(&lam2, (size_t)nslow));
    ASP_CHECK(retry.get(&nrm2, (size_t)nslow));
    ASP_CHECK(retry.get(&idx2, (size_t)nslow * topk));
    ASP_CHECK(retry.get(&sc2, (size_t)nslow * topk));
    gather_queries_kernel<<<(unsigned)nslow, 128, 0, st>>>(q_dev, qpitch, lambda_q_dev, qnorm_dev, slow_list, nslow, q2, lam2, nrm2);
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    int rc = search_tc_attempt(s, q2, nslow, qpitch, lam2, nrm2, tau, topk, idx2, sc2, nullptr, 3, false, allowed_dev, wide);
    if (rc == ASP_OK) {
        scatter_results_kernel<<<(unsigned)nslow, 32, 0, st>>>(idx2, sc2, slow_list, nslow, (int)topk, out_idx_dev, out_score_dev);
        ASP_LAUNCHED(ctx);
        if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) { asp_set_error("search retry: scatter failed"); rc = ASP_ERR_CUDA; }
    }
    return rc;
}

// MMA terms of a search's first attempt, and whether its slow queries may be retried with three
static int first_terms(bool *may_retry)
{
    const char *e = getenv("ASP_TC_FIRST_TERMS");                  // A/B knob: "auto" = the band rule decides (the earlier behaviour)
    int first = (e && e[0] == 'a') ? 0 : 1;
    if (const char *t = getenv("ASP_TC_TERMS")) { const int v = atoi(t); if (v == 1 || v == 3) first = v; }   // test knob: that mode, no retry
    const bool pinned = getenv("ASP_TC_TERMS") != nullptr;
    *may_retry = first == 1 && !pinned;
    return first;
}

// dump == nullptr: full search.  dump != nullptr: approximate cosines [nq][n_local] f32 (tests).  allowed_dev: item mask
// (local item order, packed) or nullptr.  wide: topk = 32 .. 128 takes the wide stage 2 (tc_rescore_wide_kernel) instead of
// the 32-per-warp one, whose lists cannot hold a candidate beyond the 32nd (the _k entry points only).
int asp_search_tc_impl(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                       const double *qnorm_dev, double tau, int64_t topk, int64_t *out_idx_dev, double *out_score_dev,
                       float *dump_dev, const uint32_t *allowed_dev, bool wide)
{
    bool may_retry = false;
    const int first = dump_dev ? 0 : first_terms(&may_retry);
    return search_tc_attempt(s, q_dev, nq, qpitch, lambda_q_dev, qnorm_dev, tau, topk, out_idx_dev, out_score_dev, dump_dev, first,
                             may_retry, allowed_dev, wide);
}

static int search_tc_attempt(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                             const double *qnorm_dev, double tau, int64_t topk, int64_t *out_idx_dev, double *out_score_dev,
                             float *dump_dev, int force_terms, bool may_retry, const uint32_t *allowed_dev, bool wide)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    asp_tc_batch b;
    // the wide stage 2 keeps every survivor, so its emission lists get room for k-sized lists plus the band: a chunk of a
    // million items emits about k (1 + ln(items / k)) records plus every item within the band of the k-th score
    const bool wide2 = wide && topk >= asp_lk::KMIN;
    int rc = asp_tc_stage1(s, q_dev, nq, qpitch, lambda_q_dev, qnorm_dev, tau, topk, -INFINITY, force_terms,
                           wide2 ? (int)(64 * topk) : 0, dump_dev, &b, false, allowed_dev);
    if (rc != ASP_OK || dump_dev) return rc;

    if (b.variant != 0) {                                         // profiling variants: stage 1 only, results are garbage
        ASP_CUDA(cudaStreamSynchronize(st));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        ctx->stats["search_stage1_ms"] = ms;
        ASP_CUDA(cudaMemsetAsync(out_idx_dev, 0xff, sizeof(int64_t) * (size_t)nq * topk, st));
        ASP_CUDA(cudaMemsetAsync(out_score_dev, 0, sizeof(double) * (size_t)nq * topk, st));
        return ASP_OK;
    }
    asp_scratch sc(st);
    int32_t *slow_list = nullptr, *slow_count = nullptr;
    unsigned long long *counters = nullptr;
    ASP_CHECK(sc.get(&slow_list, (size_t)nq + 1));
    ASP_CHECK(sc.get(&slow_count, 1));
    ASP_CHECK(sc.get(&counters, 2));
    ASP_CUDA(cudaMemsetAsync(slow_count, 0, sizeof(int32_t), st));
    ASP_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long), st));
    const double eps_fast = stage2_eps_fast(s, tau);
    if (wide2) {
        const size_t wsmem = (size_t)s->fp * 8 + (size_t)asp_lk::SURV_CAP * (sizeof(uint64_t) + sizeof(int32_t));
        ASP_CUDA(cudaFuncSetAttribute(tc_rescore_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        tc_rescore_wide_kernel<<<(unsigned)nq, TW_THREADS, wsmem, st>>>(
            q_dev, qpitch, s->items, s->n_local, s->f, s->fp, s->row0, s->norms, s->lambdas, qnorm_dev, lambda_q_dev, tau, (int)topk,
            b.nsub, b.capb, b.delta_q, eps_fast, b.emit_sc, b.emit_ix, b.emit_cnt, b.qperm, out_idx_dev, out_score_dev, slow_list,
            slow_count, counters, counters + 1);
    } else ASP_CHECK(launch_stage2(s, q_dev, nq, qpitch, lambda_q_dev, qnorm_dev, tau, topk, b, b.delta_q, b.emit_sc, b.emit_cnt,
                                   out_idx_dev, out_score_dev, slow_list, slow_count, counters));
    ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaEventRecord(ctx->ev2, st));
    int32_t nslow = 0;
    unsigned long long cnts[2] = {0, 0};
    ASP_CUDA(cudaMemcpyAsync(&nslow, slow_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaMemcpyAsync(cnts, counters, sizeof(cnts), cudaMemcpyDeviceToHost, st));
    if (ctx->on_wait) { auto fn = std::move(ctx->on_wait); ctx->on_wait = nullptr; fn(); }   // host work hidden behind both stages
    ASP_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f, ms2 = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    cudaEventElapsedTime(&ms2, ctx->ev1, ctx->ev2);
    ctx->stats["search_stage1_ms"] = ms;
    ctx->stats["search_stage2_ms"] = ms2;
    ctx->stats["search_slow_queries"] = nslow;
    ctx->stats["search_rescored_per_query"] = (double)cnts[0] / (double)nq;
    ctx->stats["search_exact_per_query"] = (double)cnts[1] / (double)nq;
    ctx->stats["search_stage1_is_tc"] = 1.0;
    if (may_retry) ctx->stats["search_retry_queries"] = 0.0;
    const bool wide_band = b.nterms == 1 && b.delta_cos_max > 2.5e-4;   // the three-term split has a much tighter band to offer
    if (nslow > 0 && may_retry && wide_band) {
        const std::map<std::string, double> first_stats = ctx->stats;
        b.mem.release();                                              // the retry allocates its own emission buffers
        rc = retry_three_terms(s, q_dev, qpitch, lambda_q_dev, qnorm_dev, tau, topk, slow_list, nslow, out_idx_dev, out_score_dev,
                               allowed_dev, wide);
        const double retry_slow = ctx->stats["search_slow_queries"], retry_ms = ctx->stats["search_stage1_ms"] + ctx->stats["search_stage2_ms"];
        ctx->stats = first_stats;                                     // the batch's figures stay those of the first attempt
        ctx->stats["search_retry_queries"] = nslow;
        ctx->stats["search_retry_ms"] = retry_ms;
        ctx->stats["search_slow_queries"] = retry_slow;              // what finally took the exact scan
    } else if (nslow > 0) {
        rc = asp_search_slow_path(s, q_dev, qpitch, lambda_q_dev, qnorm_dev, tau, topk, slow_list, nslow, out_idx_dev, out_score_dev,
                                  allowed_dev);
    }
    return rc;
}

// Tau sweep (DESIGN §2 item 8): one candidate pass for all ntau taus, then per tau the stage 2 above on that tau's score
// plane, and today's remedies for its slow queries (the three-term retry when the single-term band is wide, else the exact
// scan).  The stage-2 kernels of all taus run back to back; the emission buffers are released before the remedies.
int asp_search_tc_sweep(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                        const double *qnorm_dev, const double *taus, int ntau, int64_t topk, int64_t *const *out_idx_dev,
                        double *const *out_score_dev, const uint32_t *allowed_dev, int64_t *slow_out)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    bool may_retry = false;
    const int first = first_terms(&may_retry);
    asp_tc_batch b;
    // the records of ntau taus share each (query, chunk) buffer: ntau times the single-tau capacity, so that one tau's
    // records (tau = 1 on near duplicates) do not crowd out the others' and send their queries to the remedies
    ASP_CHECK(asp_tc_stage1(s, q_dev, nq, qpitch, lambda_q_dev, qnorm_dev, taus[0], topk, -INFINITY, first, 1024 * ntau, nullptr, &b,
                            false, allowed_dev, taus, ntau));
    asp_scratch sc(st);
    int32_t *slow_list = nullptr, *slow_count = nullptr;
    unsigned long long *counters = nullptr;
    ASP_CHECK(sc.get(&slow_list, (size_t)ntau * (nq + 1)));
    ASP_CHECK(sc.get(&slow_count, (size_t)ntau));
    ASP_CHECK(sc.get(&counters, 2 * (size_t)ntau));
    ASP_CUDA(cudaMemsetAsync(slow_count, 0, sizeof(int32_t) * ntau, st));
    ASP_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long) * ntau, st));
    const size_t plane = (size_t)nq * b.nsub * b.capb;
    for (int u = 0; u < ntau; ++u) {
        ASP_CHECK(launch_stage2(s, q_dev, nq, qpitch, lambda_q_dev, qnorm_dev, taus[u], topk, b, b.delta_q + (size_t)u * nq,
                                b.emit_sc + u * plane, b.emit_cnt + (size_t)u * nq * b.nsub, out_idx_dev[u], out_score_dev[u],
                                slow_list + (size_t)u * (nq + 1),
                                slow_count + u, counters + 2 * u));
        ASP_CUDA(cudaGetLastError()); ASP_LAUNCHED(ctx);
    }
    ASP_CUDA(cudaEventRecord(ctx->ev2, st));
    std::vector<int32_t> nslow(ntau), cnt((size_t)nq * b.nsub);
    ASP_CUDA(cudaMemcpyAsync(nslow.data(), slow_count, sizeof(int32_t) * ntau, cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaMemcpyAsync(cnt.data(), b.emit_cnt, sizeof(int32_t) * cnt.size(), cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f, ms2 = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    cudaEventElapsedTime(&ms2, ctx->ev1, ctx->ev2);
    double emitted = 0.0;                                         // records written (an overflowing buffer counts its capacity)
    for (int32_t c : cnt) emitted += std::min(c, b.capb);
    const bool wide_band = b.nterms == 1 && b.delta_cos_max > 2.5e-4;
    const int nterms = b.nterms;
    b.mem.release();                                              // the remedies allocate their own buffers
    for (int u = 0; u < ntau; ++u) {
        slow_out[u] = nslow[u];
        if (nslow[u] == 0) continue;
        const int32_t *list = slow_list + (size_t)u * (nq + 1);
        if (may_retry && wide_band) {
            ASP_CHECK(retry_three_terms(s, q_dev, qpitch, lambda_q_dev, qnorm_dev, taus[u], topk, list, nslow[u], out_idx_dev[u],
                                        out_score_dev[u], allowed_dev, false));
            slow_out[u] = (int64_t)ctx->stats["search_slow_queries"];   // what finally took the exact scan
        } else {
            ASP_CHECK(asp_search_slow_path(s, q_dev, qpitch, lambda_q_dev, qnorm_dev, taus[u], topk, list, nslow[u], out_idx_dev[u],
                                           out_score_dev[u], allowed_dev));
        }
    }
    ctx->stats["sweep_stage1_ms"] += ms;
    ctx->stats["sweep_stage2_ms"] += ms2;
    ctx->stats["sweep_emitted"] += emitted;
    ctx->stats["search_terms"] = nterms;
    return ASP_OK;
}
