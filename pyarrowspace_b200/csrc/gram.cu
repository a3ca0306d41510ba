// gram.cu -- K1, API orientation: Gram matrix of the feature columns, G = X^T X (f x f), the
// contraction behind every pairwise cosine distance of the feature graph
// (replaces the distance pass inside arrowspace's ArrowSpaceBuilder::build, call site
// /root/reference/src/lib.rs:289; recipe GRAPH_VARIABLES.md:7).
//
// Bound: FP64 tensor pipe, 2*n*f^2 FLOP (SURVEY.md 8(d) K1).  X is streamed once from HBM
// (8*n*f bytes); the other tile CTAs of the same slice hit L2.
//
// Decomposition (fixed, independent of the GPU count -- see ASP_GRAM_* in the header):
//   rows -> 32-row units -> 8 segments -> 24 slices each.  One CTA owns one (upper-triangular
//   128x128 output tile, slice) pair and runs ONE in-order DMMA chain over the slice's rows.
//   Slice partials are summed in slice order per segment (gram_segment_reduce), segment partials in
//   segment order after the cross-GPU all-gather (gram_final_reduce).
//
// CTA: 8 DMMA warps (4 along a, 2 along b; warp tile 32x64 = 4x8 DMMA.8x8x4 tiles, 64 f64
// accumulators per thread), thread 0 doubles as the TMA producer; 3-stage mbarrier pipeline, 64 KB per stage
// (32 rows x 128 features for the a-block and for the b-block).  Shared-memory stage layout
// [feature/4][row][4] (tensormap.cu) makes every fragment load 256 contiguous bytes per warp.
#include "common.cuh"

#include <algorithm>
#include "ptx.cuh"

namespace {

constexpr int TILE = 128;          // output tile edge (features)
constexpr int RI = ASP_ROW_UNIT;   // rows (k extent) per stage
constexpr int STAGES = 3;
constexpr int OPERAND_DOUBLES = RI * TILE;          // 4096 doubles = 32 KB
constexpr int STAGE_DOUBLES = 2 * OPERAND_DOUBLES;  // a-block + b-block
constexpr int NUM_MMA_WARPS = 8;

struct SliceRange { int unit_begin; int unit_end; };   // local 32-row units of one slice

__device__ __forceinline__ void decode_upper_tile(int t, int nt, int &ta, int &tb)
{
    ta = 0;
    int rowlen = nt;
    while (t >= rowlen) { t -= rowlen; ++ta; --rowlen; }
    tb = ta + t;
}

template <bool USE_TMA>
__global__ void __launch_bounds__(NUM_MMA_WARPS * 32, 1)
gram_slice_kernel(const __grid_constant__ CUtensorMap tmap, const double *__restrict__ items, int64_t n_local, int fp,
                  int ntile, const SliceRange *__restrict__ slices, double *__restrict__ partial)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *smem = reinterpret_cast<double *>(smem_raw);
    __shared__ __align__(8) uint64_t full_bar[STAGES];
    __shared__ __align__(8) uint64_t empty_bar[STAGES];

    int ta, tb;
    decode_upper_tile(blockIdx.x, ntile, ta, tb);
    const bool diag = (ta == tb);
    const SliceRange sr = slices[blockIdx.y];
    const int nunits = sr.unit_end - sr.unit_begin;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (USE_TMA) {
        if (threadIdx.x == 0) {
            for (int s = 0; s < STAGES; ++s) {
                asp::mbar_init(&full_bar[s], 1);
                asp::mbar_init(&empty_bar[s], NUM_MMA_WARPS);
            }
            asp::fence_barrier_init();
        }
        __syncthreads();
    }

    // TMA producer = thread 0, inline: it runs STAGES-1 units ahead of the DMMA loop.
    auto tma_issue = [&](int it) {
        const int s = it % STAGES;
        if (it >= STAGES) asp::mbar_wait(&empty_bar[s], (uint32_t)(((it / STAGES) - 1) & 1));
        double *dstA = smem + s * STAGE_DOUBLES;
        asp::mbar_arrive_expect_tx(&full_bar[s], (diag ? 1u : 2u) * OPERAND_DOUBLES * 8u);
        const int row = (sr.unit_begin + it) * RI;
        asp::tma_load_3d(dstA, &tmap, &full_bar[s], 0, row, ta * (TILE / 4));
        if (!diag) asp::tma_load_3d(dstA + OPERAND_DOUBLES, &tmap, &full_bar[s], 0, row, tb * (TILE / 4));
    };
    if (USE_TMA && threadIdx.x == 0) {
        asp::tma_prefetch_desc(&tmap);
        for (int it = 0; it < STAGES - 1 && it < nunits; ++it) tma_issue(it);
    }

    // ===== DMMA consumers =====
    const int wm = warp & 3, wn = warp >> 2;
    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // fragment offsets inside an operand block: ((outer * RI) + item) * 4 + inner
    const int frag_inner = (lane >> 2) & 3;
    const int frag_item = lane & 3;
    const int frag_outer = lane >> 4;
    const int a_base = ((wm * 8 + frag_outer) * RI + frag_item) * 4 + frag_inner;    // + mt*2*RI*4 + ks*16
    const int b_base = ((wn * 16 + frag_outer) * RI + frag_item) * 4 + frag_inner;   // + nt*2*RI*4 + ks*16

    auto load_stage_cp_async = [&](int it) {
        // fallback loader: 16-byte cp.async into the same [outer][row][4] layout
        const int s = it % STAGES;
        double *dst = smem + s * STAGE_DOUBLES;
        const int64_t row_base = (int64_t)(sr.unit_begin + it) * RI;
        const int nop = diag ? 1 : 2;
        for (int op = 0; op < nop; ++op) {
            const int col0 = (op == 0 ? ta : tb) * TILE;
            for (int c = threadIdx.x; c < RI * TILE / 2; c += NUM_MMA_WARPS * 32) {
                const int r = c / (TILE / 2);
                const int f = (c % (TILE / 2)) * 2;
                const int64_t grow = row_base + r;
                const bool valid = (grow < n_local) && (col0 + f < fp);
                const double *src = valid ? items + grow * fp + col0 + f : items;
                asp::cp_async16(dst + op * OPERAND_DOUBLES + (((f >> 2) * RI + r) * 4 + (f & 3)), src, valid);
            }
        }
    };

    if (!USE_TMA) {
        for (int it = 0; it < STAGES - 1; ++it) {
            if (it < nunits) load_stage_cp_async(it);
            asp::cp_async_commit();
        }
    }

    for (int it = 0; it < nunits; ++it) {
        const int s = it % STAGES;
        if (USE_TMA) {
            if (threadIdx.x == 0 && it + STAGES - 1 < nunits) tma_issue(it + STAGES - 1);
            asp::mbar_wait(&full_bar[s], (it / STAGES) & 1);
        } else {
            asp::cp_async_wait<STAGES - 2>();
            __syncthreads();
            if (it + STAGES - 1 < nunits) load_stage_cp_async(it + STAGES - 1);
            asp::cp_async_commit();
        }
        const double *A = smem + s * STAGE_DOUBLES;
        const double *B = diag ? A : A + OPERAND_DOUBLES;
#pragma unroll
        for (int ks = 0; ks < RI / 4; ++ks) {
            double a[4], b[8];
#pragma unroll
            for (int mt = 0; mt < 4; ++mt) a[mt] = A[a_base + mt * (2 * RI * 4) + ks * 16];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) b[nt] = B[b_base + nt * (2 * RI * 4) + ks * 16];
#pragma unroll
            for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) asp::dmma884(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
        }
        if (USE_TMA) {
            __syncwarp();
            if (lane == 0) asp::mbar_arrive(&empty_bar[s]);
        }
    }

    // epilogue: slice partial of this tile, row-major 128x128
    const int ntu = ntile * (ntile + 1) / 2;
    double *out = partial + ((size_t)blockIdx.y * ntu + blockIdx.x) * (TILE * TILE);
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int r = wm * 32 + mt * 8 + (lane >> 2);
            const int c = wn * 64 + nt * 8 + 2 * (lane & 3);
            *reinterpret_cast<double2 *>(out + r * TILE + c) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
        }
}

// seg_out[e][a][b] = sum_{j < ASP_GRAM_SLICES} partial[(e_local*SLICES + j)][tile(a,b)][..], j ascending
__global__ void gram_segment_reduce(const double *__restrict__ partial, int ntile, int f, int nseg_owned, int seg0,
                                    double *__restrict__ seg_out)
{
    const int64_t total = (int64_t)nseg_owned * f * f;
    const int ntu = ntile * (ntile + 1) / 2;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int el = (int)(i / ((int64_t)f * f));
        const int rem = (int)(i % ((int64_t)f * f));
        int a = rem / f, b = rem % f;
        if ((a / TILE) > (b / TILE)) { const int t = a; a = b; b = t; }   // lower tiles mirror the upper ones
        const int ta = a / TILE, tb = b / TILE;
        const int tidx = ta * ntile - ta * (ta - 1) / 2 + (tb - ta);
        const double *p = partial + ((size_t)el * ASP_GRAM_SLICES * ntu + tidx) * (TILE * TILE) + (a % TILE) * TILE + (b % TILE);
        double s = 0.0;
        for (int j = 0; j < ASP_GRAM_SLICES; ++j) s += p[(size_t)j * ntu * TILE * TILE];
        seg_out[(size_t)(seg0 + el) * f * f + rem] = s;
    }
}

// gram[a][b] = sum_e seg[e][a][b], e ascending
__global__ void gram_final_reduce(const double *__restrict__ seg, int f, double *__restrict__ gram)
{
    const int64_t total = (int64_t)f * f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int e = 0; e < ASP_GRAM_SEGMENTS; ++e) s += seg[(size_t)e * total + i];
        gram[i] = s;
    }
}

}  // namespace

// Geometry shared with api.cu (asp_shard_rows): units of segment e are [e*U/8, (e+1)*U/8).
static inline int64_t seg_unit_begin(int64_t units, int e) { return (units * e) / ASP_GRAM_SEGMENTS; }

int asp_launch_gram_partials(asp_space *s, double *out_dev)
{
    asp_ctx *ctx = s->ctx;
    const int64_t units_total = asp_ceil_div(s->n_total, ASP_ROW_UNIT);
    // owned segments: rank r of `world` holds segments [r*8/world, (r+1)*8/world)  (asp_shard_rows)
    const int64_t unit0 = s->row0 / ASP_ROW_UNIT;
    const int seg0 = s->rank * (ASP_GRAM_SEGMENTS / s->world), seg1 = (s->rank + 1) * (ASP_GRAM_SEGMENTS / s->world);
    const int nseg = seg1 - seg0;
    const int nslices = nseg * ASP_GRAM_SLICES;

    std::vector<SliceRange> h_slices(nslices);
    for (int e = seg0; e < seg1; ++e) {
        const int64_t b = seg_unit_begin(units_total, e), len = seg_unit_begin(units_total, e + 1) - b;
        for (int j = 0; j < ASP_GRAM_SLICES; ++j) {
            SliceRange r;
            r.unit_begin = (int)(b + (len * j) / ASP_GRAM_SLICES - unit0);
            r.unit_end = (int)(b + (len * (j + 1)) / ASP_GRAM_SLICES - unit0);
            h_slices[(e - seg0) * ASP_GRAM_SLICES + j] = r;
        }
    }
    const int ntile = (int)asp_ceil_div(s->fp, TILE);
    const int ntu = ntile * (ntile + 1) / 2;

    // The slice partials are scratch of nslices * ntu * 128 KB: 151 MB at F = 384, but quadratic in F (13 GB at 4096, 52 GB at
    // 8192 for a whole-matrix shard).  Segments are independent, so they are processed in groups whose scratch stays
    // under 2 GB (one group -- one launch -- for the usual feature counts).
    const size_t seg_bytes = sizeof(double) * (size_t)ASP_GRAM_SLICES * ntu * TILE * TILE;
    int group = (int)std::max<size_t>(1, std::min<size_t>((size_t)nseg, ((size_t)2 << 30) / seg_bytes));
    asp_scratch sc(ctx->stream);
    SliceRange *d_slices = nullptr;
    double *d_partial = nullptr;
    ASP_CHECK(sc.get(&d_slices, (size_t)nslices));
    ASP_CHECK(sc.get(&d_partial, seg_bytes / sizeof(double) * group));
    ASP_CUDA(cudaMemcpyAsync(d_slices, h_slices.data(), sizeof(SliceRange) * nslices, cudaMemcpyHostToDevice,
                             ctx->stream));

    const size_t smem = (size_t)STAGES * STAGE_DOUBLES * sizeof(double);
    for (int e0 = 0; e0 < nseg; e0 += group) {
        const int ne = std::min(group, nseg - e0);
        dim3 grid(ntu, ne * ASP_GRAM_SLICES);
        if (ctx->use_tma) {
            ASP_CUDA(cudaFuncSetAttribute(gram_slice_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            gram_slice_kernel<true><<<grid, NUM_MMA_WARPS * 32, smem, ctx->stream>>>(
                s->tmap_gram, s->items, s->n_local, s->fp, ntile, d_slices + (size_t)e0 * ASP_GRAM_SLICES, d_partial);
        } else {
            ASP_CUDA(cudaFuncSetAttribute(gram_slice_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            gram_slice_kernel<false><<<grid, NUM_MMA_WARPS * 32, smem, ctx->stream>>>(
                s->tmap_gram, s->items, s->n_local, s->fp, ntile, d_slices + (size_t)e0 * ASP_GRAM_SLICES, d_partial);
        }
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
        gram_segment_reduce<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(d_partial, ntile, s->f, ne, seg0 + e0, out_dev);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    return ASP_OK;
}

int asp_launch_gram_reduce(asp_ctx *ctx, const double *segments_dev, int32_t f, double *gram_dev)
{
    gram_final_reduce<<<ctx->num_sms * 2, 256, 0, ctx->stream>>>(segments_dev, f, gram_dev);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    return ASP_OK;
}
