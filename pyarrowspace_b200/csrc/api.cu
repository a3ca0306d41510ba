// api.cu -- the C ABI declared in include/arrowspace_b200.h (extern "C", plain pointers).
// Host-side orchestration only; every numeric step is a kernel in gram.cu / graph_select.cu /
// csr.cu / taumode.cu / search.cu / knn.cu / range.cu.  There is no CPU fallback anywhere in this file.
#include "common.cuh"
#include "sweep_bound.cuh"
#include "hybrid.cuh"

#include <algorithm>
#include <cmath>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

// ------------------------------------------------------------------ errors
static thread_local std::string g_last_error;

void asp_set_error(const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

bool asp_is_device_ptr(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

int asp_copy_in(asp_ctx *ctx, void *dst_dev, const void *src, size_t bytes)
{
    if (bytes == 0) return ASP_OK;
    ASP_CUDA(cudaMemcpyAsync(dst_dev, src, bytes, cudaMemcpyDefault, ctx->stream));
    return ASP_OK;
}

int asp_copy_out(asp_ctx *ctx, void *dst, const void *src_dev, size_t bytes)
{
    if (bytes == 0) return ASP_OK;
    ASP_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDefault, ctx->stream));
    if (!asp_is_device_ptr(dst)) ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ASP_OK;
}

namespace {

struct StageTimer {
    asp_ctx *ctx;
    const char *key;
    cudaEvent_t a, b;
    StageTimer(asp_ctx *c, const char *k) : ctx(c), key(k)
    {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, ctx->stream);
    }
    void stop()
    {
        cudaEventRecord(b, ctx->stream);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        ctx->stats[key] = ms;
    }
    ~StageTimer()
    {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
    }
};

__global__ void zero_lambda_check_kernel(const double *lam, int64_t n, int *flag)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (lam[i] == 0.0) atomicExch(flag, 1);
}

// upload an n x f row-major matrix (host or device) into a pitched, zero padded device buffer
int upload_pitched(cudaStream_t st, const double *src, int64_t n, int32_t f, int32_t pitch, double *dst)
{
    if (pitch == f) {       // one contiguous copy (a 2-D copy from pageable memory is staged row by row: ~1 GB/s)
        ASP_CUDA(cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)n * f, cudaMemcpyDefault, st));
        return ASP_OK;
    }
    ASP_CUDA(cudaMemsetAsync(dst, 0, sizeof(double) * (size_t)n * pitch, st));
    ASP_CUDA(cudaMemcpy2DAsync(dst, sizeof(double) * pitch, src, sizeof(double) * f, sizeof(double) * f, (size_t)n,
                               cudaMemcpyDefault, st));
    return ASP_OK;
}

// The packed item mask of a filtered call (ceil(n / 8) bytes, host or device) on the device as 32-bit words, the rest of the
// last word zero, held by the caller's scratch.  NULL bits: *out = NULL (every row).
int upload_allowed(asp_scratch &sc, const uint8_t *bits, int64_t n, uint32_t **out)
{
    *out = nullptr;
    if (!bits) return ASP_OK;
    cudaStream_t st = sc.st;
    const size_t nbytes = (size_t)((n + 7) / 8), nwords = (size_t)((n + 31) / 32);
    ASP_CHECK(sc.get(out, nwords));
    ASP_CUDA(cudaMemsetAsync(*out, 0, sizeof(uint32_t) * (nwords ? nwords : 1), st));
    if (nbytes) ASP_CUDA(cudaMemcpyAsync(*out, bits, nbytes, cudaMemcpyDefault, st));
    return ASP_OK;
}

}  // namespace

extern "C" {

const char *asp_last_error(void) { return g_last_error.c_str(); }
int asp_abi_version(void) { return ASP_ABI_VERSION; }

void asp_default_switches(asp_switches *sw)
{
    memset(sw, 0, sizeof(*sw));          // every switch's default is its zero value (SURVEY.md Appendix A)
    sw->kernel = ASP_KERNEL_INV_POWER;
    sw->tau_mode = ASP_TAU_MEDIAN;
    sw->tau_fixed = 0.0;
}

// range check of caller-supplied switches
static int check_switches(const asp_switches *sw)
{
    if (sw->kernel < 0 || sw->kernel > ASP_KERNEL_GAUSSIAN || sw->tau_mode < 0 || sw->tau_mode > ASP_TAU_FIXED ||
        sw->lambda_form < 0 || sw->lambda_form > ASP_LAMBDA_SYNTHETIC || sw->symmetrise < 0 || sw->symmetrise > ASP_SYM_NONE ||
        sw->laplacian < 0 || sw->laplacian > ASP_LAPLACIAN_RW || sw->distance < 0 || sw->distance > ASP_DISTANCE_L2SQ ||
        (sw->k_counts_self != 0 && sw->k_counts_self != 1) || (sw->topk_prunes != 0 && sw->topk_prunes != 1))
        ASP_FAIL(ASP_ERR_ARG, "asp_switches: value out of range");
    return ASP_OK;
}

int asp_ctx_create(int device, asp_ctx **out)
{
    if (!out) ASP_FAIL(ASP_ERR_ARG, "asp_ctx_create: out is NULL");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        ASP_FAIL(ASP_ERR_CUDA, "no CUDA device: arrowspace_b200 has no CPU fallback");
    }
    if (device < 0 || device >= ndev) ASP_FAIL(ASP_ERR_ARG, "device %d out of range [0,%d)", device, ndev);
    ASP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ASP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        ASP_FAIL(ASP_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    asp_ctx *ctx = new asp_ctx();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    ASP_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {   // keep freed blocks in the stream-ordered pool: every build/search reuses its scratch instead of
        // going back to the driver (cudaMalloc/cudaFree of GB-sized buffers cost milliseconds and synchronise).
        // Bounded (a quarter of the device by default, ASP_POOL_KEEP_GB overrides) so that another allocator in the
        // same process (PyTorch's) is not starved; asp_ctx_trim() gives the cached blocks back explicitly.
        cudaMemPool_t pool;
        ASP_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
        uint64_t keep = (uint64_t)prop.totalGlobalMem / 4;
        if (const char *e = getenv("ASP_POOL_KEEP_GB")) { const double gb = atof(e); if (gb >= 0.0) keep = (uint64_t)(gb * 1073741824.0); }
        ASP_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    ASP_CUDA(cudaEventCreate(&ctx->ev0));
    ASP_CUDA(cudaEventCreate(&ctx->ev1));
    ASP_CUDA(cudaEventCreate(&ctx->ev2));
    const char *no_tma = getenv("ASP_NO_TMA");
    ctx->use_tma = !(no_tma && no_tma[0] == '1');
    *out = ctx;
    return ASP_OK;
}

void asp_ctx_destroy(asp_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev2) cudaEventDestroy(ctx->ev2);
    if (ctx->up_stream) cudaStreamDestroy(ctx->up_stream);
    if (ctx->down_stream) cudaStreamDestroy(ctx->down_stream);
    for (auto &e : ctx->pipe_ev) if (e) cudaEventDestroy(e);
    delete ctx;
}

int asp_ctx_device(const asp_ctx *ctx) { return ctx ? ctx->device : -1; }

int asp_ctx_set_stream(asp_ctx *ctx, void *cuda_stream)
{
    if (!ctx) ASP_FAIL(ASP_ERR_ARG, "ctx is NULL");
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (cuda_stream) {
        ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
        ctx->own_stream = false;
    } else {
        ASP_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return ASP_OK;
}

int asp_ctx_synchronize(asp_ctx *ctx)
{
    if (!ctx) ASP_FAIL(ASP_ERR_ARG, "ctx is NULL");
    ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ASP_OK;
}

int64_t asp_ctx_launch_count(const asp_ctx *ctx) { return ctx ? ctx->launches : 0; }

int asp_ctx_trim(asp_ctx *ctx, size_t keep_bytes)
{
    if (!ctx) ASP_FAIL(ASP_ERR_ARG, "ctx is NULL");
    ASP_CUDA(cudaSetDevice(ctx->device));
    ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaMemPool_t pool;
    ASP_CUDA(cudaDeviceGetDefaultMemPool(&pool, ctx->device));
    ASP_CUDA(cudaMemPoolTrimTo(pool, keep_bytes));
    return ASP_OK;
}

double asp_ctx_stat(const asp_ctx *ctx, const char *key)
{
    if (!ctx || !key) return -1.0;
    auto it = ctx->stats.find(key);
    return it == ctx->stats.end() ? -1.0 : it->second;
}

// ------------------------------------------------------------------ sharding
int asp_shard_rows(int64_t n_total, int world, int rank, int64_t *row0, int64_t *row1)
{
    if (n_total <= 0 || world <= 0 || rank < 0 || rank >= world || ASP_GRAM_SEGMENTS % world != 0)
        ASP_FAIL(ASP_ERR_ARG, "asp_shard_rows: world must divide %d and 0 <= rank < world (got world=%d rank=%d)",
                 ASP_GRAM_SEGMENTS, world, rank);
    const int64_t units = asp_ceil_div(n_total, ASP_ROW_UNIT);
    const int seg0 = rank * (ASP_GRAM_SEGMENTS / world), seg1 = (rank + 1) * (ASP_GRAM_SEGMENTS / world);
    int64_t r0 = (units * seg0) / ASP_GRAM_SEGMENTS * ASP_ROW_UNIT;
    int64_t r1 = (units * seg1) / ASP_GRAM_SEGMENTS * ASP_ROW_UNIT;
    if (r0 > n_total) r0 = n_total;
    if (r1 > n_total) r1 = n_total;
    if (row0) *row0 = r0;
    if (row1) *row1 = r1;
    return ASP_OK;
}

int asp_space_create(asp_ctx *ctx, const double *items_shard, int64_t n_local, int32_t f, int64_t n_total, int world,
                     int rank, asp_space **out)
{
    if (!ctx || !out) ASP_FAIL(ASP_ERR_ARG, "asp_space_create: NULL argument");
    if (!items_shard || n_local <= 0 || f <= 0) ASP_FAIL(ASP_ERR_EMPTY, "items must be non-empty 2D array");
    int64_t r0 = 0, r1 = 0;
    ASP_CHECK(asp_shard_rows(n_total, world, rank, &r0, &r1));
    if (r1 - r0 != n_local)
        ASP_FAIL(ASP_ERR_ARG, "rank %d of %d owns rows [%lld,%lld) of %lld, got %lld rows", rank, world, (long long)r0,
                 (long long)r1, (long long)n_total, (long long)n_local);
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_space *s = new asp_space();
    s->ctx = ctx;
    s->n_local = n_local;
    s->row0 = r0;
    s->n_total = n_total;
    s->f = f;
    s->fp = (f + 3) & ~3;
    s->world = world;
    s->rank = rank;
    int rc = ASP_OK;
    if (cudaMallocAsync(&s->items, sizeof(double) * (size_t)n_local * s->fp, ctx->stream) != cudaSuccess ||
        cudaMallocAsync(&s->norms, sizeof(double) * n_local, ctx->stream) != cudaSuccess ||
        cudaMallocAsync(&s->inv_norms, sizeof(double) * n_local, ctx->stream) != cudaSuccess ||
        cudaMallocAsync(&s->lambdas, sizeof(double) * n_local, ctx->stream) != cudaSuccess) {
        cudaGetLastError();
        asp_set_error("out of device memory for the item shard");
        rc = ASP_ERR_NOMEM;
    }
    if (rc == ASP_OK) rc = upload_pitched(ctx->stream, items_shard, n_local, f, s->fp, s->items);
    if (rc == ASP_OK) rc = asp_make_items_tmap(&s->tmap_gram, s->items, n_local, s->fp, ASP_ROW_UNIT, 32);
    if (rc == ASP_OK) rc = asp_make_items_tmap(&s->tmap_rows, s->items, n_local, s->fp, 128, 4);
    if (rc == ASP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        asp_set_error("upload of the item shard failed: %s", cudaGetErrorString(cudaGetLastError()));
        rc = ASP_ERR_CUDA;
    }
    if (rc != ASP_OK) { asp_free_space(s); return rc; }
    *out = s;
    return ASP_OK;
}

// Space over a device buffer the CALLER keeps alive (n_local x f f64 row-major, f a multiple of 4, 16-byte aligned): no
// copy.  For the multi-GPU paths, where a gathered item matrix (C5: 54 GB per rank) must not exist twice.
int asp_space_adopt_shard(asp_ctx *ctx, double *items_dev, int64_t n_local, int32_t f, int64_t n_total, int world, int rank,
                          asp_space **out)
{
    if (!ctx || !out) ASP_FAIL(ASP_ERR_ARG, "asp_space_adopt_shard: NULL argument");
    if (!items_dev || n_local <= 0 || f <= 0) ASP_FAIL(ASP_ERR_EMPTY, "items must be non-empty 2D array");
    if (!asp_is_device_ptr(items_dev) || (f & 3) != 0 || (reinterpret_cast<uintptr_t>(items_dev) & 15) != 0)
        ASP_FAIL(ASP_ERR_ARG, "asp_space_adopt: needs 16-byte aligned device memory and a feature count that is a multiple of 4 (got %d)", f);
    int64_t r0 = 0, r1 = 0;
    ASP_CHECK(asp_shard_rows(n_total, world, rank, &r0, &r1));
    if (r1 - r0 != n_local)
        ASP_FAIL(ASP_ERR_ARG, "rank %d of %d owns rows [%lld,%lld) of %lld, got %lld rows", rank, world, (long long)r0,
                 (long long)r1, (long long)n_total, (long long)n_local);
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_space *s = new asp_space();
    s->ctx = ctx;
    s->n_local = n_local; s->row0 = r0; s->n_total = n_total;
    s->f = f; s->fp = f;
    s->world = world; s->rank = rank;
    s->items = items_dev;
    s->owns_items = false;
    int rc = ASP_OK;
    if (cudaMallocAsync(&s->norms, sizeof(double) * n_local, ctx->stream) != cudaSuccess ||
        cudaMallocAsync(&s->inv_norms, sizeof(double) * n_local, ctx->stream) != cudaSuccess ||
        cudaMallocAsync(&s->lambdas, sizeof(double) * n_local, ctx->stream) != cudaSuccess) {
        cudaGetLastError();
        asp_set_error("out of device memory for the item norms and lambdas");
        rc = ASP_ERR_NOMEM;
    }
    if (rc == ASP_OK) rc = asp_make_items_tmap(&s->tmap_gram, s->items, n_local, s->fp, ASP_ROW_UNIT, 32);
    if (rc == ASP_OK) rc = asp_make_items_tmap(&s->tmap_rows, s->items, n_local, s->fp, 128, 4);
    if (rc != ASP_OK) { asp_free_space(s); return rc; }
    *out = s;
    return ASP_OK;
}

int asp_space_adopt(asp_ctx *ctx, double *items_dev, int64_t n, int32_t f, asp_space **out)
{
    return asp_space_adopt_shard(ctx, items_dev, n, f, n, 1, 0, out);
}

// Per-item lambdas and norms computed elsewhere (the rank that owned the rows at build time): the multi-GPU regrouping
// all-gathers them next to the item rows instead of recomputing.  norms must be the left-to-right ones (asp_space_norms).
int asp_space_import_lambdas(asp_space *s, const double *lambdas, const double *norms)
{
    if (!s || !lambdas || !norms) ASP_FAIL(ASP_ERR_ARG, "asp_space_import_lambdas: NULL argument");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    ASP_CHECK(asp_copy_in(ctx, s->lambdas, lambdas, sizeof(double) * s->n_local));
    ASP_CHECK(asp_copy_in(ctx, s->norms, norms, sizeof(double) * s->n_local));
    ASP_CHECK(asp_launch_reciprocal(ctx, s->norms, s->n_local, s->inv_norms));
    ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    asp_free_tc_cache(s);                                           // operands in lambda order depend on the lambdas
    s->have_lambdas = true;
    return ASP_OK;
}

void asp_free_space(asp_space *s)
{
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStream_t st = s->ctx->stream;
    asp_free_tc_cache(s);
    if (s->items && s->owns_items) cudaFreeAsync(s->items, st);
    if (s->norms) cudaFreeAsync(s->norms, st);
    if (s->inv_norms) cudaFreeAsync(s->inv_norms, st);
    if (s->nsq) cudaFreeAsync(s->nsq, st);
    if (s->lambdas) cudaFreeAsync(s->lambdas, st);
    delete s;
}

void asp_free_graph(asp_graph *g)
{
    if (!g) return;
    cudaSetDevice(g->ctx->device);
    cudaStream_t st = g->ctx->stream;
    asp_graph_free_upper(g);
    void *bufs[] = {g->d_indptr, g->d_indices, g->d_data};
    for (void *b : bufs)
        if (b) cudaFreeAsync(b, st);
    delete g;
}

// ------------------------------------------------------------------ build stages
int asp_space_gram_partials(asp_space *s, double *out_dev)
{
    if (!s || !out_dev) ASP_FAIL(ASP_ERR_ARG, "asp_space_gram_partials: NULL argument");
    if (!asp_is_device_ptr(out_dev)) ASP_FAIL(ASP_ERR_ARG, "asp_space_gram_partials: out_dev must be device memory");
    ASP_CUDA(cudaSetDevice(s->ctx->device));
    StageTimer t(s->ctx, "gram_ms");
    const int rc = asp_launch_gram_partials(s, out_dev);
    t.stop();
    return rc;
}

int asp_graph_from_gram(asp_ctx *ctx, const double *gram_segments_dev, int32_t f, int64_t n_total,
                        const asp_graph_params *gp, const asp_switches *sw_in, const int32_t *exact_pairs,
                        const double *exact_sums, int64_t n_exact, int32_t *need_pairs, int64_t need_cap, int64_t *n_need,
                        asp_graph **out_graph)
{
    if (!ctx || !gram_segments_dev || !gp || !out_graph) ASP_FAIL(ASP_ERR_ARG, "asp_graph_from_gram: NULL argument");
    if (!asp_is_device_ptr(gram_segments_dev)) ASP_FAIL(ASP_ERR_ARG, "gram_segments_dev must be device memory");
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_switches sw;
    if (sw_in) sw = *sw_in; else asp_default_switches(&sw);
    ASP_CHECK(check_switches(&sw));
    cudaStream_t st = ctx->stream;
    if (n_need) *n_need = 0;
    StageTimer timer(ctx, "graph_ms");
    asp_scratch sc(st);

    double *gram = nullptr;
    ASP_CHECK(sc.get(&gram, (size_t)f * f));
    ASP_CHECK(asp_launch_gram_reduce(ctx, gram_segments_dev, f, gram));

    // exact pairs, sorted by (a, b) for the device binary search
    int32_t *d_pairs = nullptr;
    double *d_sums = nullptr;
    if (n_exact > 0) {
        std::vector<int64_t> order(n_exact);
        for (int64_t i = 0; i < n_exact; ++i) order[i] = i;
        std::sort(order.begin(), order.end(), [&](int64_t x, int64_t y) {
            if (exact_pairs[2 * x] != exact_pairs[2 * y]) return exact_pairs[2 * x] < exact_pairs[2 * y];
            return exact_pairs[2 * x + 1] < exact_pairs[2 * y + 1];
        });
        std::vector<int32_t> hp(2 * n_exact);
        std::vector<double> hs(3 * n_exact);
        for (int64_t i = 0; i < n_exact; ++i) {
            hp[2 * i] = exact_pairs[2 * order[i]];
            hp[2 * i + 1] = exact_pairs[2 * order[i] + 1];
            for (int c = 0; c < 3; ++c) hs[3 * i + c] = exact_sums[3 * order[i] + c];
        }
        ASP_CHECK(sc.get(&d_pairs, 2 * (size_t)n_exact));
        ASP_CHECK(sc.get(&d_sums, 3 * (size_t)n_exact));
        ASP_CUDA(cudaMemcpyAsync(d_pairs, hp.data(), sizeof(int32_t) * 2 * n_exact, cudaMemcpyHostToDevice, st));
        ASP_CUDA(cudaMemcpyAsync(d_sums, hs.data(), sizeof(double) * 3 * n_exact, cudaMemcpyHostToDevice, st));
        ASP_CUDA(cudaStreamSynchronize(st));
    }

    // room for every column pair (data with many duplicate columns puts most pairs inside the band), bounded at 16M pairs
    const int64_t all_pairs = (int64_t)f * (f - 1) / 2;
    const int64_t dev_cap = std::max<int64_t>(1, std::min<int64_t>(all_pairs * 2, (int64_t)1 << 24));
    int32_t *d_need = nullptr, *d_need_count = nullptr;
    ASP_CHECK(sc.get(&d_need, 2 * (size_t)dev_cap));
    ASP_CHECK(sc.get(&d_need_count, 1));
    ASP_CUDA(cudaMemsetAsync(d_need_count, 0, sizeof(int32_t), st));

    asp_knn_lists lists;
    int rc = asp_feature_select(ctx, gram, f, n_total, gp, &sw, d_pairs, d_sums, n_exact, &lists, d_need, dev_cap, d_need_count);
    int32_t need_count = 0;
    if (rc == ASP_OK) {
        ASP_CUDA(cudaMemcpyAsync(&need_count, d_need_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
    }
    asp_graph *g = nullptr;
    if (rc == ASP_OK && need_count > 0) {
        const int64_t got = need_count < dev_cap ? need_count : dev_cap;
        std::vector<int32_t> hp(2 * got);
        ASP_CUDA(cudaMemcpyAsync(hp.data(), d_need, sizeof(int32_t) * 2 * got, cudaMemcpyDeviceToHost, st));
        ASP_CUDA(cudaStreamSynchronize(st));
        std::vector<std::pair<int32_t, int32_t>> uniq(got);
        for (int64_t i = 0; i < got; ++i) uniq[i] = {hp[2 * i], hp[2 * i + 1]};
        std::sort(uniq.begin(), uniq.end());
        uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
        if (n_need) *n_need = (int64_t)uniq.size();
        ctx->stats["need_exact_pairs"] = (double)uniq.size();
        if (!need_pairs || (int64_t)uniq.size() > need_cap) {
            rc = ASP_ERR_ARG;
            asp_set_error("%lld column pairs fall inside the rounding band; need_pairs has room for %lld",
                          (long long)uniq.size(), (long long)need_cap);
        } else {
            for (size_t i = 0; i < uniq.size(); ++i) { need_pairs[2 * i] = uniq[i].first; need_pairs[2 * i + 1] = uniq[i].second; }
            rc = ASP_NEED_EXACT;
            asp_set_error("%lld column pairs need exact sums", (long long)uniq.size());
        }
    } else if (rc == ASP_OK) {
        g = new asp_graph();
        g->ctx = ctx;
        g->gp = *gp;
        if (!g->gp.has_sigma) { g->gp.sigma = gp->eps * 0.5; g->gp.has_sigma = 1; }   // src/helpers.rs:68-72
        g->sw = sw;
        rc = asp_assemble_laplacian(ctx, &lists, gp, &sw, g);
        if (rc == ASP_OK) rc = asp_graph_upload_upper(g);
        if (rc != ASP_OK) { asp_free_graph(g); g = nullptr; }
    }
    timer.stop();
    if (rc == ASP_OK) *out_graph = g;
    return rc;
}

int asp_space_exact_pairs(asp_space *s, const int32_t *pairs, int64_t n_pairs, double *sums)
{
    if (!s || (n_pairs > 0 && (!pairs || !sums))) ASP_FAIL(ASP_ERR_ARG, "asp_space_exact_pairs: NULL argument");
    if (n_pairs == 0) return ASP_OK;
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    asp_scratch sc(st);
    int32_t *d_pairs = nullptr;
    double *d_sums = nullptr;
    ASP_CHECK(sc.get(&d_pairs, 2 * (size_t)n_pairs));
    ASP_CHECK(sc.get(&d_sums, 3 * (size_t)n_pairs));
    ASP_CUDA(cudaMemcpyAsync(d_pairs, pairs, sizeof(int32_t) * 2 * n_pairs, cudaMemcpyDefault, st));
    ASP_CUDA(cudaMemcpyAsync(d_sums, sums, sizeof(double) * 3 * n_pairs, cudaMemcpyDefault, st));
    int rc = asp_launch_exact_pairs(s, d_pairs, n_pairs, d_sums);
    if (rc == ASP_OK) {
        ASP_CUDA(cudaMemcpyAsync(sums, d_sums, sizeof(double) * 3 * n_pairs, cudaMemcpyDefault, st));
        ASP_CUDA(cudaStreamSynchronize(st));
    }
    return rc;
}

int asp_space_compute_lambdas(asp_space *s, const asp_graph *g)
{
    if (!s || !g) ASP_FAIL(ASP_ERR_ARG, "asp_space_compute_lambdas: NULL argument");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_scratch sc(ctx->stream);
    int *flag = nullptr;
    ASP_CHECK(sc.get(&flag, 1));
    ASP_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), ctx->stream));
    StageTimer timer(ctx, "lambda_ms");
    int rc = asp_launch_taumode(ctx, g, &g->sw, s->items, s->n_local, s->f, s->fp, nullptr, nullptr, s->lambdas, s->norms,
                                s->inv_norms, flag);
    timer.stop();
    int h = 0;
    if (rc == ASP_OK) {
        ASP_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (rc != ASP_OK) return rc;
    if (h) ASP_FAIL(ASP_ERR_ZERO_VECTOR, "an item vector is all zeros: its Rayleigh quotient is undefined");
    s->have_lambdas = true;
    return ASP_OK;
}

// K1 (API orientation) + K2 for the rows of a world-1 space: Gram partials, selection with the exact-pair loop, Laplacian.
int asp_space_feature_graph(asp_space *s, const asp_graph_params *gp, const asp_switches *sw, asp_graph **out_graph)
{
    if (!s || !gp || !out_graph) ASP_FAIL(ASP_ERR_ARG, "asp_space_feature_graph: NULL argument");
    if (s->world != 1) ASP_FAIL(ASP_ERR_UNSUPPORTED, "asp_space_feature_graph: needs a world-1 space (the sharded build exchanges the Gram segments itself)");
    asp_ctx *ctx = s->ctx;
    const int32_t f = s->f;
    const int64_t n = s->n_local;
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_scratch sc(ctx->stream);
    double *segs = nullptr;
    asp_graph *g = nullptr;
    ASP_CHECK(sc.get(&segs, (size_t)ASP_GRAM_SEGMENTS * f * f));
    int rc = asp_space_gram_partials(s, segs);
    if (rc == ASP_OK) {
        double graph_ms = 0.0;
        std::vector<int32_t> pairs;
        std::vector<double> sums;
        int64_t cap = 1 << 16;
        std::vector<int32_t> need(2 * cap);
        for (int pass = 0; pass < 6; ++pass) {
            int64_t n_need = 0;
            rc = asp_graph_from_gram(ctx, segs, f, n, gp, sw, pairs.data(), sums.data(), (int64_t)(pairs.size() / 2),
                                     need.data(), cap, &n_need, &g);
            graph_ms += ctx->stats["graph_ms"];
            if (rc == ASP_ERR_ARG && n_need > cap) {               // more undecided pairs than the list holds: grow it, same pass again
                cap = n_need;
                need.resize(2 * cap);
                rc = ASP_NEED_EXACT;
                continue;
            }
            if (rc != ASP_NEED_EXACT) break;
            std::vector<double> add(3 * n_need, 0.0);
            rc = asp_space_exact_pairs(s, need.data(), n_need, add.data());
            if (rc != ASP_OK) break;
            pairs.insert(pairs.end(), need.begin(), need.begin() + 2 * n_need);
            sums.insert(sums.end(), add.begin(), add.end());
            rc = ASP_NEED_EXACT;
        }
        if (rc == ASP_NEED_EXACT) { asp_set_error("exact-pair resolution did not converge"); rc = ASP_ERR_CUDA; }
        ctx->stats["graph_ms"] = graph_ms;
    }
    if (rc != ASP_OK) { asp_free_graph(g); return rc; }
    *out_graph = g;
    return ASP_OK;
}

int asp_build(asp_ctx *ctx, const double *items, int64_t n, int32_t f, const asp_graph_params *gp, const asp_switches *sw,
              asp_space **out_space, asp_graph **out_graph)
{
    if (!ctx || !gp || !out_space || !out_graph) ASP_FAIL(ASP_ERR_ARG, "asp_build: NULL argument");
    if (!items || n <= 0 || f <= 0) ASP_FAIL(ASP_ERR_EMPTY, "items must be non-empty 2D array");
    asp_space *s = nullptr;
    {
        StageTimer t(ctx, "upload_ms");
        ASP_CHECK(asp_space_create(ctx, items, n, f, n, 1, 0, &s));
        t.stop();
    }
    asp_graph *g = nullptr;
    int rc = asp_space_feature_graph(s, gp, sw, &g);
    if (rc == ASP_OK) rc = asp_space_compute_lambdas(s, g);
    if (rc != ASP_OK) { asp_free_space(s); asp_free_graph(g); return rc; }
    *out_space = s;
    *out_graph = g;
    return ASP_OK;
}

// SURVEY.md 8(f)-1: sample -> two-NN -> k-means (reduce.cu), graph on the centroid matrix, lambdas of every item from it.
int asp_build_reduced(asp_ctx *ctx, const double *items, int64_t n, int32_t f, const asp_graph_params *gp,
                      const asp_switches *sw, const asp_reduction *red, asp_space **out_space, asp_graph **out_graph,
                      asp_reduction_info *info, asp_space **out_centroids)
{
    if (!ctx || !gp || !out_space || !out_graph) ASP_FAIL(ASP_ERR_ARG, "asp_build_reduced: NULL argument");
    if (!items || n <= 0 || f <= 0) ASP_FAIL(ASP_ERR_EMPTY, "items must be non-empty 2D array");
    asp_space *s = nullptr, *cs = nullptr;
    {
        StageTimer t(ctx, "upload_ms");
        ASP_CHECK(asp_space_create(ctx, items, n, f, n, 1, 0, &s));
        t.stop();
    }
    asp_graph *g = nullptr;
    int rc;
    {
        StageTimer t(ctx, "reduce_ms");
        rc = asp_space_reduce(s, red, n, info, &cs);
        t.stop();
    }
    if (rc == ASP_OK) rc = asp_space_feature_graph(cs, gp, sw, &g);
    if (rc == ASP_OK) rc = asp_space_compute_lambdas(s, g);
    if (rc != ASP_OK) { asp_free_space(s); asp_free_space(cs); asp_free_graph(g); return rc; }
    if (out_centroids) *out_centroids = cs; else asp_free_space(cs);
    *out_space = s;
    *out_graph = g;
    return ASP_OK;
}

// ------------------------------------------------------------------ accessors
int asp_space_dims(const asp_space *s, int64_t *n_local, int32_t *f, int64_t *row0, int64_t *n_total)
{
    if (!s) ASP_FAIL(ASP_ERR_ARG, "space is NULL");
    if (n_local) *n_local = s->n_local;
    if (f) *f = s->f;
    if (row0) *row0 = s->row0;
    if (n_total) *n_total = s->n_total;
    return ASP_OK;
}

int asp_space_lambdas(const asp_space *s, double *out)
{
    if (!s || !out) ASP_FAIL(ASP_ERR_ARG, "asp_space_lambdas: NULL argument");
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "lambdas have not been computed yet");
    ASP_CUDA(cudaSetDevice(s->ctx->device));
    return asp_copy_out(s->ctx, out, s->lambdas, sizeof(double) * s->n_local);
}

int asp_space_norms(const asp_space *s, double *out)
{
    if (!s || !out) ASP_FAIL(ASP_ERR_ARG, "asp_space_norms: NULL argument");
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "norms are computed together with the lambdas");
    ASP_CUDA(cudaSetDevice(s->ctx->device));
    return asp_copy_out(s->ctx, out, s->norms, sizeof(double) * s->n_local);
}

int asp_space_items(const asp_space *s, double *out)
{
    if (!s || !out) ASP_FAIL(ASP_ERR_ARG, "asp_space_items: NULL argument");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    ASP_CUDA(cudaMemcpy2DAsync(out, sizeof(double) * s->f, s->items, sizeof(double) * s->fp, sizeof(double) * s->f, (size_t)s->n_local,
                               cudaMemcpyDefault, ctx->stream));
    ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ASP_OK;
}

int asp_space_get_item(const asp_space *s, int64_t local_idx, double *out_features, double *out_lambda)
{
    if (!s) ASP_FAIL(ASP_ERR_ARG, "space is NULL");
    if (local_idx < 0 || local_idx >= s->n_local)
        ASP_FAIL(ASP_ERR_ARG, "index %lld out of range [0, %lld)", (long long)local_idx, (long long)s->n_local);
    ASP_CUDA(cudaSetDevice(s->ctx->device));
    if (out_features) ASP_CHECK(asp_copy_out(s->ctx, out_features, s->items + local_idx * s->fp, sizeof(double) * s->f));
    if (out_lambda) {
        if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "lambdas have not been computed yet");
        ASP_CHECK(asp_copy_out(s->ctx, out_lambda, s->lambdas + local_idx, sizeof(double)));
    }
    return ASP_OK;
}

int asp_graph_info(const asp_graph *g, int64_t *nnodes, int64_t *nnz, asp_graph_params *gp)
{
    if (!g) ASP_FAIL(ASP_ERR_ARG, "graph is NULL");
    if (nnodes) *nnodes = g->nnodes;
    if (nnz) *nnz = g->nnz;
    if (gp) *gp = g->gp;
    return ASP_OK;
}

int asp_graph_csr(const asp_graph *g, int64_t *indptr, int32_t *indices, double *data)
{
    if (!g) ASP_FAIL(ASP_ERR_ARG, "graph is NULL");
    ASP_CUDA(cudaSetDevice(g->ctx->device));
    if (indptr) ASP_CHECK(asp_copy_out(g->ctx, indptr, g->d_indptr, sizeof(int64_t) * (g->nnodes + 1)));
    if (indices) ASP_CHECK(asp_copy_out(g->ctx, indices, g->d_indices, sizeof(int32_t) * g->nnz));
    if (data) ASP_CHECK(asp_copy_out(g->ctx, data, g->d_data, sizeof(double) * g->nnz));
    return ASP_OK;
}

// ------------------------------------------------------------------ search
int asp_query_lambda(asp_ctx *ctx, const asp_graph *g, const asp_switches *sw_in, const double *queries, int64_t nq,
                     double *out_energy, double *out_tau, double *out_lambda)
{
    if (!ctx || !g || (nq > 0 && !queries)) ASP_FAIL(ASP_ERR_ARG, "asp_query_lambda: NULL argument");
    if (nq == 0) return ASP_OK;
    ASP_CUDA(cudaSetDevice(ctx->device));
    const asp_switches sw = sw_in ? *sw_in : g->sw;
    const int32_t f = (int32_t)g->nnodes;
    cudaStream_t st = ctx->stream;
    asp_scratch sc(st);
    double *dq = nullptr, *de = nullptr;
    int *flag = nullptr;
    ASP_CHECK(sc.get(&dq, (size_t)nq * f));
    ASP_CHECK(sc.get(&de, 3 * (size_t)nq));
    ASP_CHECK(sc.get(&flag, 1));
    ASP_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    ASP_CUDA(cudaMemcpyAsync(dq, queries, sizeof(double) * (size_t)nq * f, cudaMemcpyDefault, st));
    int rc = asp_launch_taumode(ctx, g, &sw, dq, nq, f, f, de, de + nq, de + 2 * nq, nullptr, nullptr, flag);
    int h = 0;
    if (rc == ASP_OK) {
        ASP_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        if (out_energy) rc = asp_copy_out(ctx, out_energy, de, sizeof(double) * nq);
        if (rc == ASP_OK && out_tau) rc = asp_copy_out(ctx, out_tau, de + nq, sizeof(double) * nq);
        if (rc == ASP_OK && out_lambda) rc = asp_copy_out(ctx, out_lambda, de + 2 * nq, sizeof(double) * nq);
        ASP_CUDA(cudaStreamSynchronize(st));
    }
    if (rc != ASP_OK) return rc;
    if (h) ASP_FAIL(ASP_ERR_ZERO_VECTOR, "a query vector is all zeros: its Rayleigh quotient is undefined");
    return ASP_OK;
}

// One device-resident batch: lambda_q (src/lib.rs:154), the lambda_q != 0 guard (src/lib.rs:156-159), candidate pass +
// exact stage 2.  `flags` is a 2-int device scratch.  allowed: the item mask as upload_allowed left it, or nullptr.
// Synchronises ctx->stream before returning.  wide (the _k entry points only): topk 32 .. 64 stays on the tensor-core route
// with the wide stage 2; without it such a topk takes the batched exact scan, as the graph-topk entry points always have.
// Whether a batch of nq queries at tau with topk results takes stage 1 on tcgen05 (fp16 split); otherwise FP64 DMMA / GEMV.
// Same exact stage 2, same answers.  Small batches against a large shard stream the fp16 operands (2 * kp bytes per item)
// instead of the f64 rows.
static bool search_takes_tc(const asp_space *s, int64_t nq, int64_t topk, double tau, bool wide)
{
    const char *force = getenv("ASP_SEARCH_STAGE1");
    const bool want_fp64 = force && force[0] == 'f';
    const bool want_tc = force && force[0] == 't';
    return !want_fp64 && asp_search_tc_supported(s, nq, topk, tau, wide) && (want_tc || nq >= 256 || s->n_local >= 131072);
}

// The search of a device batch whose lambda_q (dlam) and norms (dnorm) are known.  Synchronises ctx->stream.
static int search_device_stage(const asp_space *s, const asp_graph *g, const double *dq, int64_t nq, double tau, int64_t topk,
                               const double *dlam, const double *dnorm, int64_t *didx, double *dscore, const uint32_t *allowed, bool wide)
{
    int rc;
    if (search_takes_tc(s, nq, topk, tau, wide))
        rc = asp_search_tc_impl(s, dq, nq, s->fp, dlam, dnorm, tau, topk, didx, dscore, nullptr, allowed, wide);
    else
        rc = asp_search_impl(s, g, dq, nq, s->fp, dlam, dnorm, tau, topk, didx, dscore, allowed);
    if (rc == ASP_OK) ASP_CUDA(cudaStreamSynchronize(s->ctx->stream));
    return rc;
}

static int search_device_batch(const asp_space *s, const asp_graph *g, const double *dq, int64_t nq, double tau, int64_t topk,
                               double *dlam, double *dnorm, int *flags, int64_t *didx, double *dscore,
                               bool assert_lambda_nonzero = true, const uint32_t *allowed = nullptr, bool wide = false)
{
    asp_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int32_t f = s->f, fp = s->fp;
    const double t_in = asp_now_us();
    ASP_CUDA(cudaMemsetAsync(flags, 0, sizeof(int) * 2, st));
    ASP_CHECK(asp_launch_taumode(ctx, g, &g->sw, dq, nq, f, fp, nullptr, nullptr, dlam, dnorm, nullptr, flags));
    zero_lambda_check_kernel<<<64, 256, 0, st>>>(dlam, nq, flags + 1);
    ASP_LAUNCHED(ctx);
    int h[2] = {0, 0};
    ASP_CUDA(cudaMemcpyAsync(h, flags, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    if (h[0]) ASP_FAIL(ASP_ERR_ZERO_VECTOR, "a query vector is all zeros: its Rayleigh quotient is undefined");
    if (h[1] && assert_lambda_nonzero)
        ASP_FAIL(ASP_ERR_LAMBDA_ZERO, "The lambdas are zero, check the magnitude of items and eps.");   // src/lib.rs:156-159
    ctx->stats["search_host_lambda_us"] = asp_now_us() - t_in;
    if (topk <= 0) return ASP_OK;
    const int rc = search_device_stage(s, g, dq, nq, tau, topk, dlam, dnorm, didx, dscore, allowed, wide);
    ctx->stats["search_host_device_batch_us"] = asp_now_us() - t_in;
    return rc;
}

// Large host batches are pipelined in TWO pieces: a short head (3/64 of the batch) and the rest.  The head's kernels run
// under the H2D copy of the rest (copy stream `up`), the head's D2H copy (copy stream `down`) under the kernels of the
// rest.  The head is sized so that its kernels last about as long as the rest's upload: more or larger pieces were
// measured and lose, because every piece pays its own host synchronisations, GEMM tail and threshold warm-up (an 8k-query
// head costs 7.9 ms against 6.7 ms pro rata at C4; tools/latency.py, profiles/latency_r01.json).
// Result arrays handed in by the caller are usually freshly allocated pageable memory whose first touch page-faults at
// ~3 GB/s inside the D2H copy (10.5 MB per 64k queries: 3 ms after the last kernel); they are touched on this thread
// while the kernels run instead (ctx->on_wait).
constexpr int64_t ASP_PIPE_MIN_BATCH = 32768;
constexpr int ASP_CALL_K_MAX = 1024;          // asp_xs::TOPK_MAX: the longest list the batched exact scan keeps

int asp_search_batch(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                     int64_t *out_idx, double *out_score, double *out_lambda_q)
{
    return asp_search_batch_filtered(s, g, queries, nq, tau, out_idx, out_score, out_lambda_q, nullptr);
}

// k of a per-call search: 1 .. the exact scan's list length
static int check_call_k(int64_t k)
{
    if (k < 1) ASP_FAIL(ASP_ERR_ARG, "k must be >= 1 (got %lld)", (long long)k);
    if (k > ASP_CALL_K_MAX) ASP_FAIL(ASP_ERR_UNSUPPORTED, "k = %lld is beyond the %d results the exact scan keeps per query", (long long)k, ASP_CALL_K_MAX);
    return ASP_OK;
}

static int search_batch_topk(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t topk,
                             bool wide, int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits);

int asp_search_batch_filtered(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                              int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits)
{
    return search_batch_topk(s, g, queries, nq, tau, g ? g->gp.topk : 0, false, out_idx, out_score, out_lambda_q, allowed_bits);
}

int asp_search_batch_k(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t k,
                       int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits)
{
    if (!s || !g || (nq > 0 && (!queries || !out_idx || !out_score))) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch_k: NULL argument");
    ASP_CHECK(check_call_k(k));
    return search_batch_topk(s, g, queries, nq, tau, k, true, out_idx, out_score, out_lambda_q, allowed_bits);
}

// topk: the graph's (src/lib.rs:169) or the call's k (wide: the _k route, see search_device_batch)
static int search_batch_topk(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t topk,
                             bool wide, int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits)
{
    if (!s || !g || (nq > 0 && (!queries || !out_idx || !out_score))) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch: NULL argument");
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch: item lambdas have not been computed");
    if (g->nnodes != s->f)
        ASP_FAIL(ASP_ERR_ARG, "graph has %lld nodes but items have %d features", (long long)g->nnodes, s->f);
    if (nq == 0) return ASP_OK;
    if (s->f > 6144) ASP_FAIL(ASP_ERR_UNSUPPORTED, "search supports at most 6144 features (got %d)", s->f);
    asp_ctx *ctx = s->ctx;
    const double t_call = asp_now_us();
    struct CallTimer { asp_ctx *c; double t0; ~CallTimer() { c->stats["search_host_call_us"] = asp_now_us() - t0; } } call_timer{ctx, t_call};
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int32_t f = s->f, fp = s->fp;

    asp_scratch sc(st);
    double *dq = nullptr, *dlam = nullptr, *dnorm = nullptr, *dscore = nullptr;
    int64_t *didx = nullptr;
    int *flags = nullptr;
    ASP_CHECK(sc.get(&dq, (size_t)nq * fp));
    ASP_CHECK(sc.get(&dlam, (size_t)nq));
    ASP_CHECK(sc.get(&dnorm, (size_t)nq));
    ASP_CHECK(sc.get(&flags, 2));
    if (topk > 0) {
        ASP_CHECK(sc.get(&didx, (size_t)nq * topk));
        ASP_CHECK(sc.get(&dscore, (size_t)nq * topk));
    }
    uint32_t *dallowed = nullptr;                                 // once per call, before the batch is split
    int rc = upload_allowed(sc, allowed_bits, s->n_local, &dallowed);
    const char *nopipe = getenv("ASP_NO_PIPELINE");
    const bool host_io = !asp_is_device_ptr(queries) && !asp_is_device_ptr(out_idx) && !asp_is_device_ptr(out_score) &&
                         (!out_lambda_q || !asp_is_device_ptr(out_lambda_q));
    int64_t head = std::max<int64_t>(1024, (nq * 3 / 64 + 127) / 128 * 128);   // 3072 of 65536: its kernels (~2.5 ms) cover most of the rest's upload
    if (const char *e = getenv("ASP_PIPE_HEAD")) { const long v = atol(e); if (v >= 128 && v < nq) head = v; }   // tuning knob
    auto prefault = [=](int64_t q0, int64_t qn) {                 // first touch of the caller's result pages
        if (out_lambda_q) memset(out_lambda_q + q0, 0, sizeof(double) * qn);
        if (topk > 0) {
            memset(out_idx + q0 * topk, 0, sizeof(int64_t) * (size_t)qn * topk);
            memset(out_score + q0 * topk, 0, sizeof(double) * (size_t)qn * topk);
        }
    };
    const bool touch = host_io && (size_t)nq * (topk + 1) * 16 >= (1u << 18);
    if (rc == ASP_OK && host_io && nq >= ASP_PIPE_MIN_BATCH && !(nopipe && nopipe[0] == '1')) {
        if (!ctx->up_stream) {                                     // streams and events live as long as the context
            ASP_CUDA(cudaStreamCreateWithFlags(&ctx->up_stream, cudaStreamNonBlocking));
            ASP_CUDA(cudaStreamCreateWithFlags(&ctx->down_stream, cudaStreamNonBlocking));
        }
        for (auto &e : ctx->pipe_ev)
            if (!e) ASP_CUDA(cudaEventCreate(&e));
        const int nch = 2;
        const int64_t bounds[3] = {0, head, nq};
        // every call ends with both copy streams and the compute stream drained, so the events are free again
        cudaEvent_t *const up = ctx->pipe_ev, *const done = ctx->pipe_ev + 2;
        cudaEvent_t *const start_c = ctx->pipe_ev + 4;             // timeline diagnostics (search_pipe_* stats)
        const cudaEvent_t alloc_ready = ctx->pipe_ev[6];
        // the copy stream may touch dq only once the allocation is ordered on st
        cudaEventRecord(alloc_ready, st);
        cudaStreamWaitEvent(ctx->up_stream, alloc_ready, 0);
        for (int c = 0; c < nch && rc == ASP_OK; ++c) {
            const int64_t q0 = bounds[c], qn = bounds[c + 1] - q0;
            rc = upload_pitched(ctx->up_stream, queries + q0 * f, qn, f, fp, dq + q0 * fp);
            if (rc == ASP_OK && cudaEventRecord(up[c], ctx->up_stream) != cudaSuccess) rc = ASP_ERR_CUDA;
        }
        prefault(0, head);                                         // under the head's upload
        for (int c = 0; c < nch && rc == ASP_OK; ++c) {
            const int64_t q0 = bounds[c], qn = bounds[c + 1] - q0;
            cudaStreamWaitEvent(st, up[c], 0);
            cudaEventRecord(start_c[c], st);
            if (c == 1) ctx->on_wait = [=]() { prefault(head, nq - head); };   // under the kernels of the rest (the head's are too short)
            rc = search_device_batch(s, g, dq + q0 * fp, qn, tau, topk, dlam + q0, dnorm + q0, flags,
                                     didx ? didx + q0 * topk : nullptr, dscore ? dscore + q0 * topk : nullptr, true, dallowed,
                                     wide);
            if (ctx->on_wait) { auto fn = std::move(ctx->on_wait); ctx->on_wait = nullptr; if (rc == ASP_OK) fn(); }
            if (rc != ASP_OK) break;
            // results of this piece: D2H on the second copy stream (for pageable destinations the runtime stages the copy
            // and returns when it has landed; the piece is small next to the kernels that follow)
            cudaEventRecord(done[c], st);
            cudaStreamWaitEvent(ctx->down_stream, done[c], 0);
            if (out_lambda_q)
                cudaMemcpyAsync(out_lambda_q + q0, dlam + q0, sizeof(double) * qn, cudaMemcpyDeviceToHost, ctx->down_stream);
            if (topk > 0) {
                cudaMemcpyAsync(out_idx + q0 * topk, didx + q0 * topk, sizeof(int64_t) * (size_t)qn * topk, cudaMemcpyDeviceToHost, ctx->down_stream);
                cudaMemcpyAsync(out_score + q0 * topk, dscore + q0 * topk, sizeof(double) * (size_t)qn * topk, cudaMemcpyDeviceToHost, ctx->down_stream);
            }
        }
        const cudaError_t e1 = cudaStreamSynchronize(ctx->up_stream), e2 = cudaStreamSynchronize(ctx->down_stream);
        if (rc == ASP_OK && (e1 != cudaSuccess || e2 != cudaSuccess)) {
            asp_set_error("pipelined search: copy stream failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
            rc = ASP_ERR_CUDA;
        }
        if (rc == ASP_OK) {                                        // device timeline relative to the start of the uploads
            float ms = 0.f;
            const char *names[6] = {"search_pipe_up0_ms", "search_pipe_up1_ms", "search_pipe_start0_ms", "search_pipe_done0_ms",
                                    "search_pipe_start1_ms", "search_pipe_done1_ms"};
            cudaEvent_t evs[6] = {up[0], up[1], start_c[0], done[0], start_c[1], done[1]};
            for (int i = 0; i < 6; ++i)
                if (cudaEventElapsedTime(&ms, alloc_ready, evs[i]) == cudaSuccess) ctx->stats[names[i]] = ms; else cudaGetLastError();
        }
        ctx->stats["search_pipeline_chunks"] = nch;
    } else if (rc == ASP_OK) {
        rc = upload_pitched(st, queries, nq, f, fp, dq);
        if (touch) ctx->on_wait = [=]() { prefault(0, nq); };
        if (rc == ASP_OK) rc = search_device_batch(s, g, dq, nq, tau, topk, dlam, dnorm, flags, didx, dscore, true, dallowed, wide);
        if (ctx->on_wait) { auto fn = std::move(ctx->on_wait); ctx->on_wait = nullptr; if (rc == ASP_OK) fn(); }
        if (rc == ASP_OK && out_lambda_q) rc = asp_copy_out(ctx, out_lambda_q, dlam, sizeof(double) * nq);
        if (rc == ASP_OK && topk > 0) {
            rc = asp_copy_out(ctx, out_idx, didx, sizeof(int64_t) * (size_t)nq * topk);
            if (rc == ASP_OK) rc = asp_copy_out(ctx, out_score, dscore, sizeof(double) * (size_t)nq * topk);
            ASP_CUDA(cudaStreamSynchronize(st));
        }
        ctx->stats["search_pipeline_chunks"] = 1;
    }
    return rc;
}

// Tau sweep (DESIGN §2 item 8): lambda_q once, then the taus that qualify for the tensor-core pass with k <= 16 in groups of at
// most asp_sweep::NT_MAX, one candidate pass per group, and every other tau through the per-call-k search, in the caller's
// order.  A lone qualifying tau takes the per-tau route too.  Each tau's rows are those of asp_search_batch_k at that tau.
int asp_search_batch_taus(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, const double *taus,
                          int64_t ntau, int64_t k, int64_t *out_idx, double *out_score, double *out_lambda_q,
                          const uint8_t *allowed_bits)
{
    if (!s || !g || !taus || (nq > 0 && (!queries || !out_idx || !out_score))) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch_taus: NULL argument");
    ASP_CHECK(check_call_k(k));
    if (ntau < 1) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch_taus: at least one tau is needed (got %lld)", (long long)ntau);
    for (int64_t t = 0; t < ntau; ++t)
        if (!std::isfinite(taus[t])) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch_taus: tau %lld is not finite", (long long)t);
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "asp_search_batch: item lambdas have not been computed");
    if (g->nnodes != s->f)
        ASP_FAIL(ASP_ERR_ARG, "graph has %lld nodes but items have %d features", (long long)g->nnodes, s->f);
    if (nq == 0) return ASP_OK;
    if (s->f > 6144) ASP_FAIL(ASP_ERR_UNSUPPORTED, "search supports at most 6144 features (got %d)", s->f);
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t rows = (size_t)nq * k;

    asp_scratch sc(st);
    double *dq = nullptr, *dlam = nullptr, *dnorm = nullptr, *dscore = nullptr;
    int64_t *didx = nullptr;
    int *flags = nullptr;
    ASP_CHECK(sc.get(&dq, (size_t)nq * s->fp));
    ASP_CHECK(sc.get(&dlam, (size_t)nq));
    ASP_CHECK(sc.get(&dnorm, (size_t)nq));
    ASP_CHECK(sc.get(&flags, 2));
    ASP_CHECK(sc.get(&didx, rows * ntau));
    ASP_CHECK(sc.get(&dscore, rows * ntau));
    uint32_t *dallowed = nullptr;
    ASP_CHECK(upload_allowed(sc, allowed_bits, s->n_local, &dallowed));
    ASP_CHECK(upload_pitched(st, queries, nq, s->f, s->fp, dq));
    ASP_CHECK(search_device_batch(s, g, dq, nq, taus[0], 0, dlam, dnorm, flags, nullptr, nullptr, true, dallowed));   // lambda_q, panics

    // fused groups: the qualifying taus split into ceil(n / NT_MAX) groups of near-equal size (two or more each)
    std::vector<int> fused;
    for (int64_t t = 0; t < ntau; ++t)
        if (k <= 16 && search_takes_tc(s, nq, k, taus[t], false)) fused.push_back((int)t);
    if (fused.size() < 2) fused.clear();
    const int ngroups = (int)asp_ceil_div((int64_t)fused.size(), asp_sweep::NT_MAX);
    std::vector<int> group_of(ntau, -1);
    for (size_t i = 0; i < fused.size(); ++i) group_of[fused[i]] = (int)(i * ngroups / fused.size());

    for (const char *key : {"sweep_stage1_ms", "sweep_stage2_ms", "sweep_emitted"}) ctx->stats[key] = 0.0;
    std::vector<int64_t> slow(ntau, 0);
    std::vector<bool> done(ntau, false);
    for (int64_t t = 0; t < ntau; ++t) {
        if (done[t]) continue;
        if (group_of[t] < 0) {
            ctx->stats["search_slow_queries"] = 0.0;
            ASP_CHECK(search_device_stage(s, g, dq, nq, taus[t], k, dlam, dnorm, didx + t * rows, dscore + t * rows, dallowed, true));
            slow[t] = (int64_t)ctx->stats["search_slow_queries"];
            done[t] = true;
            continue;
        }
        std::vector<int> members;
        std::vector<double> gt;
        std::vector<int64_t *> gi;
        std::vector<double *> gs;
        for (int64_t u = t; u < ntau; ++u)
            if (group_of[u] == group_of[t]) {
                members.push_back((int)u); gt.push_back(taus[u]); gi.push_back(didx + u * rows); gs.push_back(dscore + u * rows);
            }
        std::vector<int64_t> gslow(members.size(), 0);
        ASP_CHECK(asp_search_tc_sweep(s, dq, nq, s->fp, dlam, dnorm, gt.data(), (int)members.size(), k, gi.data(), gs.data(), dallowed,
                                      gslow.data()));
        ASP_CUDA(cudaStreamSynchronize(st));
        for (size_t i = 0; i < members.size(); ++i) { slow[members[i]] = gslow[i]; done[members[i]] = true; }
    }

    if (out_lambda_q) ASP_CHECK(asp_copy_out(ctx, out_lambda_q, dlam, sizeof(double) * nq));
    ASP_CHECK(asp_copy_out(ctx, out_idx, didx, sizeof(int64_t) * rows * ntau));
    ASP_CHECK(asp_copy_out(ctx, out_score, dscore, sizeof(double) * rows * ntau));
    ASP_CUDA(cudaStreamSynchronize(st));
    double total = 0.0;
    for (int64_t t = 0; t < ntau; ++t) {
        total += (double)slow[t];
        ctx->stats["sweep_slow_queries_" + std::to_string(t)] = (double)slow[t];
    }
    ctx->stats["search_slow_queries"] = total;
    ctx->stats["sweep_fused_taus"] = (double)fused.size();
    ctx->stats["sweep_stage1_passes"] = ngroups;
    ctx->stats["sweep_emitted_per_query"] = ngroups ? ctx->stats["sweep_emitted"] / ((double)nq * ngroups) : 0.0;
    return ASP_OK;
}

int64_t asp_hybrid_pool(int64_t n_total, int64_t topk, int64_t pool)
{
    int64_t m = pool > 0 ? pool : std::min<int64_t>(2 * topk, 31);   // H2: shortlist length (31: the longest tensor-core list)
    if (m < topk) m = topk;
    return std::min(m, n_total);
}

// Hybrid search (src/lib.rs:182-219 -> the crate's search_lambda_aware_hybrid; restatement H1-H3 of the header): the cosine
// shortlist is the search above at tau = 1 with topk = pool (same candidate passes, same exact stage 2), the re-ranking is
// hybrid.cuh.  No lambda_q != 0 assertion (search_hybrid has none).
int asp_search_hybrid_batch(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                            int64_t *out_idx, double *out_score, double *out_lambda_q)
{
    return asp_search_hybrid_batch_filtered(s, g, queries, nq, tau, pool, out_idx, out_score, out_lambda_q, nullptr);
}

// Filtered: the shortlist is the m ALLOWED items of largest cosine (the filtered search at tau = 1), m still from n.
static int hybrid_batch_topk(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                             int64_t topk, bool wide, int64_t *out_idx, double *out_score, double *out_lambda_q,
                             const uint8_t *allowed_bits);

int asp_search_hybrid_batch_filtered(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                                     int64_t pool, int64_t *out_idx, double *out_score, double *out_lambda_q,
                                     const uint8_t *allowed_bits)
{
    return hybrid_batch_topk(s, g, queries, nq, tau, pool, g ? g->gp.topk : 0, false, out_idx, out_score, out_lambda_q, allowed_bits);
}

int asp_search_hybrid_batch_k(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                              int64_t k, int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits)
{
    if (!s || !g || (nq > 0 && (!queries || !out_idx || !out_score)))
        ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_batch_k: NULL argument");
    ASP_CHECK(check_call_k(k));
    return hybrid_batch_topk(s, g, queries, nq, tau, pool, k, true, out_idx, out_score, out_lambda_q, allowed_bits);
}

// topk: the graph's (src/lib.rs:214) or the call's k, which also sets the default shortlist (asp_hybrid_pool)
static int hybrid_batch_topk(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                             int64_t topk, bool wide, int64_t *out_idx, double *out_score, double *out_lambda_q,
                             const uint8_t *allowed_bits)
{
    if (!s || !g || (nq > 0 && (!queries || !out_idx || !out_score)))
        ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_batch: NULL argument");
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_batch: item lambdas have not been computed");
    if (g->nnodes != s->f)
        ASP_FAIL(ASP_ERR_ARG, "graph has %lld nodes but items have %d features", (long long)g->nnodes, s->f);
    if (s->n_local != s->n_total)
        ASP_FAIL(ASP_ERR_UNSUPPORTED, "asp_search_hybrid_batch needs every item on this GPU (rows [%lld, %lld) of %lld are here): "
                 "the shortlist is a property of the whole item set", (long long)s->row0, (long long)(s->row0 + s->n_local),
                 (long long)s->n_total);
    if (nq == 0) return ASP_OK;
    if (s->f > 6144) ASP_FAIL(ASP_ERR_UNSUPPORTED, "search supports at most 6144 features (got %d)", s->f);
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int32_t f = s->f, fp = s->fp;
    const int64_t m = asp_hybrid_pool(s->n_local, topk, pool);
    const bool whole_set = (m >= s->n_local);                     // the shortlist is every item: H3 is the plain search
    if (!whole_set && m > 1024)
        ASP_FAIL(ASP_ERR_UNSUPPORTED, "hybrid search: a shortlist of %lld items is beyond the 1024 the exact scan keeps per query "
                 "(use pool >= nitems = %lld for no shortlist at all)", (long long)m, (long long)s->n_local);

    asp_scratch scratch(st);
    double *dq = nullptr, *dlam = nullptr, *dnorm = nullptr, *pscore = nullptr, *dscore = nullptr;
    int64_t *pidx = nullptr, *didx = nullptr;
    int *flags = nullptr;
    ASP_CHECK(scratch.get(&dq, (size_t)nq * fp));
    ASP_CHECK(scratch.get(&dlam, (size_t)nq));
    ASP_CHECK(scratch.get(&dnorm, (size_t)nq));
    ASP_CHECK(scratch.get(&flags, 2));
    if (topk > 0) {
        if (!whole_set) {
            ASP_CHECK(scratch.get(&pidx, (size_t)nq * m));
            ASP_CHECK(scratch.get(&pscore, (size_t)nq * m));
        }
        ASP_CHECK(scratch.get(&didx, (size_t)nq * topk));
        ASP_CHECK(scratch.get(&dscore, (size_t)nq * topk));
    }
    ASP_CHECK(upload_pitched(st, queries, nq, f, fp, dq));
    uint32_t *dallowed = nullptr;
    ASP_CHECK(upload_allowed(scratch, allowed_bits, s->n_local, &dallowed));
    // H1 + H2: lambda_q, then the m largest cosines per query (the score at tau = 1 is the cosine), ties by the smaller index
    if (whole_set)
        ASP_CHECK(search_device_batch(s, g, dq, nq, tau, topk, dlam, dnorm, flags, didx, dscore, false, dallowed, wide));
    else
        ASP_CHECK(search_device_batch(s, g, dq, nq, 1.0, topk > 0 ? m : 0, dlam, dnorm, flags, pidx, pscore, false, dallowed, wide));
    if (topk > 0 && !whole_set) {
        // H3: reference-order scores of the shortlist, best topk by (score desc, index asc)
        const int64_t total = nq * m;
        const unsigned blocks_r = (unsigned)std::min<int64_t>(asp_ceil_div(total, 256), (int64_t)ctx->num_sms * 8);
        asp_hybrid::hybrid_rescore_kernel<<<blocks_r, 256, 0, st>>>(total, m, dq, fp, s->items, fp, f, s->row0, s->norms, s->lambdas,
                                                                     dnorm, dlam, tau, pidx, pscore);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
        const unsigned blocks_s = (unsigned)std::min<int64_t>(asp_ceil_div(nq, 128), (int64_t)ctx->num_sms * 8);
        asp_hybrid::hybrid_select_kernel<<<blocks_s, 128, 0, st>>>(nq, m, topk, pidx, pscore, didx, dscore);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    if (out_lambda_q) ASP_CHECK(asp_copy_out(ctx, out_lambda_q, dlam, sizeof(double) * nq));
    if (topk > 0) {
        ASP_CHECK(asp_copy_out(ctx, out_idx, didx, sizeof(int64_t) * (size_t)nq * topk));
        ASP_CHECK(asp_copy_out(ctx, out_score, dscore, sizeof(double) * (size_t)nq * topk));
    }
    ASP_CUDA(cudaStreamSynchronize(st));
    ctx->stats["hybrid_pool"] = (double)m;
    return ASP_OK;
}

// One row shard's half of the hybrid search of a row-sharded space: H1, then the shard's own top-m by cosine (the search at
// tau = 1 with topk = m, m from the WHOLE item count) and the H3 score of every slot beside its cosine.  asp_hybrid_merge
// takes the global top-m by cosine from the shards' lists and re-ranks it, which is what the one-GPU shortlist holds.
int asp_search_hybrid_shard(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                            int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q)
{
    return asp_search_hybrid_shard_filtered(s, g, queries, nq, tau, pool, out_idx, out_cos, out_score, out_lambda_q, nullptr);
}

static int hybrid_shard_topk(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                             int64_t topk, bool wide, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q,
                             const uint8_t *allowed_bits);

int asp_search_hybrid_shard_filtered(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                                     int64_t pool, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q,
                                     const uint8_t *allowed_bits)
{
    return hybrid_shard_topk(s, g, queries, nq, tau, pool, g ? g->gp.topk : 0, false, out_idx, out_cos, out_score, out_lambda_q,
                             allowed_bits);
}

int asp_search_hybrid_shard_k(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                              int64_t k, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q,
                              const uint8_t *allowed_bits)
{
    if (!s || !g || (nq > 0 && (!queries || !out_idx || !out_score)))
        ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_shard_k: NULL argument");
    ASP_CHECK(check_call_k(k));
    return hybrid_shard_topk(s, g, queries, nq, tau, pool, k, true, out_idx, out_cos, out_score, out_lambda_q, allowed_bits);
}

static int hybrid_shard_topk(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                             int64_t topk, bool wide, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q,
                             const uint8_t *allowed_bits)
{
    if (!s || !g || (nq > 0 && (!queries || !out_idx || !out_score)))
        ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_shard: NULL argument");
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_shard: item lambdas have not been computed");
    if (g->nnodes != s->f)
        ASP_FAIL(ASP_ERR_ARG, "graph has %lld nodes but items have %d features", (long long)g->nnodes, s->f);
    if (nq == 0) return ASP_OK;
    if (s->f > 6144) ASP_FAIL(ASP_ERR_UNSUPPORTED, "search supports at most 6144 features (got %d)", s->f);
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int32_t f = s->f, fp = s->fp;
    const int64_t m = asp_hybrid_pool(s->n_total, topk, pool);
    const bool whole_set = (m >= s->n_total);
    if (!whole_set && m > 1024)
        ASP_FAIL(ASP_ERR_UNSUPPORTED, "hybrid search: a shortlist of %lld items is beyond the 1024 the exact scan keeps per query "
                 "(use pool >= nitems = %lld for no shortlist at all)", (long long)m, (long long)s->n_total);
    if (!whole_set && topk > 0 && !out_cos) ASP_FAIL(ASP_ERR_ARG, "asp_search_hybrid_shard: NULL out_cos");
    const int64_t width = whole_set ? topk : m;                   // entries per query of the outputs
    const int64_t kl = std::min(m, s->n_local);                   // a shard smaller than m answers all its rows

    asp_scratch scratch(st);
    double *dq = nullptr, *dlam = nullptr, *dnorm = nullptr, *dcos = nullptr, *dscore = nullptr;
    int64_t *didx = nullptr;
    int *flags = nullptr;
    ASP_CHECK(scratch.get(&dq, (size_t)nq * fp));
    ASP_CHECK(scratch.get(&dlam, (size_t)nq));
    ASP_CHECK(scratch.get(&dnorm, (size_t)nq));
    ASP_CHECK(scratch.get(&flags, 2));
    if (topk > 0) {
        ASP_CHECK(scratch.get(&didx, (size_t)nq * width));
        ASP_CHECK(scratch.get(&dscore, (size_t)nq * width));
        if (!whole_set) ASP_CHECK(scratch.get(&dcos, (size_t)nq * width));
    }
    ASP_CHECK(upload_pitched(st, queries, nq, f, fp, dq));
    uint32_t *dallowed = nullptr;
    ASP_CHECK(upload_allowed(scratch, allowed_bits, s->n_local, &dallowed));
    if (whole_set) {
        // no shortlist: the shard's best topk by the lambda-aware score, merged like asp_search_batch's lists
        ASP_CHECK(search_device_batch(s, g, dq, nq, tau, topk, dlam, dnorm, flags, didx, dscore, false, dallowed, wide));
    } else {
        int64_t *sidx = didx;
        double *scos = dcos;
        if (topk > 0 && kl < m) {
            ASP_CHECK(scratch.get(&sidx, (size_t)nq * kl));
            ASP_CHECK(scratch.get(&scos, (size_t)nq * kl));
        }
        // the score at tau = 1 is the cosine
        ASP_CHECK(search_device_batch(s, g, dq, nq, 1.0, topk > 0 ? kl : 0, dlam, dnorm, flags, sidx, scos, false, dallowed, wide));
        if (topk > 0) {
            if (kl < m) {                                         // lists padded to m with -1 / NaN
                ASP_CUDA(cudaMemsetAsync(didx, 0xff, sizeof(int64_t) * (size_t)nq * m, st));
                ASP_CUDA(cudaMemsetAsync(dcos, 0xff, sizeof(double) * (size_t)nq * m, st));
                if (kl > 0) {
                    ASP_CUDA(cudaMemcpy2DAsync(didx, sizeof(int64_t) * m, sidx, sizeof(int64_t) * kl, sizeof(int64_t) * kl,
                                               (size_t)nq, cudaMemcpyDeviceToDevice, st));
                    ASP_CUDA(cudaMemcpy2DAsync(dcos, sizeof(double) * m, scos, sizeof(double) * kl, sizeof(double) * kl,
                                               (size_t)nq, cudaMemcpyDeviceToDevice, st));
                }
            }
            const int64_t total = nq * m;
            const unsigned blocks = (unsigned)std::min<int64_t>(asp_ceil_div(total, 256), (int64_t)ctx->num_sms * 8);
            asp_hybrid::hybrid_rescore_kernel<<<blocks, 256, 0, st>>>(total, m, dq, fp, s->items, fp, f, s->row0, s->norms,
                                                                       s->lambdas, dnorm, dlam, tau, didx, dscore);
            ASP_CUDA(cudaGetLastError());
            ASP_LAUNCHED(ctx);
        }
    }
    if (out_lambda_q) ASP_CHECK(asp_copy_out(ctx, out_lambda_q, dlam, sizeof(double) * nq));
    if (topk > 0) {
        ASP_CHECK(asp_copy_out(ctx, out_idx, didx, sizeof(int64_t) * (size_t)nq * width));
        ASP_CHECK(asp_copy_out(ctx, out_score, dscore, sizeof(double) * (size_t)nq * width));
        if (!whole_set) ASP_CHECK(asp_copy_out(ctx, out_cos, dcos, sizeof(double) * (size_t)nq * width));
    }
    ASP_CUDA(cudaStreamSynchronize(st));
    ctx->stats["hybrid_pool"] = (double)m;
    return ASP_OK;
}

int asp_hybrid_merge(asp_ctx *ctx, const int64_t *idx, const double *cosv, const double *score, int parts, int64_t nq, int64_t m,
                     int64_t topk, int64_t *out_idx, double *out_score)
{
    if (!ctx || parts <= 0 || nq < 0 || m < 0 || topk < 0 ||
        (nq > 0 && topk > 0 && (!idx || !cosv || !score || !out_idx || !out_score)))
        ASP_FAIL(ASP_ERR_ARG, "asp_hybrid_merge: bad argument");
    if (nq == 0 || topk == 0) return ASP_OK;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t n_in = (size_t)parts * nq * m, n_pool = (size_t)nq * m, n_out = (size_t)nq * topk;
    asp_scratch scratch(st);
    int64_t *d_idx = nullptr, *d_pidx = nullptr, *d_oidx = nullptr;
    double *d_cos = nullptr, *d_sc = nullptr, *d_psc = nullptr, *d_osc = nullptr;
    ASP_CHECK(scratch.get(&d_idx, n_in));
    ASP_CHECK(scratch.get(&d_cos, n_in));
    ASP_CHECK(scratch.get(&d_sc, n_in));
    ASP_CHECK(scratch.get(&d_pidx, n_pool));
    ASP_CHECK(scratch.get(&d_psc, n_pool));
    ASP_CHECK(scratch.get(&d_oidx, n_out));
    ASP_CHECK(scratch.get(&d_osc, n_out));
    if (n_in) {
        ASP_CUDA(cudaMemcpyAsync(d_idx, idx, sizeof(int64_t) * n_in, cudaMemcpyDefault, st));
        ASP_CUDA(cudaMemcpyAsync(d_cos, cosv, sizeof(double) * n_in, cudaMemcpyDefault, st));
        ASP_CUDA(cudaMemcpyAsync(d_sc, score, sizeof(double) * n_in, cudaMemcpyDefault, st));
    }
    ASP_CUDA(cudaMemsetAsync(d_pidx, 0xff, sizeof(int64_t) * n_pool, st));   // -1: a position no slot reaches stays padding
    if (n_in) {
        const unsigned blocks = (unsigned)std::min<int64_t>(asp_ceil_div((int64_t)n_in, 256), (int64_t)ctx->num_sms * 8);
        asp_hybrid::hybrid_merge_kernel<<<blocks, 256, 0, st>>>((int64_t)n_in, parts, nq, m, d_idx, d_cos, d_sc, d_pidx, d_psc);
        ASP_CUDA(cudaGetLastError());
        ASP_LAUNCHED(ctx);
    }
    const unsigned blocks_s = (unsigned)std::min<int64_t>(asp_ceil_div(nq, 128), (int64_t)ctx->num_sms * 8);
    asp_hybrid::hybrid_select_kernel<<<blocks_s, 128, 0, st>>>(nq, m, topk, d_pidx, d_psc, d_oidx, d_osc);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    ASP_CHECK(asp_copy_out(ctx, out_idx, d_oidx, sizeof(int64_t) * n_out));
    ASP_CHECK(asp_copy_out(ctx, out_score, d_osc, sizeof(double) * n_out));
    ASP_CUDA(cudaStreamSynchronize(st));
    return ASP_OK;
}

int asp_debug_tc_dots(const asp_space *s, const double *queries, int64_t nq, float *out)
{
    if (!s || !queries || !out || nq <= 0) ASP_FAIL(ASP_ERR_ARG, "asp_debug_tc_dots: bad argument");
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "asp_debug_tc_dots: build the space first");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // test hook: query norms on the host (left to right), lambdas irrelevant
    std::vector<double> hq((size_t)nq * s->f), hz(2 * nq, 0.0);
    ASP_CUDA(cudaMemcpyAsync(hq.data(), queries, sizeof(double) * hq.size(), cudaMemcpyDefault, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < nq; ++i) {
        double n2 = 0.0;
        for (int j = 0; j < s->f; ++j) n2 += hq[i * s->f + j] * hq[i * s->f + j];
        hz[nq + i] = sqrt(n2);
    }
    asp_scratch sc(st);
    double *dq = nullptr, *dz = nullptr;
    float *dd = nullptr;
    ASP_CHECK(sc.get(&dq, (size_t)nq * s->fp));
    ASP_CHECK(sc.get(&dz, 2 * (size_t)nq));
    ASP_CHECK(sc.get(&dd, (size_t)nq * s->n_local));
    ASP_CUDA(cudaMemcpyAsync(dz, hz.data(), sizeof(double) * 2 * nq, cudaMemcpyHostToDevice, st));
    ASP_CUDA(cudaMemsetAsync(dd, 0, sizeof(float) * (size_t)nq * s->n_local, st));
    int rc = upload_pitched(ctx->stream, hq.data(), nq, s->f, s->fp, dq);
    if (rc == ASP_OK) rc = asp_search_tc_impl(s, dq, nq, s->fp, dz, dz + nq, 1.0, 1, nullptr, nullptr, dd);
    if (rc == ASP_OK) rc = asp_copy_out(ctx, out, dd, sizeof(float) * (size_t)nq * s->n_local);
    ASP_CUDA(cudaStreamSynchronize(st));
    return rc;
}

int asp_topk_merge(asp_ctx *ctx, const int64_t *idx, const double *score, int parts, int64_t nq, int64_t topk,
                   int64_t *out_idx, double *out_score)
{
    if (!ctx || !idx || !score || !out_idx || !out_score || parts <= 0) ASP_FAIL(ASP_ERR_ARG, "asp_topk_merge: bad argument");
    if (nq == 0 || topk == 0) return ASP_OK;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t n_in = (size_t)parts * nq * topk, n_out = (size_t)nq * topk;
    asp_scratch sc(st);
    int64_t *d_idx = nullptr, *d_oidx = nullptr;
    double *d_sc = nullptr, *d_osc = nullptr;
    ASP_CHECK(sc.get(&d_idx, n_in));
    ASP_CHECK(sc.get(&d_sc, n_in));
    ASP_CHECK(sc.get(&d_oidx, n_out));
    ASP_CHECK(sc.get(&d_osc, n_out));
    ASP_CUDA(cudaMemcpyAsync(d_idx, idx, sizeof(int64_t) * n_in, cudaMemcpyDefault, st));
    ASP_CUDA(cudaMemcpyAsync(d_sc, score, sizeof(double) * n_in, cudaMemcpyDefault, st));
    int rc = asp_topk_merge_impl(ctx, d_idx, d_sc, parts, nq, topk, d_oidx, d_osc);
    if (rc == ASP_OK) rc = asp_copy_out(ctx, out_idx, d_oidx, sizeof(int64_t) * n_out);
    if (rc == ASP_OK) rc = asp_copy_out(ctx, out_score, d_osc, sizeof(double) * n_out);
    ASP_CUDA(cudaStreamSynchronize(st));
    return rc;
}

// ------------------------------------------------------------------ range search (csrc/range.cu)
int asp_search_range_batch(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, double min_score,
                           const uint8_t *allowed_bits, int64_t max_hits, int64_t *out_counts, double *out_lambda_q,
                           asp_range_result **out)
{
    if (!s || !g || !out || nq < 0 || (nq > 0 && (!queries || !out_counts))) ASP_FAIL(ASP_ERR_ARG, "asp_search_range_batch: NULL argument");
    *out = nullptr;
    if (!s->have_lambdas) ASP_FAIL(ASP_ERR_ARG, "asp_search_range_batch: item lambdas have not been computed");
    if (g->nnodes != s->f) ASP_FAIL(ASP_ERR_ARG, "graph has %lld nodes but items have %d features", (long long)g->nnodes, s->f);
    if (std::isnan(min_score)) ASP_FAIL(ASP_ERR_ARG, "asp_search_range_batch: min_score is NaN");
    if (std::isnan(tau)) ASP_FAIL(ASP_ERR_ARG, "asp_search_range_batch: tau is NaN");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    asp_range_result *res = new asp_range_result();
    res->ctx = ctx;
    ctx->stats["search_slow_queries"] = 0.0;
    ctx->stats["range_stage1_ms"] = 0.0;
    ctx->stats["range_stage2_ms"] = 0.0;
    const int32_t f = s->f, fp = s->fp;
    const int64_t sub = std::min<int64_t>(std::max<int64_t>(nq, 1), asp_range_sub_batch());
    std::vector<int64_t> h_counts((size_t)nq);
    asp_scratch scratch(st);
    double *dq = nullptr, *dlam = nullptr, *dnorm = nullptr;
    int *flags = nullptr;
    uint32_t *dallowed = nullptr;
    int rc = scratch.get(&dq, (size_t)sub * fp);
    if (rc == ASP_OK) rc = scratch.get(&dlam, (size_t)sub);
    if (rc == ASP_OK) rc = scratch.get(&dnorm, (size_t)sub);
    if (rc == ASP_OK) rc = scratch.get(&flags, 2);
    if (rc == ASP_OK) rc = upload_allowed(scratch, allowed_bits, s->n_local, &dallowed);   // once per call
    for (int64_t q0 = 0; q0 < nq && rc == ASP_OK; q0 += sub) {
        const int64_t qn = std::min(sub, nq - q0);
        rc = upload_pitched(st, queries + q0 * f, qn, f, fp, dq);
        // lambda_q, the zero-vector check and the lambda_q != 0 assertion of the search (topk = 0: no search)
        if (rc == ASP_OK) rc = search_device_batch(s, g, dq, qn, tau, 0, dlam, dnorm, flags, nullptr, nullptr, true, nullptr);
        asp_range_result::Piece p;
        if (rc == ASP_OK)
            rc = asp_range_impl(s, dq, qn, fp, dlam, dnorm, tau, min_score, dallowed, max_hits, res->total, q0, h_counts.data() + q0, &p);
        if (p.n > 0) { res->total += p.n; res->pieces.push_back(std::move(p)); }
        if (rc == ASP_OK && out_lambda_q) rc = asp_copy_out(ctx, out_lambda_q + q0, dlam, sizeof(double) * qn);
    }
    if (rc == ASP_OK && nq > 0) rc = asp_copy_out(ctx, out_counts, h_counts.data(), sizeof(int64_t) * nq);
    if (rc == ASP_OK && cudaStreamSynchronize(st) != cudaSuccess) { asp_set_error("range search: stream failed"); rc = ASP_ERR_CUDA; }
    if (rc != ASP_OK) { asp_range_result_free(res); return rc; }
    *out = res;
    return ASP_OK;
}

int asp_range_result_fetch(const asp_range_result *r, int64_t *out_idx, double *out_score)
{
    if (!r || (r->total > 0 && (!out_idx || !out_score))) ASP_FAIL(ASP_ERR_ARG, "asp_range_result_fetch: NULL argument");
    asp_ctx *ctx = r->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    int64_t o = 0;
    for (const auto &p : r->pieces) {
        ASP_CHECK(asp_copy_out(ctx, out_idx + o, p.idx, sizeof(int64_t) * p.n));
        ASP_CHECK(asp_copy_out(ctx, out_score + o, p.score, sizeof(double) * p.n));
        o += p.n;
    }
    ASP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ASP_OK;
}

void asp_range_result_free(asp_range_result *r)
{
    if (!r) return;
    cudaSetDevice(r->ctx->device);
    delete r;
}

int asp_range_merge(asp_ctx *ctx, int parts, int64_t nq, const int64_t *counts, const int64_t *idx, const double *score,
                    int64_t *out_idx, double *out_score)
{
    if (!ctx || parts <= 0 || nq < 0 || (nq > 0 && !counts)) ASP_FAIL(ASP_ERR_ARG, "asp_range_merge: bad argument");
    if (nq == 0) return ASP_OK;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::vector<int64_t> h_counts((size_t)parts * nq);
    ASP_CUDA(cudaMemcpyAsync(h_counts.data(), counts, sizeof(int64_t) * h_counts.size(), cudaMemcpyDefault, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    int64_t total = 0;
    for (int64_t c : h_counts) {
        if (c < 0) ASP_FAIL(ASP_ERR_ARG, "asp_range_merge: negative count");
        total += c;
    }
    if (total == 0) return ASP_OK;
    if (!idx || !score || !out_idx || !out_score) ASP_FAIL(ASP_ERR_ARG, "asp_range_merge: NULL argument");
    asp_scratch scratch(st);
    int64_t *d_idx = nullptr, *d_oidx = nullptr;
    double *d_sc = nullptr, *d_osc = nullptr;
    ASP_CHECK(scratch.get(&d_idx, (size_t)total));
    ASP_CHECK(scratch.get(&d_sc, (size_t)total));
    ASP_CHECK(scratch.get(&d_oidx, (size_t)total));
    ASP_CHECK(scratch.get(&d_osc, (size_t)total));
    ASP_CUDA(cudaMemcpyAsync(d_idx, idx, sizeof(int64_t) * total, cudaMemcpyDefault, st));
    ASP_CUDA(cudaMemcpyAsync(d_sc, score, sizeof(double) * total, cudaMemcpyDefault, st));
    ASP_CHECK(asp_range_merge_impl(ctx, parts, nq, h_counts.data(), d_idx, d_sc, d_oidx, d_osc));
    ASP_CHECK(asp_copy_out(ctx, out_idx, d_oidx, sizeof(int64_t) * total));
    ASP_CHECK(asp_copy_out(ctx, out_score, d_osc, sizeof(double) * total));
    ASP_CUDA(cudaStreamSynchronize(st));
    return ASP_OK;
}

// Persistence: a graph handle from a stored Laplacian (what asp_graph_csr exported).  feature_graph != 0 also prepares the
// lambda pass (the graph then serves asp_query_lambda / asp_search_batch exactly like the one it was saved from).
int asp_graph_from_csr(asp_ctx *ctx, int64_t nnodes, int64_t nnz, const int64_t *indptr, const int32_t *indices, const double *data,
                       const asp_graph_params *gp, const asp_switches *sw_in, int feature_graph, asp_graph **out_graph)
{
    if (!ctx || !indptr || !indices || !data || !gp || !out_graph || nnodes <= 0 || nnz < 0)
        ASP_FAIL(ASP_ERR_ARG, "asp_graph_from_csr: bad argument");
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    asp_switches sw;
    if (sw_in) sw = *sw_in; else asp_default_switches(&sw);
    ASP_CHECK(check_switches(&sw));
    asp_graph *g = new asp_graph();
    g->ctx = ctx;
    g->gp = *gp;
    if (!g->gp.has_sigma) { g->gp.sigma = gp->eps * 0.5; g->gp.has_sigma = 1; }
    g->sw = sw;
    g->nnodes = nnodes;
    g->nnz = nnz;
    int rc = ASP_OK;
    if (cudaMallocAsync(&g->d_indptr, sizeof(int64_t) * (nnodes + 1), st) != cudaSuccess ||
        cudaMallocAsync(&g->d_indices, sizeof(int32_t) * (nnz > 0 ? nnz : 1), st) != cudaSuccess ||
        cudaMallocAsync(&g->d_data, sizeof(double) * (nnz > 0 ? nnz : 1), st) != cudaSuccess) {
        asp_set_error("out of device memory for the stored Laplacian");
        rc = ASP_ERR_NOMEM;
    }
    if (rc == ASP_OK) rc = asp_copy_in(ctx, g->d_indptr, indptr, sizeof(int64_t) * (nnodes + 1));
    if (rc == ASP_OK) rc = asp_copy_in(ctx, g->d_indices, indices, sizeof(int32_t) * nnz);
    if (rc == ASP_OK) rc = asp_copy_in(ctx, g->d_data, data, sizeof(double) * nnz);
    if (rc == ASP_OK && cudaStreamSynchronize(st) != cudaSuccess) { asp_set_error("upload of the stored Laplacian failed"); rc = ASP_ERR_CUDA; }
    if (rc == ASP_OK && feature_graph) rc = asp_graph_upload_upper(g);
    if (rc != ASP_OK) { asp_free_graph(g); return rc; }
    *out_graph = g;
    return ASP_OK;
}

int asp_graph_switches(const asp_graph *g, asp_switches *sw)
{
    if (!g || !sw) ASP_FAIL(ASP_ERR_ARG, "asp_graph_switches: NULL argument");
    *sw = g->sw;
    return ASP_OK;
}

int asp_item_graph(asp_space *s, const asp_graph_params *gp, const asp_switches *sw_in, asp_graph **out_graph)
{
    if (!s || !gp || !out_graph) ASP_FAIL(ASP_ERR_ARG, "asp_item_graph: NULL argument");
    if (s->world != 1) ASP_FAIL(ASP_ERR_UNSUPPORTED, "asp_item_graph is single-GPU in this version");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_switches sw;
    if (sw_in) sw = *sw_in; else asp_default_switches(&sw);
    ASP_CHECK(check_switches(&sw));
    asp_knn_lists lists;
    asp_graph_params gpe = *gp;
    gpe.k = asp_neighbour_cap(gp, &sw, s->n_total);               // k convention switches (k_counts_self, topk_prunes)
    ASP_CHECK(asp_item_knn(s, &gpe, sw.distance, &lists));
    asp_graph *g = new asp_graph();
    g->ctx = ctx;
    g->gp = *gp;
    if (!g->gp.has_sigma) { g->gp.sigma = gp->eps * 0.5; g->gp.has_sigma = 1; }
    g->sw = sw;
    int rc = asp_assemble_laplacian(ctx, &lists, gp, &sw, g);
    if (rc == ASP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        asp_set_error("item graph: %s", cudaGetErrorString(cudaGetLastError()));
        rc = ASP_ERR_CUDA;
    }
    if (rc != ASP_OK) { asp_free_graph(g); return rc; }
    *out_graph = g;
    return ASP_OK;
}

int asp_item_knn_rows(asp_space *s, const asp_graph_params *gp, const asp_switches *sw_in, int64_t row_begin, int64_t row_end,
                      int32_t *out_idx, double *out_dist, int32_t *out_cnt, int32_t *out_kk)
{
    if (!s || !gp || !out_cnt || !out_kk) ASP_FAIL(ASP_ERR_ARG, "asp_item_knn_rows: NULL argument");
    asp_ctx *ctx = s->ctx;
    ASP_CUDA(cudaSetDevice(ctx->device));
    asp_switches sw;
    if (sw_in) sw = *sw_in; else asp_default_switches(&sw);
    ASP_CHECK(check_switches(&sw));
    asp_knn_lists lists;
    asp_graph_params gpe = *gp;
    gpe.k = asp_neighbour_cap(gp, &sw, s->n_total);
    int rc = asp_item_knn_rows_impl(s, &gpe, sw.distance, row_begin, row_end, &lists);
    if (rc == ASP_OK) {
        const size_t rows = (size_t)lists.m;
        *out_kk = lists.kk;
        if (rows > 0 && out_idx) rc = asp_copy_out(ctx, out_idx, lists.idx, sizeof(int32_t) * rows * lists.kk);
        if (rc == ASP_OK && rows > 0 && out_dist) rc = asp_copy_out(ctx, out_dist, lists.dist, sizeof(double) * rows * lists.kk);
        if (rc == ASP_OK && rows > 0) rc = asp_copy_out(ctx, out_cnt, lists.cnt, sizeof(int32_t) * rows);
        cudaStreamSynchronize(ctx->stream);
    }
    return rc;
}

int asp_graph_from_knn(asp_ctx *ctx, int64_t m, int32_t kk, const int32_t *idx, const double *dist, const int32_t *cnt,
                       const asp_graph_params *gp, const asp_switches *sw_in, asp_graph **out_graph)
{
    if (!ctx || !idx || !dist || !cnt || !gp || !out_graph || m <= 0 || kk <= 0) ASP_FAIL(ASP_ERR_ARG, "asp_graph_from_knn: bad argument");
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    asp_switches sw;
    if (sw_in) sw = *sw_in; else asp_default_switches(&sw);
    ASP_CHECK(check_switches(&sw));
    asp_knn_lists lists;
    ASP_CHECK(lists.alloc(st, m, kk));
    int rc = asp_copy_in(ctx, lists.idx, idx, sizeof(int32_t) * (size_t)m * kk);
    if (rc == ASP_OK) rc = asp_copy_in(ctx, lists.dist, dist, sizeof(double) * (size_t)m * kk);
    if (rc == ASP_OK) rc = asp_copy_in(ctx, lists.cnt, cnt, sizeof(int32_t) * (size_t)m);
    asp_graph *g = nullptr;
    if (rc == ASP_OK) {
        g = new asp_graph();
        g->ctx = ctx;
        g->gp = *gp;
        if (!g->gp.has_sigma) { g->gp.sigma = gp->eps * 0.5; g->gp.has_sigma = 1; }
        g->sw = sw;
        rc = asp_assemble_laplacian(ctx, &lists, gp, &sw, g);
    }
    if (rc == ASP_OK && cudaStreamSynchronize(st) != cudaSuccess) {
        asp_set_error("graph from kNN lists: %s", cudaGetErrorString(cudaGetLastError()));
        rc = ASP_ERR_CUDA;
    }
    if (rc != ASP_OK) { asp_free_graph(g); return rc; }
    *out_graph = g;
    return ASP_OK;
}

}  // extern "C"
