// common.cuh -- shared declarations of the sm_100a implementation of the arrowspace hot path.
#pragma once

#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <functional>
#include <map>
#include <vector>

#include "../../include/arrowspace_b200.h"

// ------------------------------------------------------------------ errors
void asp_set_error(const char *fmt, ...);

#define ASP_CUDA(call)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (call);                                                             \
        if (_e != cudaSuccess) {                                                             \
            asp_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__,      \
                          __LINE__, cudaGetErrorString(_e));                                 \
            return ASP_ERR_CUDA;                                                             \
        }                                                                                    \
    } while (0)

#define ASP_CHECK(expr)                                                                      \
    do {                                                                                     \
        int _rc = (expr);                                                                    \
        if (_rc != ASP_OK) return _rc;                                                       \
    } while (0)

#define ASP_FAIL(code, ...)                                                                  \
    do {                                                                                     \
        asp_set_error(__VA_ARGS__);                                                          \
        return (code);                                                                       \
    } while (0)

// ------------------------------------------------------------------ device scratch
// Owner of stream-ordered device buffers: every buffer taken with get() is given back (cudaFreeAsync on the owner's
// stream) by release() or by the destructor, so no return path leaks one.  Move-only: a moved-from owner holds nothing.
struct asp_scratch {
    cudaStream_t st = nullptr;
    std::vector<void *> ptrs;

    asp_scratch() = default;
    explicit asp_scratch(cudaStream_t s) : st(s) {}
    asp_scratch(const asp_scratch &) = delete;
    asp_scratch &operator=(const asp_scratch &) = delete;
    asp_scratch(asp_scratch &&o) noexcept : st(o.st), ptrs(std::move(o.ptrs)) { o.ptrs.clear(); }
    asp_scratch &operator=(asp_scratch &&o) noexcept
    {
        if (this != &o) { release(); st = o.st; ptrs = std::move(o.ptrs); o.ptrs.clear(); }
        return *this;
    }
    ~asp_scratch() { release(); }

    // count elements of T (count == 0: one element); ASP_ERR_NOMEM with the byte count when the pool has no room
    template <class T> int get(T **out, size_t count)
    {
        const size_t bytes = sizeof(T) * (count ? count : 1);
        void *p = nullptr;
        if (cudaMallocAsync(&p, bytes, st) != cudaSuccess) {
            cudaGetLastError();
            asp_set_error("out of device memory (%zu bytes)", bytes);
            return ASP_ERR_NOMEM;
        }
        ptrs.push_back(p);
        *out = static_cast<T *>(p);
        return ASP_OK;
    }
    void release()
    {
        for (void *p : ptrs) cudaFreeAsync(p, st);
        ptrs.clear();
    }
};

// ------------------------------------------------------------------ handles
struct asp_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    int64_t launches = 0;
    bool use_tma = true;                 // ASP_NO_TMA=1 switches the operand loaders to cp.async
    std::map<std::string, double> stats;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    cudaStream_t up_stream = nullptr, down_stream = nullptr;   // copy streams of the pipelined host search (lazily created)
    cudaEvent_t pipe_ev[7] = {};         // its events (uploads, piece done, piece start, allocation ready), created with the streams
    std::function<void()> on_wait;       // host work the search runs once, right before its long wait for the kernels
};

struct asp_space {
    asp_ctx *ctx = nullptr;
    int64_t n_local = 0, row0 = 0, n_total = 0;
    int32_t f = 0;
    int32_t fp = 0;                      // row pitch in doubles: f rounded up to a multiple of 4, zero padded
    double *items = nullptr;             // device, n_local x fp
    bool owns_items = true;              // false: adopted from the caller (asp_space_adopt)
    double *norms = nullptr;             // device, n_local: sqrt(sum x^2), left-to-right
    double *inv_norms = nullptr;         // device, n_local: 1/norm (0 for zero rows)
    double *nsq = nullptr;               // device, n_local: sum x^2, left-to-right (Euclidean item graph; allocated on first use)
    double *lambdas = nullptr;           // device, n_local
    bool have_lambdas = false;
    CUtensorMap tmap_gram;               // (4, n_local, fp/4), box (4, 32 rows, 32 quads): Gram kernel
    CUtensorMap tmap_rows;               // same tensor, box (4, 128 rows, 4 quads): search / kNN GEMM
    int world = 1, rank = 0;             // shard = Gram segments [rank*8/world, (rank+1)*8/world)
    void *tc_cache = nullptr;            // fp16 split copies (lambda order) for the tcgen05 search path (search_tc.cu), lazily built
};

struct asp_graph {
    asp_ctx *ctx = nullptr;
    int64_t nnodes = 0, nnz = 0;
    asp_graph_params gp;
    asp_switches sw;
    // Laplacian CSR, device + host mirror
    int64_t *d_indptr = nullptr;
    int32_t *d_indices = nullptr;
    double  *d_data = nullptr;
    std::vector<int64_t> h_indptr;
    std::vector<int32_t> h_indices;
    std::vector<double>  h_data;
    // graph-only inputs of the lambda pass (taumode.cu: the symmetrised quadratic form, pre-cut into chunks); feature graphs only
    void *tm_blob = nullptr;
};

// hits of asp_search_range_batch: one device piece per sub-batch (query-major, concatenated in query order)
struct asp_range_result {
    asp_ctx *ctx = nullptr;
    int64_t total = 0;
    struct Piece { int64_t *idx = nullptr; double *score = nullptr; int64_t n = 0; asp_scratch mem; };   // mem owns idx, score
    std::vector<Piece> pieces;
};

// host wall clock in microseconds (diagnostic stats "search_host_*_us": where a call's time goes between the kernels)
#include <chrono>
static inline double asp_now_us()
{
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ------------------------------------------------------------------ launch bookkeeping
#define ASP_LAUNCHED(ctx) ((ctx)->launches++)

static inline int64_t asp_ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// neighbour cap of one node (SURVEY.md Appendix A4 + the unpinned conventions): min(k, topk) when topk prunes, minus the
// node itself when k counts it; never more than m - 1 others
static inline int64_t asp_neighbour_cap(const asp_graph_params *gp, const asp_switches *sw, int64_t m)
{
    int64_t kk = gp->k;
    if (sw && sw->topk_prunes && gp->topk < kk) kk = gp->topk;
    if (sw && sw->k_counts_self) kk -= 1;
    if (kk > m - 1) kk = m - 1;
    return kk < 0 ? 0 : kk;
}

// Item filter of a search: bit i of the packed mask (LSB-first bytes, read as little-endian 32-bit words) says whether local
// row i may be returned.  nullptr = every row.
__device__ __forceinline__ bool asp_allowed(const uint32_t *bits, int64_t i) { return (bits[i >> 5] >> (i & 31)) & 1u; }

// host helpers implemented in api.cu
int  asp_copy_in(asp_ctx *ctx, void *dst_dev, const void *src, size_t bytes);
int  asp_copy_out(asp_ctx *ctx, void *dst, const void *src_dev, size_t bytes);
bool asp_is_device_ptr(const void *p);

// tensormap.cu
int asp_make_items_tmap(CUtensorMap *out, const double *base, int64_t rows, int32_t fp,
                        int box_rows, int box_outer);

// gram.cu
int asp_launch_gram_partials(asp_space *s, double *out_dev);
int asp_launch_gram_reduce(asp_ctx *ctx, const double *segments_dev, int32_t f, double *gram_dev);

// graph_select.cu
struct asp_knn_lists {                    // device buffers, m rows x kk slots
    int64_t m = 0; int32_t kk = 0;
    int32_t *idx = nullptr; double *dist = nullptr; int32_t *cnt = nullptr;
    asp_scratch mem;                      // owns idx, dist, cnt
    int alloc(cudaStream_t st, int64_t rows, int32_t k)   // room for max(rows, 1) rows
    {
        m = rows; kk = k; mem = asp_scratch(st);
        const size_t r = (size_t)(rows > 0 ? rows : 1);
        int rc = mem.get(&idx, r * k);
        if (rc == ASP_OK) rc = mem.get(&dist, r * k);
        if (rc == ASP_OK) rc = mem.get(&cnt, r);
        return rc;
    }
};
int asp_feature_select(asp_ctx *ctx, const double *gram_dev, int32_t f, int64_t n_total,
                       const asp_graph_params *gp, const asp_switches *sw, const int32_t *exact_pairs_dev,
                       const double *exact_sums_dev, int64_t n_exact, asp_knn_lists *lists,
                       int32_t *need_pairs_dev, int64_t need_cap, int32_t *need_count_dev);
int asp_launch_exact_pairs(asp_space *s, const int32_t *pairs_dev, int64_t n_pairs, double *sums_dev);

// csr.cu
int asp_graph_host_mirror(asp_graph *g);
int asp_assemble_laplacian(asp_ctx *ctx, const asp_knn_lists *lists, const asp_graph_params *gp,
                           const asp_switches *sw, asp_graph *g);

// taumode.cu
int asp_graph_upload_upper(asp_graph *g);
void asp_graph_free_upper(asp_graph *g);
int asp_launch_taumode(asp_ctx *ctx, const asp_graph *g, const asp_switches *sw, const double *x_dev,
                       int64_t n, int32_t f, int32_t pitch, double *out_energy, double *out_tau,
                       double *out_lambda, double *out_norm, double *out_inv_norm, int *zero_flag_dev);

// search.cu
int asp_search_impl(const asp_space *s, const asp_graph *g, const double *q_dev, int64_t nq, int32_t qpitch,
                    const double *lambda_q_dev, const double *qnorm_dev, double tau, int64_t topk,
                    int64_t *out_idx_dev, double *out_score_dev, const uint32_t *allowed_dev = nullptr);
int asp_topk_merge_impl(asp_ctx *ctx, const int64_t *idx_dev, const double *score_dev, int parts,
                        int64_t nq, int64_t topk, int64_t *out_idx_dev, double *out_score_dev);

// search_tc.cu (tcgen05 stage 1)
struct asp_tc_batch {                     // device buffers of one batch of query vectors between stage 1 and stage 2
    int64_t nq = 0;
    int nsub = 0, capb = 0, nterms = 0, variant = 0;
    double delta_cos_max = 0.0;
    void *q_hi = nullptr, *q_lo = nullptr;
    float *lam_q32 = nullptr, *delta_q = nullptr;    // visiting order
    double *inv_nq = nullptr, *rho_q = nullptr;
    int32_t *qperm = nullptr, *center = nullptr;     // visiting position -> caller's query index (nullptr: identity)
    float *emit_sc = nullptr;                        // [nq][nsub][capb] approximate scores
    int32_t *emit_ix = nullptr, *emit_cnt = nullptr; // local item indices; [nq][nsub] counts (> capb: overflow)
    uint32_t *theta_glob = nullptr;
    uint32_t *vbits = nullptr;                       // filtered search: the item mask in visiting order
    asp_scratch mem;                                 // owns every buffer above; *b = asp_tc_batch() frees them
};
enum { ASP_TC_ORDER_IDENTITY = 0, ASP_TC_ORDER_LAMBDA = 1, ASP_TC_ORDER_NORM = 2 };   // item order of the operand cache
int asp_tc_stage1(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                  const double *qnorm_dev, double tau, int64_t topk, double score_floor, int force_terms, int capb_override,
                  float *dump_dev, asp_tc_batch *b, bool l2 = false, const uint32_t *allowed_dev = nullptr,
                  const double *sweep_taus = nullptr, int ntau = 1);
int asp_device_max(asp_ctx *ctx, const double *v_dev, int64_t n, double *out);   // max(0, max v), synchronises
// wide: topk up to 128 on the tensor-core route (wide stage 2 from 32 on); otherwise topk <= 32 as the graph-topk entry points use
bool asp_search_tc_supported(const asp_space *s, int64_t nq, int64_t topk, double tau, bool wide = false);
int asp_search_tc_impl(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                       const double *qnorm_dev, double tau, int64_t topk, int64_t *out_idx_dev, double *out_score_dev,
                       float *dump_dev, const uint32_t *allowed_dev = nullptr, bool wide = false);
// Tau sweep: ONE candidate pass for ntau = 2 .. asp_sweep::NT_MAX taus (topk <= 16, each tau asp_search_tc_supported), then
// per tau the search's stage 2 and remedies.  out_idx_dev[u] / out_score_dev[u]: [nq][topk] of tau u; slow_out[u]: the
// queries of tau u that took the exact scan.
int asp_search_tc_sweep(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lambda_q_dev,
                        const double *qnorm_dev, const double *taus, int ntau, int64_t topk, int64_t *const *out_idx_dev,
                        double *const *out_score_dev, const uint32_t *allowed_dev, int64_t *slow_out);
void asp_free_tc_cache(asp_space *s);
int asp_launch_reciprocal(asp_ctx *ctx, const double *x, int64_t n, double *out);
int asp_search_slow_path(const asp_space *s, const double *q_dev, int32_t qpitch, const double *lambda_q_dev,
                         const double *qnorm_dev, double tau, int64_t topk, const int32_t *slow_list_dev, int nslow,
                         int64_t *out_idx_dev, double *out_score_dev, const uint32_t *allowed_dev = nullptr);
int asp_make_f16_tmap(CUtensorMap *out, const void *base, int64_t rows, int32_t kp, int box_rows);
int asp_make_f16_tmap_narrow(CUtensorMap *out, const void *base, int64_t rows, int32_t kp, int box_rows, int nw);

// range.cu (range search after the tcgen05 candidate pass)
int asp_range_impl(const asp_space *s, const double *q_dev, int64_t nq, int32_t qpitch, const double *lam_dev, const double *norm_dev,
                   double tau, double min_score, const uint32_t *allowed_dev, int64_t max_hits, int64_t hits_before, int64_t q_base,
                   int64_t *h_counts, asp_range_result::Piece *out);
int asp_range_merge_impl(asp_ctx *ctx, int parts, int64_t nq, const int64_t *h_counts, const int64_t *idx_dev,
                         const double *score_dev, int64_t *out_idx_dev, double *out_score_dev);

// knn.cu
// distance: ASP_DISTANCE_COSINE | L2 | L2SQ
int asp_item_knn(asp_space *s, const asp_graph_params *gp, int distance, asp_knn_lists *lists);
int asp_item_knn_rows_impl(asp_space *s, const asp_graph_params *gp, int distance, int64_t row_begin, int64_t row_end,
                           asp_knn_lists *lists);
