/*
 * arrowspace_b200.h -- C ABI of the B200-native build-and-search hot path of pyarrowspace.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / numpy types.  Each entry
 * point names the call of the reference binding it replaces (/root/reference, a pyo3 module
 * whose numerics all live in the crate `arrowspace` 0.18.0, Cargo.lock:94-97).  The crate
 * functions below are exactly the ones `src/lib.rs` imports (src/lib.rs:7-11) and calls.
 *
 * Conventions
 *   - every function returns 0 (ASP_OK) or an ASP_ERR_* code; asp_last_error() gives the
 *     message of the last failure on the calling thread;
 *   - `items`, `queries`, outputs may be HOST or DEVICE pointers (detected with
 *     cudaPointerGetAttributes); inputs are copied (src/helpers.rs:45, src/lib.rs:139);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with ASP_ERR_CUDA;
 *   - one asp_ctx per process and GPU; multi-GPU = one process per GPU, each owning a row
 *     shard (asp_shard_rows); the host (torch.distributed / NCCL) moves the small exchange
 *     buffers between the staged calls marked [exchange].
 */
#ifndef ARROWSPACE_B200_H
#define ARROWSPACE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASP_ABI_VERSION 2

/* Fixed reduction geometry of the feature Gram (makes results independent of the GPU count):
 * rows are cut into 32-row units, the units into ASP_GRAM_SEGMENTS contiguous segments (the
 * sharding granularity) and every segment into ASP_GRAM_SLICES contiguous slices.  The Gram is
 * sum_seg ( sum_slice ( in-order DMMA chain over the slice rows ) ), both sums in index order. */
#define ASP_GRAM_SEGMENTS 8
#define ASP_GRAM_SLICES   24
#define ASP_ROW_UNIT      32

enum {
    ASP_OK = 0,
    ASP_ERR_EMPTY = 1,        /* "items must be non-empty 2D array"            src/helpers.rs:27-29 */
    ASP_ERR_ZERO_VECTOR = 2,  /* all-zero vector in the Rayleigh quotient      TAUMODE.md:13 */
    ASP_ERR_LAMBDA_ZERO = 3,  /* "The lambdas are zero, check the magnitude of items and eps."  src/lib.rs:156-159 */
    ASP_ERR_ARG = 4,
    ASP_ERR_NOMEM = 5,        /* a device allocation failed (every path; the message gives the bytes asked for) */
    ASP_ERR_CUDA = 6,         /* no device / CUDA failure: there is no CPU fallback */
    ASP_ERR_UNSUPPORTED = 7,
    ASP_NEED_EXACT = 8,       /* asp_graph_from_gram: decisions inside the rounding band, see below */
    ASP_ERR_LIMIT = 9         /* asp_search_range_batch: more hits than max_hits */
};

/* (eps, k, topk, p, sigma) as parsed by parse_graph_params, src/helpers.rs:48-77.
 * has_sigma == 0  ->  sigma := eps * 0.5 (src/helpers.rs:68-72). */
typedef struct {
    double  eps;
    int64_t k;
    int64_t topk;
    double  p;
    double  sigma;
    int32_t has_sigma;
} asp_graph_params;

/* Named switches for the choices the reference's tests cannot pin (SURVEY.md section 8(c), Appendix A).  The arithmetic
 * lives in the un-vendored crate arrowspace 0.18.0 (Cargo.lock:94-97); the binding only shows the call sites
 * (src/lib.rs:278-289).  Zero-initialised = the default spec of Appendix A.  The same switches, with the same meaning,
 * exist in the CPU oracle (oracle/oracle.h) and every one is parity-tested GPU == oracle. */
enum { ASP_KERNEL_INV_POWER = 0, ASP_KERNEL_GAUSSIAN = 1 };
enum { ASP_TAU_MEDIAN = 0, ASP_TAU_MEDIAN_ABS = 1, ASP_TAU_MEAN = 2, ASP_TAU_FIXED = 3 };
enum { ASP_LAMBDA_BOUNDED = 0, ASP_LAMBDA_SYNTHETIC = 1 };                /* TAUMODE.md:19,25 | TAUMODE.md:8,26-27 */
enum { ASP_SYM_MAX = 0, ASP_SYM_AVG = 1, ASP_SYM_MIN = 2, ASP_SYM_NONE = 3 };  /* GRAPH_VARIABLES.md:8 "symmetrized": rule unpinned */
enum { ASP_LAPLACIAN_COMBINATORIAL = 0, ASP_LAPLACIAN_SYM = 1, ASP_LAPLACIAN_RW = 2 };
enum { ASP_DISTANCE_COSINE = 0, ASP_DISTANCE_L2 = 1, ASP_DISTANCE_L2SQ = 2 };  /* GRAPH_VARIABLES.md:7 | Gram-form Euclidean */
typedef struct {
    int32_t kernel;        /* ASP_KERNEL_*    : w = 1/(1+(d/sigma)^p)  |  exp(-(d/sigma)^p)                      */
    int32_t tau_mode;      /* ASP_TAU_*       : tau of a vector (floored at 1e-9)                                */
    double  tau_fixed;
    int32_t lambda_form;   /* ASP_LAMBDA_*    : E/(E+tau)  |  tau E/(E+tau) + (1-tau) G(x)                        */
    int32_t symmetrise;    /* ASP_SYM_*       : W = max(W,W^T) | (W+W^T)/2 | min(W,W^T) (mutual edges) | W (directed) */
    int32_t laplacian;     /* ASP_LAPLACIAN_* : D - W | I - D^-1/2 W D^-1/2 | I - D^-1 W   (D = row sums of W)   */
    int32_t k_counts_self; /* 1: a node is its own first neighbour, so k keeps k - 1 others                      */
    int32_t topk_prunes;   /* 1: the neighbour cap is min(k, topk) (graph_params.topk also prunes the graph)     */
    int32_t distance;      /* ASP_DISTANCE_*  : 1 - max(0,cos) | sqrt(|a|^2+|b|^2-2<a,b>) | its square (feature and item graph) */
} asp_switches;

typedef struct asp_ctx   asp_ctx;    /* device, streams, scratch */
typedef struct asp_space asp_space;  /* replaces arrowspace::core::ArrowSpace   (src/lib.rs:64-67)  */
typedef struct asp_graph asp_graph;  /* replaces arrowspace::graph::GraphLaplacian (src/lib.rs:26-29) */
typedef struct asp_range_result asp_range_result;   /* hits of asp_search_range_batch, in device memory */

const char *asp_last_error(void);
int  asp_abi_version(void);
void asp_default_switches(asp_switches *sw);

int  asp_ctx_create(int device, asp_ctx **out);
void asp_ctx_destroy(asp_ctx *ctx);
int  asp_ctx_device(const asp_ctx *ctx);
/* Adopt a caller-owned CUDA stream (e.g. torch.cuda.current_stream().cuda_stream); 0 = own stream. */
int  asp_ctx_set_stream(asp_ctx *ctx, void *cuda_stream);
int  asp_ctx_synchronize(asp_ctx *ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t asp_ctx_launch_count(const asp_ctx *ctx);
/* Scratch is served from the device's stream-ordered memory pool and kept there between calls (up to a quarter of the
 * device, env ASP_POOL_KEEP_GB); this returns everything above keep_bytes to the driver (synchronises the stream). */
int asp_ctx_trim(asp_ctx *ctx, size_t keep_bytes);

/* ---- one-call single-GPU path --------------------------------------------------------------
 * Replaces RustBuilder::new().with_lambda_graph(eps,k,topk,p,sigma)...build(rows)
 * (src/lib.rs:278-289): feature graph (nodes = columns of items), Laplacian CSR, per-item lambda. */
int asp_build(asp_ctx *ctx, const double *items, int64_t n, int32_t f,
              const asp_graph_params *gp, const asp_switches *sw,
              asp_space **out_space, asp_graph **out_graph);

/* ---- staged path (what asp_build does; the multi-GPU host calls the stages itself) --------- */

/* Row range [row0,row1) owned by `rank` of `world` (world in {1,2,4,8}): whole Gram segments. */
int asp_shard_rows(int64_t n_total, int world, int rank, int64_t *row0, int64_t *row1);

/* Upload (copy) the row shard of `rank` (of `world`): items_shard is n_local x f row-major f64 and
 * must hold exactly the rows asp_shard_rows(n_total, world, rank) names.  Replaces
 * pyarray2_to_vecvec + ArrowSpace construction (src/helpers.rs:24-46, src/lib.rs:277). */
int asp_space_create(asp_ctx *ctx, const double *items_shard, int64_t n_local, int32_t f,
                     int64_t n_total, int world, int rank, asp_space **out);

/* World-1 space over a device buffer the caller keeps alive until asp_free_space (n x f f64 row-major, f % 4 == 0,
 * 16-byte aligned): no copy.  Used by the multi-GPU item graph so that the all-gathered item matrix (the halo rows
 * of BASELINE.json config C5: 54 GB per rank) exists once.  No reference counterpart (the reference always copies,
 * src/helpers.rs:24-46). */
int asp_space_adopt(asp_ctx *ctx, double *items_dev, int64_t n, int32_t f, asp_space **out);
/* The same for the row shard of `rank` of `world` (rows asp_shard_rows names). */
int asp_space_adopt_shard(asp_ctx *ctx, double *items_dev, int64_t n_local, int32_t f, int64_t n_total, int world, int rank,
                          asp_space **out);
/* Per-item lambdas + left-to-right norms computed by another rank (the one that owned the rows when the space was built):
 * the multi-GPU regrouping (api.py build_sharded, item_shards < world) all-gathers them with the rows.  Host or device. */
int asp_space_import_lambdas(asp_space *s, const double *lambdas, const double *norms);

/* K1 (API orientation): per-segment partial Gram X_s^T X_s of the owned segments, FP64 DMMA fed
 * by TMA.  out_dev: DEVICE buffer [ASP_GRAM_SEGMENTS][f][f] f64; only the owned segments'
 * blocks are written (the others are left untouched).  [exchange]: all-gather the blocks. */
int asp_space_gram_partials(asp_space *s, double *out_dev);

/* K1 selection + K2: graph from the complete set of segment partials.
 * gram_segments_dev: DEVICE [ASP_GRAM_SEGMENTS][f][f].  Distances d = 1 - max(0, cos) between
 * feature columns, eps-radius, k smallest by (d, index), weights, W = max(W, W^T), L = D - W as
 * CSR (GRAPH_VARIABLES.md:3,7-10).  Decisions (d <= eps, k-th neighbour) are guaranteed equal to
 * the ones made on left-to-right f64 sums: any comparison inside the rounding band of the DMMA
 * Gram is listed in need_pairs (pairs a<b, 2 int32 each, at most need_cap pairs) and the call
 * returns ASP_NEED_EXACT; resolve them with asp_space_exact_pairs and call again.
 * exact_pairs/exact_sums (n_exact pairs, 3 sums each: <a,b>, <a,a>, <b,b>) may be NULL/0. */
int asp_graph_from_gram(asp_ctx *ctx, const double *gram_segments_dev, int32_t f, int64_t n_total,
                        const asp_graph_params *gp, const asp_switches *sw,
                        const int32_t *exact_pairs, const double *exact_sums, int64_t n_exact,
                        int32_t *need_pairs, int64_t need_cap, int64_t *n_need,
                        asp_graph **out_graph);

/* Continue the left-to-right sums of the listed column pairs over this shard's rows:
 * sums[3*i+0] += sum_r x[r][a]*x[r][b], [1] += x[r][a]^2, [2] += x[r][b]^2 (r ascending, product
 * rounded then added).  [exchange]: rank r+1 continues from rank r's sums.  HOST arrays. */
int asp_space_exact_pairs(asp_space *s, const int32_t *pairs, int64_t n_pairs, double *sums);

/* K3: per-item taumode lambda (Rayleigh quotient on the feature Laplacian, median tau, bounded
 * transform: TAUMODE.md:18-19,24-25) for the shard's rows.  Replaces the lambda computation inside
 * ArrowSpaceBuilder::build (read back by lambdas(), src/lib.rs:122-124). */
int asp_space_compute_lambdas(asp_space *s, const asp_graph *g);

/* ---- accessors (src/lib.rs:40-61, 78-124) -------------------------------------------------- */
int asp_space_dims(const asp_space *s, int64_t *n_local, int32_t *f, int64_t *row0, int64_t *n_total);
int asp_space_lambdas(const asp_space *s, double *out /* n_local, host or device */);
int asp_space_norms(const asp_space *s, double *out /* n_local */);
int asp_space_get_item(const asp_space *s, int64_t local_idx, double *out_features /* f */, double *out_lambda);
int asp_space_items(const asp_space *s, double *out /* n_local x f row-major, host or device: the stored rows (persistence) */);
int asp_graph_info(const asp_graph *g, int64_t *nnodes, int64_t *nnz, asp_graph_params *gp);
int asp_graph_csr(const asp_graph *g, int64_t *indptr /* nnodes+1 */, int32_t *indices /* nnz */, double *data /* nnz */);

/* ---- persistence (SURVEY.md 8(f)-4; no reference counterpart: the pyo3 objects cannot be pickled) ------------------
 * A graph handle from a stored Laplacian (the arrays asp_graph_csr exported; host or device).  feature_graph != 0 also
 * prepares the lambda pass, so the handle serves asp_query_lambda / asp_search_batch like the graph it was saved from.
 * Together with asp_space_create + asp_space_import_lambdas this restores a built (aspace, gl) pair without rebuilding. */
int asp_graph_from_csr(asp_ctx *ctx, int64_t nnodes, int64_t nnz, const int64_t *indptr, const int32_t *indices, const double *data,
                       const asp_graph_params *gp, const asp_switches *sw, int feature_graph, asp_graph **out_graph);
int asp_graph_switches(const asp_graph *g, asp_switches *sw);

/* ---- search -------------------------------------------------------------------------------- */

/* lambda of nq query vectors (nq x f).  Replaces ArrowSpace::prepare_query_item (src/lib.rs:154).
 * Any of out_energy / out_tau / out_lambda may be NULL. */
int asp_query_lambda(asp_ctx *ctx, const asp_graph *g, const asp_switches *sw, const double *queries,
                     int64_t nq, double *out_energy, double *out_tau, double *out_lambda);

/* K4: batched lambda-aware search of nq queries against this shard.  Replaces prepare_query_item +
 * search_lambda_aware(&query, gl.graph_params.topk, tau) (src/lib.rs:154-173), batched.
 * score_i = tau*cos(q,x_i) + (1-tau)/(1+|lambda_q-lambda_i|)   (TAUMODE.md:33)
 * Returns per query min(topk, n_local) hits, best first, ties by smaller index, GLOBAL row indices;
 * rows are padded to topk with index -1 / score NaN.  Scores of the returned hits are evaluated
 * in the reference order (left-to-right f64 dot); the candidate set is proven complete against the
 * rounding band of the tensor-core pass, otherwise the query is re-scanned exactly.
 * Stage 1 runs on tcgen05 (fp16 operands: exact rank-1 mean-direction term + one or two fp16 terms of the residuals)
 * for topk <= 31 when nq >= 256 or the shard has >= 131072 items -- which includes the reference's ONE query per call:
 * the candidate pass then streams the fp16 operands instead of the f64 rows -- and on FP64 DMMA / the HBM-bound GEMV
 * kernel (nq <= 8) otherwise; env ASP_SEARCH_STAGE1=fp64|tc forces one.  The answers are bit-identical whichever
 * stage 1 produced the candidates.  topk >= 32 is answered by the batched exact scan of every query (reference-order score of
 * every item; ~3300 queries/s at 1M x 384: the completeness test needs one kept candidate beyond the k-th and the kernels keep 32).
 * asp_search_batch_k with k = 32 .. 64 keeps such lists on the tensor cores.
 * queries / outputs may be host or device memory.  Host batches of >= 32768 queries are processed in two pieces so that
 * the PCIe copies run under the kernels (env ASP_NO_PIPELINE=1: single shot); the result is the same either way.
 * One caller per ctx at a time (the reference holds the GIL for the whole call, src/lib.rs:132).
 * Fails with ASP_ERR_LAMBDA_ZERO if some lambda_q == 0.0 (src/lib.rs:156-159).
 * out_lambda_q (nq) may be NULL.  [exchange]: all-gather (idx, score) and asp_topk_merge. */
int asp_search_batch(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq,
                     double tau, int64_t *out_idx, double *out_score, double *out_lambda_q);

/* Filtered search: asp_search_batch over the items whose bit is set in allowed_bits only -- per query the best topk ALLOWED
 * items by (score desc, index asc), the oracle's scores bit for bit, rows padded with -1 / NaN when fewer items are allowed.
 * allowed_bits: a packed mask over this space's LOCAL rows, ceil(n_local / 8) bytes, LSB-first (bit i % 8 of byte i / 8 =
 * local row i; numpy.packbits(mask, bitorder="little")), host or device memory; NULL = every row, which is asp_search_batch
 * itself.  The mask is the same for every query of the call and changes neither lambda_q nor the lambda_q != 0 assertion.
 * A row shard passes the slice of the global mask for its own rows [row0, row0 + n_local); the per-shard lists merge with
 * asp_topk_merge as they are. */
int asp_search_batch_filtered(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                              int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits);

/* Search with a per-call k: asp_search_batch_filtered returning k hits per query instead of gl.graph_params.topk, so a
 * different k needs no rebuild (under topk_prunes a rebuild would also change the graph and every lambda).  out_idx /
 * out_score are [nq][k], padded with -1 / NaN when fewer than k items exist or are allowed; allowed_bits NULL = every row.
 * 1 <= k <= 1024 (k < 1: ASP_ERR_ARG; k > 1024, the exact scan's list length: ASP_ERR_UNSUPPORTED).  Same answers, bit for
 * bit, as asp_search_batch on a graph of topk = k.  Route: k <= 31 as asp_search_batch; 32 <= k <= 64 stays on the tcgen05
 * candidate pass (64-entry running lists) with a wide stage 2 of one CTA per query that keeps every survivor of the
 * cut (csrc/large_k.cuh), on the tensor-core pass's conditions (0.001 < tau <= 1, <= 6144 features, nq >= 256 or >= 131072
 * items); k > 64 (a 128-entry list spills registers in stage 1) and everything else take the batched exact scan.  The graph-topk entry points keep their routes: a graph
 * topk >= 32 there still takes the exact scan; moving them onto the wide route is a separate change that needs its own
 * B200 measurements. */
int asp_search_batch_k(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t k,
                       int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits);

/* Tau sweep: the same queries at ntau >= 1 taus (host array taus, finite, duplicates allowed) in one call.  out_idx /
 * out_score are [ntau][nq][k]; rows t are, bit for bit, asp_search_batch_k(s, g, queries, nq, taus[t], k, ...) with the same
 * allowed_bits.  k as in asp_search_batch_k (the Python layer passes the graph topk for k=None).  lambda_q is computed once
 * (out_lambda_q [nq], may be NULL); the lambda_q == 0 and zero-vector failures are those of asp_search_batch.  Route: the
 * taus that take the tcgen05 candidate pass in asp_search_batch_k with k <= 16 share ONE candidate pass per group of at most
 * 3 taus (two or more per group; tc_gemm_kernel holds every tau's running list in registers, and a fourth spills), then each
 * runs its own stage 2 and slow-query remedies; every other tau, and a lone qualifying one, takes asp_search_batch_k's route.
 * queries / outputs may be host or device memory.  Single-GPU spaces: a sharded layout loops over asp_search_batch_k in the
 * Python layer.  asp_ctx_stat keys: sweep_fused_taus, sweep_stage1_passes (shared candidate passes), search_slow_queries
 * (summed over the taus), sweep_slow_queries_<t>, sweep_stage1_ms / sweep_stage2_ms / sweep_emitted_per_query (shared passes). */
int asp_search_batch_taus(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, const double *taus,
                          int64_t ntau, int64_t k, int64_t *out_idx, double *out_score, double *out_lambda_q,
                          const uint8_t *allowed_bits);

/* Hybrid search, batched (SURVEY.md 8(f)-2).  Replaces prepare_query_item + search_lambda_aware_hybrid(&query,
 * gl.graph_params.topk, tau) of ArrowSpace.search_hybrid (src/lib.rs:182-219).  The crate function's body is not in the
 * reference and nothing there documents or tests it, so this is a restatement (PARITY UNPINNED against the crate; GPU ==
 * oracle: indices identical; scores the oracle's bit for bit on the shortlist route, as asp_search_batch's when pool >= n)
 * of the two-stage reading of "hybrid", the shortlist length an argument:
 *   H1 lambda_q as in asp_search_batch, WITHOUT the lambda_q != 0 assertion (search_hybrid has none);
 *   H2 shortlist = the `pool` items of largest cosine, ties -> smaller index (pool <= 0: min(2 * topk, 31); raised to topk, cut to n):
 *      asp_search_batch's own path at tau = 1 with topk = pool (tcgen05 candidates + exact stage 2 for pool <= 31, the
 *      batched exact scan beyond -- the default keeps every topk <= 31, the reference scripts' 15 and 25 included, on the
 *      tensor cores);
 *   H3 score_i = tau*cos_i + (1-tau)/(1+|lambda_q-lambda_i|) over the shortlist, evaluated in the reference order; the best
 *      min(topk, n) by (score desc, index asc).
 * pool >= n: no shortlist, i.e. asp_search_batch without the assertion; otherwise pool <= 1024 (what the exact scan keeps).
 * Output layout as asp_search_batch.  Needs every item on this GPU (world-1 space or a replicated item shard);
 * ASP_ERR_UNSUPPORTED on a row shard: a row-sharded space answers with asp_search_hybrid_shard + asp_hybrid_merge. */
int asp_search_hybrid_batch(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                            int64_t pool, int64_t *out_idx, double *out_score, double *out_lambda_q);

/* Filtered hybrid search: H2's shortlist is the m ALLOWED items of largest cosine (ties -> smaller index), with m still
 * asp_hybrid_pool(n, topk, pool) of the whole item count; H3 re-ranks it.  allowed_bits as in asp_search_batch_filtered. */
int asp_search_hybrid_batch_filtered(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                                     int64_t pool, int64_t *out_idx, double *out_score, double *out_lambda_q,
                                     const uint8_t *allowed_bits);

/* Hybrid search with a per-call k: k replaces gl.graph_params.topk in H2 and H3 (pool <= 0: asp_hybrid_pool(n, k, 0) =
 * min(2k, 31) raised to k), outputs [nq][k].  k as in asp_search_batch_k; shortlists of up to 64 stay on the tensor-core
 * route.  allowed_bits NULL = every row. */
int asp_search_hybrid_batch_k(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                              int64_t k, int64_t *out_idx, double *out_score, double *out_lambda_q, const uint8_t *allowed_bits);

/* The shortlist length m of H2 for n_total items: pool (<= 0: min(2 * topk, 31)), raised to topk, cut to n_total.
 * m == n_total (with n_total > 0) means no shortlist: the whole set. */
int64_t asp_hybrid_pool(int64_t n_total, int64_t topk, int64_t pool);

/* Hybrid search on a row-sharded space, bit for bit the one-GPU asp_search_hybrid_batch over all n_total items.  Every
 * rank holding an item shard calls asp_search_hybrid_shard with the same queries; [exchange]: all-gather the outputs;
 * then merge.  With m = asp_hybrid_pool(n_total, topk, pool):
 *   m < n_total   out_idx / out_cos / out_score are [nq][m]: the shard's own top-m by (cosine desc, index asc) -- the
 *                 search at tau = 1 with topk = m -- as GLOBAL indices, their cosines and their H3 scores at tau; lists
 *                 padded with -1 / NaN.  m <= 1024, else ASP_ERR_UNSUPPORTED.  asp_hybrid_merge of the parts' lists
 *                 ([parts][nq][m], shards in any order) takes the global top-m by cosine, which lies in the union of the
 *                 shards' top-m lists, and returns its best topk by (score desc, index asc).
 *   m == n_total  no shortlist: out_idx / out_score are [nq][topk], the shard's best topk by the lambda-aware score at tau
 *                 (asp_search_batch without the assertion); out_cos is not used; merge with asp_topk_merge.
 * H1 as asp_search_hybrid_batch (no lambda_q != 0 assertion; every rank gets the same lambda_q).  Host or device
 * pointers.  asp_hybrid_merge output layout as asp_search_batch. */
int asp_search_hybrid_shard(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                            int64_t pool, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q);
/* The same over this shard's allowed rows (allowed_bits: the shard's slice of the global mask, as in
 * asp_search_batch_filtered).  asp_hybrid_merge / asp_topk_merge of the filtered lists give the filtered one-GPU answer. */
int asp_search_hybrid_shard_filtered(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                                     int64_t pool, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q,
                                     const uint8_t *allowed_bits);
/* The same with a per-call k in place of gl.graph_params.topk (m = asp_hybrid_pool(n_total, k, pool); [nq][k] lists when
 * m == n_total), k as in asp_search_batch_k; merge with asp_hybrid_merge / asp_topk_merge at list width k. */
int asp_search_hybrid_shard_k(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau, int64_t pool,
                              int64_t k, int64_t *out_idx, double *out_cos, double *out_score, double *out_lambda_q,
                              const uint8_t *allowed_bits);
int asp_hybrid_merge(asp_ctx *ctx, const int64_t *idx, const double *cos, const double *score, int parts, int64_t nq,
                     int64_t m, int64_t topk, int64_t *out_idx, double *out_score);

/* Range search (no reference counterpart): per query EVERY item with score >= min_score, ordered by (score desc, index asc),
 * GLOBAL indices, the oracle-order scores bit for bit (score and lambda_q as in asp_search_batch, including the
 * lambda_q != 0 assertion and the zero-vector check).  min_score is inclusive and compared in f64 against the reference-order
 * value; -inf returns every item, > 1 returns empty rows, NaN is ASP_ERR_ARG.  allowed_bits as in asp_search_batch_filtered
 * (NULL = all).  out_counts[nq] (host or device) receives the per-query hit counts; the hits stay in device memory owned by
 * *out until asp_range_result_fetch copies them out (sum(counts) entries, query-major; host or device) and
 * asp_range_result_free releases them.  max_hits > 0: when the running total of the call exceeds it the call fails with
 * ASP_ERR_LIMIT, naming the total and the query at which it was crossed; batches are processed in sub-batches of
 * asp_range_sub_batch() queries and the cap is checked on each sub-batch's counts before its hits get device memory.
 * Candidates: the tcgen05 pass of the search with topk = 0 and min_score (clamped to [-2, 2]) as its emission floor, for
 * 0.001 < tau <= 1 and <= 6144 features; queries whose emission buffers overflow, and every query outside those bounds, take
 * the exact range scan (env ASP_RANGE_STAGE1=scan forces it: a test knob, the same bits).  [exchange]: a row shard passes
 * its slice of the mask; the per-shard results merge with asp_range_merge. */
int  asp_search_range_batch(const asp_space *s, const asp_graph *g, const double *queries, int64_t nq, double tau,
                            double min_score, const uint8_t *allowed_bits, int64_t max_hits, int64_t *out_counts,
                            double *out_lambda_q, asp_range_result **out);
int  asp_range_result_fetch(const asp_range_result *r, int64_t *out_idx, double *out_score);
void asp_range_result_free(asp_range_result *r);
int64_t asp_range_sub_batch(void);
/* Merge of per-shard range results over the same nq queries into the one-GPU order: counts [parts][nq] and the concatenated
 * parts' hits (each part query-major, each query's hits sorted) -> sum(counts) hits query-major.  Shards must be contiguous
 * global row ranges (then ties resolve as on one GPU, whatever the number or order of the shards).  Host or device pointers. */
int  asp_range_merge(asp_ctx *ctx, int parts, int64_t nq, const int64_t *counts, const int64_t *idx, const double *score,
                     int64_t *out_idx, double *out_score);

/* Test hook of the tcgen05 candidate pass: the approximate cosines (unit-scaled operands, bf16 two-term split,
 * f32 accumulation in TMEM) of nq queries against every item of the shard, out[nq][n_local] f32 (host or device). */
int asp_debug_tc_dots(const asp_space *s, const double *queries, int64_t nq, float *out);

/* K5: merge `parts` candidate lists per query ([parts][nq][topk], as produced by
 * asp_search_batch on each shard) into the global top-k by (score desc, index asc). */
int asp_topk_merge(asp_ctx *ctx, const int64_t *idx, const double *score, int parts, int64_t nq,
                   int64_t topk, int64_t *out_idx, double *out_score);

/* K5 over NVLink peer memory (no NCCL call in the exchange): every rank stores its [nq][topk] lists into slot [rank] of
 * EVERY rank's exchange buffer (P2P stores), raises a flag there, and merges when all flags show `epoch`.
 * peer_bases[r] = device address, valid in THIS process, of rank r's exchange buffer (asp_peer_exchange_bytes(world,
 * cap, topk) bytes, zero-filled before the first call; mapping it is the caller's plumbing -- api.py uses
 * torch.distributed._symmetric_memory).  `epoch` = 1, 2, 3 ... per call on that buffer, the same on every rank;
 * nq <= cap.  idx / score / outputs are device memory.  A rank that never shows up is reported (ASP_ERR_CUDA) after
 * a bounded wait.  No reference counterpart.  Checked on 2 GPUs (bitwise equal to the NCCL route); not yet run on 4 / 8
 * GPUs nor timed: opt-in through ASP_PEER_MERGE=1 in the Python layer. */
#define ASP_PEER_MAX_WORLD 8
size_t asp_peer_exchange_bytes(int world, int64_t cap, int64_t topk);
int asp_peer_merge(asp_ctx *ctx, int world, int rank, const uint64_t *peer_bases, int64_t cap, int64_t epoch,
                   const int64_t *idx_dev, const double *score_dev, int64_t nq, int64_t topk, int64_t *out_idx_dev,
                   double *out_score_dev);

/* ---- item graph (nodes = items; the graph-build workload of configs C4/C5) ------------------ */

/* K1 (item orientation) + K2 for the shard's rows against `all_items` (n_total x f, host or
 * device; NULL = the shard itself, single GPU): eps / k-NN graph on the distance of sw->distance (rectified cosine by
 * default; l2 / l2sq: the oracle's Gram form (<a,a> + <b,b>) - 2<a,b> from left-to-right sums, clamped at 0),
 * weights, symmetrised Laplacian CSR over n_total nodes.  Single GPU; candidates on the tensor cores (tcgen05) for
 * n >= 8192, k <= 30 and <= 6144 features; below that FP64 DMMA (cosine) or the exact scan of every row (l2 / l2sq);
 * same exact stage 2 and answers.  l2 / l2sq: k > 30, more than 6144 features at n >= 8192, or norms above 1e18 on the
 * tensor-core route fail with ASP_ERR_UNSUPPORTED. */
int asp_item_graph(asp_space *s, const asp_graph_params *gp, const asp_switches *sw, asp_graph **out_graph);

/* Multi-GPU item graph (BASELINE.json configs C4/C5: "items sharded over 8 GPUs, NCCL halo exchange"; any distance): every rank
 * holds ALL items (the halo rows arrive by all-gather) in a world-1 space and resolves the eps / k-NN lists of ITS rows
 * [row_begin, row_end) on the tensor cores; the lists are all-gathered and the Laplacian is assembled from them.
 *   asp_item_knn_rows: out_idx / out_dist [rows][*out_kk] (only the first out_cnt[r] entries of a row are valid,
 *                      ascending (distance, index)), out_cnt [rows]; host or device pointers.  Replaces the per-row scan
 *                      of the crate's graph construction (src/lib.rs:289; GRAPH_VARIABLES.md:7-8).
 *   asp_graph_from_knn: K2 from complete lists of m nodes (host or device pointers). */
int asp_item_knn_rows(asp_space *s, const asp_graph_params *gp, const asp_switches *sw, int64_t row_begin, int64_t row_end,
                      int32_t *out_idx, double *out_dist, int32_t *out_cnt, int32_t *out_kk);
int asp_graph_from_knn(asp_ctx *ctx, int64_t m, int32_t kk, const int32_t *idx, const double *dist, const int32_t *cnt,
                       const asp_graph_params *gp, const asp_switches *sw, asp_graph **out_graph);

/* ---- pre-graph reduction (SURVEY.md 8(f)-1) --------------------------------------------------------------------------
 * What the crate runs inside ArrowSpaceBuilder::build before graph construction (with_dims_reduction / with_seed,
 * src/lib.rs:282-283; log evidence tests/output/1760705545_v0_16/suggested_eps.md:3-11: "Simple random sampler with keep
 * rate 60.0%", "Two-NN mean ratio: 1.3560, estimated ID: 3", "Testing K in range [178, 179]" for N = 313841): the items
 * are sampled, clustered, and the graph is built on the CENTROID matrix (n_clusters x f) instead of the item matrix;
 * lambdas are still computed for every item.  The crate's arithmetic and RNG stream are not in the reference, so this is a
 * deterministic restatement (PARITY UNPINNED against the crate; GPU == oracle bit for bit on the centroids):
 *   R1 sample   row i is kept iff u(seed, i) < sample_rate, u = (splitmix64(seed + (i+1)*0x9E3779B97F4A7C15) >> 11) * 2^-53;
 *               sample_rate >= 1 keeps every row.  S = kept rows, ascending.
 *   R2 two-NN   probes = S[floor(j*|S|/P)], P = min(probes, |S|); r1 <= r2 = the two smallest Euclidean distances from a
 *               probe to the other rows of S (squared distances summed left to right, ties by position); probes with
 *               r1 == 0 are skipped; mean ratio = mean(r2/r1) in probe order; intrinsic dimension = trunc(m/(m-1))
 *               clamped to [1, f] (the mean of a Pareto(d) variable is d/(d-1); 1.3560 -> 3 as in the log).
 *   R3 K        n_clusters if > 0, else ceil(sqrt(n_total/10)) (the one published data point: 313841 -> 178), at most |S|.
 *   R4 k-means  centroid j starts at row S[floor(j*|S|/K)]; Lloyd iterations: assign every row of S to the nearest centroid
 *               (squared Euclidean, left to right, ties -> smaller centroid), stop when no assignment changed, else
 *               centroid = (sum of its rows in ascending row order) / count (an empty cluster keeps its centroid); at most
 *               max_iters updates.
 *   R5 graph    the usual recipe (asp_graph_params / asp_switches) with nodes = the f columns of the centroid matrix.
 *   R6 lambdas  per item, from that Laplacian.
 * Not restated: the crate's optional JL projection (with_dims_reduction(true, Some(eps))) -- searched vectors stay raw. */
typedef struct {
    double   sample_rate;   /* default 0.6 */
    uint64_t seed;          /* default 42 (src/lib.rs:283) */
    int32_t  n_clusters;    /* 0 = rule R3 */
    int32_t  max_iters;     /* default 10 */
    int32_t  probes;        /* default 2048; 0 = skip the two-NN estimate */
    int32_t  reserved;
} asp_reduction;
typedef struct {
    int64_t n_sampled;
    int64_t n_probes;          /* probes that entered the mean (r1 > 0) */
    double  two_nn_mean_ratio; /* NaN when skipped */
    int32_t intrinsic_dim;     /* 0 when skipped */
    int32_t n_clusters;
    int32_t iters;             /* centroid updates done */
    int32_t converged;         /* 1: an assignment pass changed nothing */
} asp_reduction_info;
void asp_default_reduction(asp_reduction *red);
/* R1 on the host: kept rows of [row0, row0 + n_local) as LOCAL indices, ascending; out_rows holds n_local entries. */
int asp_reduction_sample(const asp_reduction *red, int64_t row0, int64_t n_local, int32_t *out_rows, int64_t *out_count);
/* R1-R4 on a resident space (world 1): a new space whose rows are the centroids (read them with asp_space_items).
 * n_total_for_k = the N of rule R3 (0: the space's own row count). */
int asp_space_reduce(asp_space *s, const asp_reduction *red, int64_t n_total_for_k, asp_reduction_info *info,
                     asp_space **out_centroids);
/* R5: the feature graph of the rows of a space (what asp_build does between upload and lambdas). */
int asp_space_feature_graph(asp_space *s, const asp_graph_params *gp, const asp_switches *sw, asp_graph **out_graph);
/* R1-R6 in one call; out_centroids may be NULL. */
int asp_build_reduced(asp_ctx *ctx, const double *items, int64_t n, int32_t f, const asp_graph_params *gp,
                      const asp_switches *sw, const asp_reduction *red, asp_space **out_space, asp_graph **out_graph,
                      asp_reduction_info *info, asp_space **out_centroids);

/* ---- teardown / stats ---------------------------------------------------------------------- */
void asp_free_space(asp_space *s);
void asp_free_graph(asp_graph *g);

/* Last-call statistics (diagnostics; -1 = not applicable).  keys: "gram_ms", "graph_ms",
 * "lambda_ms", "search_gemm_ms", "search_rescore_ms", "search_slow_queries", "need_exact_pairs". */
double asp_ctx_stat(const asp_ctx *ctx, const char *key);

#ifdef __cplusplus
}
#endif
#endif
