// peer.cu -- K5 over NVLink peer memory: the exchange step of the sharded search without NCCL calls.
//
// The sharded search is [per-shard exact top-k] -> [all ranks see all lists] -> [merge by (score desc, index asc)].
// With NCCL that is two all_gather_into_tensor calls on torch's stream plus two host-side stream hand-offs around the
// merge kernel.  Here every rank owns one EXCHANGE BUFFER that all ranks of the box have mapped (the mapping is plumbing:
// torch.distributed._symmetric_memory, see pyarrowspace_b200/api.py); a rank
//   1. stores its [nq][topk] (index, score) lists straight into slot [own rank] of EVERY rank's buffer (P2P stores through
//      NVSwitch; 10.5 MB per peer for 64k x top-10), fences system-wide and raises its flag on every rank
//      (st.release.sys), and
//   2. merges as soon as the flags of all ranks show the current epoch (ld.acquire.sys on its own memory).
// No rank waits on another before it has published its own lists, so the wait cannot deadlock; it is bounded anyway
// (60 s of clock64 by default) and reports a timeout instead of hanging the GPU; after a timeout the Python layer drops the
// exchange buffer, so the next call re-rendezvouses on zeroed flags behind a barrier.
//
// Buffer layout (the same on every rank; `cap` = queries the buffer was sized for):
//   [0, 4096)                                   uint32 flag[2 parities][ASP_PEER_MAX_WORLD]
//   4096 + (parity * world + src) * slot_bytes  slot of rank `src`: int64 idx[cap * topk], then f64 score[cap * topk]
// Two parities: rank A may start call e+1 while a slower rank still merges call e.  A rank raises flag e+1 only after its
// merge of e, and nobody finishes e+1 before all flags e+1 are up, so when A overwrites the parity of e (call e+2) every
// rank is done reading it.
//
// STATUS (end of round 1): correct on 2 GPUs -- `CHECK_PEER=1 QUICK=1 torchrun --nproc-per-node 2 tools/mgpu_check.py` gives
// results bitwise equal to the NCCL route over three consecutive calls (both parities, slot reuse;
// profiles/mgpu_check_peer_merge_2gpu_r01.log).  Not yet run on 4 / 8 GPUs and not yet timed, so it stays OFF unless
// ASP_PEER_MERGE=1 (api.py).
#include "common.cuh"

#include <algorithm>
#include <math.h>
#include <stdlib.h>

namespace {

constexpr int PEER_MAX_WORLD = ASP_PEER_MAX_WORLD;
constexpr size_t PEER_HEADER = 4096;

struct PeerPtrs { unsigned char *base[PEER_MAX_WORLD]; };

__device__ __forceinline__ void st_release_sys_u32(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// the exchange buffer is written by REMOTE GPUs while this kernel runs: no const / __restrict__ on it (the compiler could
// emit ld.global.nc, undefined for data modified during the kernel's lifetime) and system-scope relaxed loads after the acquire
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const void *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__host__ __device__ __forceinline__ size_t peer_slot_bytes(int64_t cap, int64_t topk) { return (size_t)cap * topk * 16; }

// step 1: publish this rank's lists in every rank's buffer, then raise the flag everywhere (last block to finish)
__global__ void __launch_bounds__(256)
peer_scatter_kernel(PeerPtrs pp, int world, int rank, int parity, uint32_t epoch, const int64_t *__restrict__ idx,
                    const double *__restrict__ score, int64_t n_elem, int64_t cap, int64_t topk, unsigned int *done_counter)
{
    const size_t slot = peer_slot_bytes(cap, topk);
    const size_t off = PEER_HEADER + ((size_t)parity * world + rank) * slot;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_elem; e += stride) {
        const int64_t vi = idx[e];
        const double vs = score[e];
        for (int k = 0; k < world; ++k) {
            const int r = (rank + 1 + k) % world;                       // every rank starts with a different peer
            int64_t *di = reinterpret_cast<int64_t *>(pp.base[r] + off);
            double *ds = reinterpret_cast<double *>(di + (size_t)cap * topk);
            di[e] = vi;
            ds[e] = vs;
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(done_counter, 1u);
        if (prev == gridDim.x - 1) {                                    // all blocks have fenced their stores
            *done_counter = 0u;                                         // the next call on this stream starts from zero
            __threadfence_system();
            for (int r = 0; r < world; ++r)
                st_release_sys_u32(reinterpret_cast<uint32_t *>(pp.base[r]) + parity * PEER_MAX_WORLD + rank, epoch);
        }
    }
}

struct PKey { double s; int64_t i; };
__device__ __forceinline__ bool pkey_better(const PKey &x, const PKey &y) { return (x.s > y.s) || (x.s == y.s && x.i < y.i); }

// step 2: one block per query; waits for all flags, then the same bitonic merge as topk_merge_kernel (search.cu)
__global__ void __launch_bounds__(128)
peer_merge_kernel(unsigned char *own, int world, int parity, uint32_t epoch, int64_t nq, int64_t cap,
                  int topk, int p2, long long timeout_cycles, int64_t *__restrict__ out_idx, double *__restrict__ out_score,
                  int *status)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PKey *keys = reinterpret_cast<PKey *>(smem_raw);
    __shared__ int s_ok;
    if (threadIdx.x == 0) {
        const uint32_t *flags = reinterpret_cast<const uint32_t *>(own) + parity * PEER_MAX_WORLD;
        const long long t0 = clock64();
        int ok = 1;
        for (int r = 0; r < world && ok; ++r) {
            while (ld_acquire_sys_u32(flags + r) != epoch) {
                if (clock64() - t0 > timeout_cycles || *reinterpret_cast<volatile int *>(status) != 0) { ok = 0; break; }
                __nanosleep(200);
            }
        }
        if (!ok) atomicExch(status, 1);
        s_ok = ok;
    }
    __syncthreads();
    if (!s_ok) return;
    const int64_t qi = blockIdx.x;
    const size_t slot = peer_slot_bytes(cap, topk);
    const int total = world * topk;
    for (int i = threadIdx.x; i < p2; i += blockDim.x) {
        PKey k; k.s = -INFINITY; k.i = INT64_MAX;
        if (i < total) {
            const int p = i / topk, j = i % topk;
            const int64_t *pi = reinterpret_cast<const int64_t *>(own + PEER_HEADER + ((size_t)parity * world + p) * slot);
            const double *ps = reinterpret_cast<const double *>(pi + (size_t)cap * topk);
            const int64_t id = (int64_t)ld_relaxed_sys_u64(pi + qi * topk + j);
            if (id >= 0) { k.s = __longlong_as_double((long long)ld_relaxed_sys_u64(ps + qi * topk + j)); k.i = id; }
        }
        keys[i] = k;
    }
    for (int size = 2; size <= p2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < p2 / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool first = ((lo & size) == 0);
                const PKey a = keys[lo], b = keys[hi];
                if (first ? pkey_better(b, a) : pkey_better(a, b)) { keys[lo] = b; keys[hi] = a; }
            }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < topk; i += blockDim.x) {
        const bool ok = (i < p2) && keys[i].i != INT64_MAX;
        out_idx[qi * topk + i] = ok ? keys[i].i : -1;
        out_score[qi * topk + i] = ok ? keys[i].s : NAN;
    }
}

}  // namespace

extern "C" {

size_t asp_peer_exchange_bytes(int world, int64_t cap, int64_t topk)
{
    if (world <= 0 || world > PEER_MAX_WORLD || cap <= 0 || topk <= 0) return 0;
    return PEER_HEADER + 2 * (size_t)world * peer_slot_bytes(cap, topk);
}

int asp_peer_merge(asp_ctx *ctx, int world, int rank, const uint64_t *peer_bases, int64_t cap, int64_t epoch,
                   const int64_t *idx_dev, const double *score_dev, int64_t nq, int64_t topk, int64_t *out_idx_dev,
                   double *out_score_dev)
{
    if (!ctx || !peer_bases || !idx_dev || !score_dev || !out_idx_dev || !out_score_dev)
        ASP_FAIL(ASP_ERR_ARG, "asp_peer_merge: NULL argument");
    if (world < 1 || world > PEER_MAX_WORLD || rank < 0 || rank >= world || nq < 0 || nq > cap || topk <= 0 || epoch <= 0)
        ASP_FAIL(ASP_ERR_ARG, "asp_peer_merge: bad shape (world %d, rank %d, nq %lld, cap %lld, topk %lld, epoch %lld)", world, rank,
                 (long long)nq, (long long)cap, (long long)topk, (long long)epoch);
    if (nq == 0) return ASP_OK;
    ASP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    PeerPtrs pp;
    for (int r = 0; r < PEER_MAX_WORLD; ++r) pp.base[r] = (r < world) ? reinterpret_cast<unsigned char *>(peer_bases[r]) : nullptr;
    for (int r = 0; r < world; ++r)
        if (!pp.base[r]) ASP_FAIL(ASP_ERR_ARG, "asp_peer_merge: exchange buffer of rank %d is not mapped", r);
    int p2 = 1;
    while (p2 < world * topk) p2 <<= 1;
    const size_t smem = (size_t)p2 * sizeof(PKey);
    if (smem > 200 * 1024) ASP_FAIL(ASP_ERR_UNSUPPORTED, "peer merge of %d x %lld entries does not fit in shared memory", world, (long long)topk);
    asp_scratch sc(st);
    unsigned int *scratch = nullptr;                                    // [0] block counter of the scatter, [1] status
    ASP_CHECK(sc.get(&scratch, 2));
    ASP_CUDA(cudaMemsetAsync(scratch, 0, 2 * sizeof(unsigned int), st));
    const int parity = (int)(epoch & 1);
    const uint32_t e32 = (uint32_t)epoch;
    const int64_t n_elem = nq * topk;
    const int grid = (int)std::min<int64_t>(asp_ceil_div(n_elem, 256), (int64_t)ctx->num_sms * 8);
    peer_scatter_kernel<<<grid, 256, 0, st>>>(pp, world, rank, parity, e32, idx_dev, score_dev, n_elem, cap, topk, scratch);
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    ASP_CUDA(cudaFuncSetAttribute(peer_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // a missing rank is an error, not a hang -- but ordinary rank skew (a first-call cache build, page faults, a GC pause on
    // another rank) is not an error: 60 s by default, ASP_PEER_TIMEOUT_S overrides
    double timeout_s = 60.0;
    if (const char *e = getenv("ASP_PEER_TIMEOUT_S")) { const double v = atof(e); if (v > 0.0) timeout_s = v; }
    const long long timeout_cycles = (long long)(timeout_s * 2.0e9);
    peer_merge_kernel<<<(unsigned)nq, 128, smem, st>>>(pp.base[rank], world, parity, e32, nq, cap, (int)topk, p2, timeout_cycles,
                                                       out_idx_dev, out_score_dev, reinterpret_cast<int *>(scratch + 1));
    ASP_CUDA(cudaGetLastError());
    ASP_LAUNCHED(ctx);
    int status = 0;
    ASP_CUDA(cudaMemcpyAsync(&status, scratch + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    ASP_CUDA(cudaStreamSynchronize(st));
    if (status != 0) ASP_FAIL(ASP_ERR_CUDA, "asp_peer_merge: timed out waiting for the lists of the other ranks (epoch %lld)", (long long)epoch);
    return ASP_OK;
}

}  // extern "C"
