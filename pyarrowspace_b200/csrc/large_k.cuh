// large_k.cuh -- the selection logic of the wide stage 2 (tc_rescore_wide_kernel, csrc/search_tc.cu): a search with a per-call
// k of 32 .. 64 on the tensor-core candidate pass (asp_search_batch_k and the hybrid _k entry points).
//
// One CTA per query.  Stage 1 left the query's emitted candidates (approximate f32 scores, distinct items) in nstreams
// lists.  The kernel then
//   (1) CUT      the kk-th largest approximate score over ALL emitted candidates (kk = min(k, n_local)), found by a radix
//                select of its order-preserving 32-bit key (four 8-bit digits, most significant first): a function of the
//                SET of candidates, so the result does not depend on the schedule or on the number of item chunks;
//   (2) COLLECT  every candidate at or above cut - 2 DELTA (the row's band) into shared memory, up to SURV_CAP of them;
//   (3) FAST     re-scores each survivor in f64 (warp-cooperative dot, error <= EPS), sorts them by (fast desc, index asc);
//   (4) BAND     keeps the prefix whose fast score is >= the kk-th best fast score - 2 EPS, re-scores it in the reference
//                order (the oracle's expression), sorts it by (score desc, index asc) and emits the first kk, padded to k.
// The completeness argument of search_tc.cu holds unchanged: the true top-kk all pass the cut and the band.
// A query takes the exact scan (slow list) when an emission list overflowed, when more than SURV_CAP candidates survive
// the cut, or when fewer than kk were emitted (a filter with fewer than k allowed items, or k > n).
//
// Everything that decides the result is a plain function here, so that tests/host_emul/large_k_host.cpp can compile this
// header with g++ and walk the phases thread by thread on the CPU (tests/test_large_k_cpu.py).
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#define ASP_RANGE_KEYS_ONLY
#include "range.cuh"
#undef ASP_RANGE_KEYS_ONLY

#if defined(__CUDACC__)
#define ASP_LK_FN __host__ __device__ __forceinline__
#else
#define ASP_LK_FN static inline
#endif

namespace asp_lk {

constexpr int SURV_CAP = 4096;       // survivors of the cut kept per query (shared memory); more take the exact scan
constexpr int KMAX = 64;             // widest k on the tensor-core route: stage 1 keeps ceil(k / 4) <= 16 scores per thread (a
                                     // 128-entry instantiation, 32 per thread, spills 56 bytes under the kernel's register cap)
constexpr int KMIN = 32;             // narrower k keep the 32-per-warp stage 2 (tc_rescore_kernel)

enum Route { ROUTE_OK = 0, ROUTE_SLOW = 1 };

// order-preserving key of an f32 score: key(a) < key(b) iff a < b (the two zeros tie)
ASP_LK_FN uint32_t f32_key(float f)
{
    if (f == 0.0f) f = 0.0f;
    uint32_t b;
#if defined(__CUDA_ARCH__)
    b = __float_as_uint(f);
#else
    memcpy(&b, &f, sizeof(b));
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

ASP_LK_FN float key_f32(uint32_t k)
{
    const uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(b);
#else
    float f;
    memcpy(&f, &b, sizeof(f));
    return f;
#endif
}

// radix select, pass 0..3: the digit of a key, and whether the key's digits above this pass equal the prefix found so far
ASP_LK_FN int digit(uint32_t key, int pass) { return (int)((key >> (24 - 8 * pass)) & 255u); }
ASP_LK_FN bool prefix_match(uint32_t key, uint32_t prefix, int pass)
{
    return pass == 0 || (key >> (32 - 8 * pass)) == (prefix >> (32 - 8 * pass));
}

// one thread, after the histogram of a pass: the digit that holds the k_rem-th largest key among the matching ones, walked
// from the largest digit down; k_rem becomes its rank inside that digit.  The caller guarantees k_rem <= the matching count.
ASP_LK_FN int select_digit(const int *hist, int *k_rem)
{
    int d = 255;
    for (; d > 0; --d) {
        if (*k_rem <= hist[d]) break;
        *k_rem -= hist[d];
    }
    return d;
}

// cut - 2 DELTA: the survivors' threshold from the kk-th largest approximate score (f32, as in tc_rescore_kernel)
ASP_LK_FN float survivor_cutoff(uint32_t kth_key, float delta) { return key_f32(kth_key) - 2.0f * delta; }

// the query's route once the survivors are known
ASP_LK_FN int route(bool overflow, int64_t emitted, int64_t n_surv, int kk)
{
    if (overflow || emitted < kk || n_surv > SURV_CAP || n_surv < kk) return ROUTE_SLOW;
    return ROUTE_OK;
}

ASP_LK_FN int next_pow2(int n)
{
    int p = 1;
    while (p < n) p <<= 1;
    return p;
}

// sort keys: (desc_key(score), index) ascending = (score desc, index asc); padding (~0, INT32_MAX) sorts last
ASP_LK_FN bool key_before(uint64_t ka, int32_t ia, uint64_t kb, int32_t ib) { return ka < kb || (ka == kb && ia < ib); }

// bitonic sort of n (a power of two) pairs, ascending: compare-exchange t (0 <= t < n / 2) of step (size, stride);
// every t of a step touches its own two slots
ASP_LK_FN void bitonic_cx(uint64_t *key, int32_t *ix, int t, int size, int stride)
{
    const int i = 2 * stride * (t / stride) + (t % stride), j = i + stride;
    const bool up = (i & size) == 0;
    const bool swap = up ? key_before(key[j], ix[j], key[i], ix[i]) : key_before(key[i], ix[i], key[j], ix[j]);
    if (swap) {
        const uint64_t k = key[i]; key[i] = key[j]; key[j] = k;
        const int32_t v = ix[i]; ix[i] = ix[j]; ix[j] = v;
    }
}

// after the fast sort: slot i (< n_surv) is in the band of the kk-th best fast score
ASP_LK_FN bool in_band(const uint64_t *key, int i, int kk, double eps)
{
    const double kth = asp_range::key_score(key[kk - 1]);
    return asp_range::key_score(key[i]) >= kth - 2.0 * eps;
}

// output slot j (< k) of a finished query: the band sorted by (exact score desc, index asc), first kk, padded with -1 / NaN
ASP_LK_FN void emit_slot(int j, int kk, const uint64_t *key, const int32_t *ix, int64_t row0, int64_t *out_idx, double *out_score)
{
    const bool ok = j < kk;
    out_idx[j] = ok ? row0 + ix[j] : -1;
    out_score[j] = ok ? asp_range::key_score(key[j]) : NAN;
}

}  // namespace asp_lk
