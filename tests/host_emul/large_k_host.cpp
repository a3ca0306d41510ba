// CPU walk of the wide stage 2's selection (pyarrowspace_b200/csrc/large_k.cuh, tc_rescore_wide_kernel in search_tc.cu)
// (test infrastructure: tests/test_large_k_cpu.py).  The phases run as the kernel runs them, one CTA of 256 threads per query,
// every thread index walked between the barriers; the survivors are collected in reverse thread order (the GPU's order is
// whatever the atomics give), which the sorts must make irrelevant.  The two f64 re-scores (warp dot, reference-order dot)
// are table look-ups here: fast[q][item] and exact[q][item].
// Build: g++ -O2 -ffp-contract=off -shared -fPIC.
#include <vector>

#include "../../pyarrowspace_b200/csrc/large_k.cuh"

static const int T = 256;

static void bitonic(uint64_t *key, int32_t *ix, int n)
{
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1)
            for (int t = n / 2 - 1; t >= 0; --t) asp_lk::bitonic_cx(key, ix, t, size, stride);
}

// route[q]: 0 finished here, 1 exact scan; nsurv / nband: the counts the kernel reports
extern "C" void lk_emulate(int nq, int k, int64_t n_local, int nstreams, int capb, const int32_t *cnt, const float *esc,
                           const int32_t *eix, const float *delta, double eps, const double *fast, const double *exact,
                           int64_t row0, int64_t *out_idx, double *out_score, int32_t *route, int32_t *nsurv_out, int32_t *nband_out)
{
    std::vector<uint64_t> key(asp_lk::SURV_CAP);
    std::vector<int32_t> ix(asp_lk::SURV_CAP);
    const int kk = k < n_local ? k : (int)n_local;
    for (int q = 0; q < nq; ++q) {
        bool overflow = false;
        int64_t emitted = 0;
        for (int c = 0; c < nstreams; ++c) {
            overflow |= cnt[q * nstreams + c] > capb;
            emitted += cnt[q * nstreams + c];
        }
        nsurv_out[q] = 0; nband_out[q] = 0;
        if (overflow) { route[q] = asp_lk::ROUTE_SLOW; continue; }
        float cutoff = -INFINITY;
        if (emitted >= kk) {
            uint32_t prefix = 0;
            int krem = kk;
            for (int pass = 0; pass < 4; ++pass) {
                int hist[256] = {0};
                for (int c = 0; c < nstreams; ++c)
                    for (int t = 0; t < T; ++t)
                        for (int e = t; e < cnt[q * nstreams + c]; e += T) {
                            const uint32_t kv = asp_lk::f32_key(esc[((size_t)q * nstreams + c) * capb + e]);
                            if (asp_lk::prefix_match(kv, prefix, pass)) ++hist[asp_lk::digit(kv, pass)];
                        }
                const int d = asp_lk::select_digit(hist, &krem);
                prefix |= (uint32_t)d << (24 - 8 * pass);
            }
            cutoff = asp_lk::survivor_cutoff(prefix, delta[q]);
        }
        int nsurv = 0;
        for (int c = nstreams - 1; c >= 0; --c)
            for (int t = T - 1; t >= 0; --t)
                for (int e = t; e < cnt[q * nstreams + c]; e += T) {
                    const size_t at = ((size_t)q * nstreams + c) * capb + e;
                    if (esc[at] >= cutoff) {
                        const int pos = nsurv++;
                        if (pos < asp_lk::SURV_CAP) ix[pos] = eix[at];
                    }
                }
        nsurv_out[q] = nsurv;
        if (asp_lk::route(false, emitted, nsurv, kk) != asp_lk::ROUTE_OK) { route[q] = asp_lk::ROUTE_SLOW; continue; }
        for (int s = 0; s < nsurv; ++s) key[s] = asp_range::desc_key(fast[(size_t)q * n_local + ix[s]]);
        const int n2 = asp_lk::next_pow2(nsurv);
        for (int s = nsurv; s < n2; ++s) { key[s] = ~0ull; ix[s] = 0x7fffffff; }
        bitonic(key.data(), ix.data(), n2);
        int nb = 0;
        for (int i0 = 0; i0 < nsurv; i0 += T) {
            int cntb = 0;
            for (int t = 0; t < T; ++t) cntb += (i0 + t < nsurv && asp_lk::in_band(key.data(), i0 + t, kk, eps)) ? 1 : 0;
            nb += cntb;
            if (cntb < T) break;
        }
        nband_out[q] = nb;
        const int n3 = asp_lk::next_pow2(nb);
        for (int i = 0; i < n3; ++i) {
            if (i < nb) key[i] = asp_range::desc_key(exact[(size_t)q * n_local + ix[i]]);
            else { key[i] = ~0ull; ix[i] = 0x7fffffff; }
        }
        bitonic(key.data(), ix.data(), n3);
        for (int j = 0; j < k; ++j) asp_lk::emit_slot(j, kk, key.data(), ix.data(), row0, out_idx + (size_t)q * k, out_score + (size_t)q * k);
        route[q] = asp_lk::ROUTE_OK;
    }
}
