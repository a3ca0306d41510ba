// The f32 scores and the combined raw-accumulator threshold of the tau sweep's tensor-core pass
// (pyarrowspace_b200/csrc/sweep_bound.cuh), exported for tests/test_tau_sweep_cpu.py.
// Build: g++ -O2 -ffp-contract=off -fno-fast-math -shared -fPIC.
#include "../../pyarrowspace_b200/csrc/sweep_bound.cuh"

extern "C" int sw_nt_max() { return asp_sweep::NT_MAX; }
extern "C" float sw_prox(float lq, float lam) { return asp_sweep::prox(lq, lam); }
extern "C" float sw_score(float tau, float beta, float px, float acc) { return asp_sweep::score(tau, beta, px, acc); }
extern "C" float sw_prox_bound(float lq, float tl, float th) { return asp_sweep::prox_bound(lq, tl, th); }
// the single-tau epilogue's score (search_tc.cu, tc_gemm_kernel with NT == 1) verbatim, its __fdividef written as the host's /
extern "C" float sw_single_tau_score(float tau, float beta, float lq, float lam, float a)
{
    return fmaf(beta, 1.0f / (1.0f + fabsf(lq - lam)), tau * (a * (1.0f / 16384.0f)));
}
extern "C" float sw_combined(const float *theta_emit, const float *beta, const float *inv_tau, float pb, int nt)
{
    return asp_sweep::combined_threshold(theta_emit, beta, inv_tau, pb, nt);
}
