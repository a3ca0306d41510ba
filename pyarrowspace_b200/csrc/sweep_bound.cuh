// sweep_bound.cuh -- the f32 scores and the per-(row, tile) raw-accumulator threshold of a tau sweep's tensor-core
// candidate pass (search_tc.cu, tc_gemm_kernel with NT > 1: one pass, up to NT_MAX taus).  Plain functions: the device
// calls them in the epilogue, the CPU tests (tests/host_emul/sweep_bound_host.cpp) call the very same code.  Build the host
// side with -ffp-contract=off: every product that feeds an addition is written as an explicit fmaf, so both sides round
// identically.  The one exception is the reciprocal of the proximity term: the device takes __fdividef (what the
// single-tau epilogue takes), the host the correctly rounded quotient; the 1.000001 factor of beta_bound() is there to
// absorb the device's 2-ulp reciprocal.
#pragma once

#include <math.h>

#ifdef __CUDACC__
#define ASP_SW_HD __host__ __device__ __forceinline__
#else
#define ASP_SW_HD inline
#endif

namespace asp_sweep {

constexpr int NT_MAX = 3;                    // taus per candidate pass (the sweep instantiations of tc_gemm_kernel; 4 spills registers)
constexpr float ACC_SCALE = 16384.0f;        // the raw accumulator is 2^14 cos~ (search_tc.cu ACC_SCALE)

ASP_SW_HD float rcp(float x)
{
#ifdef __CUDA_ARCH__
    return __fdividef(1.0f, x);
#else
    return 1.0f / x;
#endif
}

// 1 / (1 + |lambda_q - lambda_x|): shared by the T scores of one column
ASP_SW_HD float prox(float lq, float lam) { return rcp(1.0f + fabsf(lq - lam)); }

// The approximate score of one column at one tau, the single-tau epilogue's expression: beta prox + tau cos~.
ASP_SW_HD float score(float tau, float beta, float px, float acc) { return fmaf(beta, px, tau * (acc * (1.0f / ACC_SCALE))); }

// Upper bound of prox over a tile whose lambdas lie in [tl, th], shared by the taus: beta_bound(beta, it) is the
// single-tau epilogue's bound of beta prox (the 2.5e-7 / 1.000001 keep it safe against the f32 roundings of lambda_q and
// the interval, and the device's reciprocal).
ASP_SW_HD float prox_bound(float lq, float tl, float th)
{
    const float gap = fmaxf(0.f, fmaxf(lq - th, tl - lq) - 2.5e-7f);
    return rcp(1.0f + gap);
}
ASP_SW_HD float beta_bound(float beta, float pb) { return beta * pb * 1.000001f; }

// The single-tau threshold: a column whose score at this tau reaches theta_emit has acc >= it (-inf: no pruning).
ASP_SW_HD float tau_threshold(float theta_emit, float beta_ub, float inv_tau)
{
    return fmaf(theta_emit - beta_ub, inv_tau, -1e-6f) * ACC_SCALE;
}

// One threshold for the sweep's common path: the smallest of the taus' own, so a column that some tau would emit is
// never dropped by the max-tree compare.  Unused slots carry theta_emit = +inf and do not lower it.
ASP_SW_HD float combined_threshold(const float *theta_emit, const float *beta, const float *inv_tau, float pb, int nt)
{
    float m = INFINITY;
    for (int t = 0; t < nt; ++t) m = fminf(m, tau_threshold(theta_emit[t], beta_bound(beta[t], pb), inv_tau[t]));
    return m;
}

}  // namespace asp_sweep
