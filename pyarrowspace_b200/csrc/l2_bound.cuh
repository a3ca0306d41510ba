// l2_bound.cuh -- the f32 score of the Euclidean item graph's tensor-core candidate pass (search_tc.cu, score kind L2) and
// its per-(row, tile) raw-accumulator threshold.  Plain functions: the device calls them in the epilogue, the CPU tests
// (tests/host_emul/l2_bound_host.cpp) call the very same code.  Build the host side with -ffp-contract=off: every product
// that feeds an addition is written as an explicit fmaf, so both sides round identically.
#pragma once

#include <math.h>

#ifdef __CUDACC__
#define ASP_L2_HD __host__ __device__ __forceinline__
#else
#define ASP_L2_HD inline
#endif

namespace asp_l2 {

constexpr float ACC_INV = 1.0f / 16384.0f;   // the raw accumulator is 2^14 cos~ (search_tc.cu ACC_SCALE)
constexpr float K_REL = 1e-5f;               // relative slack of the bound (>= 160 f32 ulps, see threshold())
constexpr float Z_ABS = 1e-36f;              // absolute slack: f32 underflow of squares of tiny norms

// -d^2~ of a row of norm A and a column of norm B (f32 copies of the left-to-right norms) whose raw accumulator is acc:
//     d^2 = (A - B)^2 + 2AB (1 - cos)        (no cancellation: both terms are >= 0 up to the band of cos~)
// A zero row or column has a zero operand, hence acc = 0 and d^2 = B^2 (or A^2).  The product acc * 2^-14 is exact.
ASP_L2_HD float score(float A, float B, float acc)
{
    const float t = A - B;
    const float w = (2.0f * A) * B;
    const float u = 1.0f - acc * ACC_INV;
    return -fmaf(t, t, w * u);
}

// Smallest raw accumulator a column of a tile with norms in [lo, hi] (0 <= lo <= hi) can have if score(A, B, acc) >= theta.
// Norms up to 1e18 (A, hi): their squares and the score stay finite in f32 (the item graph refuses larger norms).
// Every column whose f32 score reaches theta has acc >= threshold(A, lo, hi, theta); -inf: no pruning, +inf: none can.
//
// With D^2 = -theta, score >= theta means fl(d^2) <= D^2.  The three roundings of score() and the one of the fma leave
// |fl(d^2) - (A^2 + B^2 - 2ABc)| <= 5.01 u ((A - B)^2 + 2AB|1 - c|) <= 5.01 u (1 + |c|)(A^2 + B^2), u = 2^-24, so for
// |c| < 2 a passing column satisfies (1 - K)(A^2 + B^2) - 2ABc <= D^2 + Z, i.e.
//     c >= g(B) = (1 - K) / (2A) * (E^2 / B + B),     E^2 = A^2 - (D^2 + Z) / (1 - K).
// g is convex on B > 0: for E^2 > 0 its minimum over [lo, hi] is at B* = E clamped into [lo, hi] (g(E) = (1 - K) E / A);
// for E^2 <= 0 it increases, so the minimum is at lo (lo = 0: no bound).  The f32 evaluation of g below errs by a few ulps
// of max(A^2, D^2, B^2) / (2AB); K = 160 u absorbs that wherever g lies in [-1.5, 1.5], and outside that range the answer
// (reject all / keep all) does not depend on it.  The result is rounded down once more by 2 ulps before scaling.
ASP_L2_HD float threshold(float A, float lo, float hi, float theta)
{
    if (!(theta > -INFINITY)) return -INFINITY;                        // no finite threshold yet
    const float r = 1.0f - K_REL;
    const float D2 = Z_ABS - theta;                                    // -theta + Z
    if (!(A > 0.0f)) {                                                 // zero row: acc = 0, fl(d^2) = fl(B^2) >= (1 - u) lo^2
        const float lo2 = lo * lo;
        return (r * lo2 > D2) ? INFINITY : -INFINITY;
    }
    const float E2 = fmaf(A, A, -(D2 / r));
    float b;
    if (E2 > 0.0f) {
        b = fminf(fmaxf(sqrtf(E2), lo), hi);
        if (!(b > 0.0f)) return INFINITY;                              // only zero columns: d^2 = A^2 > D^2
    } else {
        if (!(lo > 0.0f)) return -INFINITY;
        b = lo;
    }
    const float g = (r / (2.0f * A)) * (E2 / b + b);
    if (!(g > -2.0f)) return -INFINITY;                                // |c~| < 2: every column passes
    if (g > 2.0f) return INFINITY;
    return (g - 2.4e-7f) * 16384.0f;                                   // g in (-2, 2]: 2 ulps of 2 below, then exact scaling
}

}  // namespace asp_l2
