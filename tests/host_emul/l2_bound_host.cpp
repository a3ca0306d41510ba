// The f32 score and the per-(row, tile) raw-accumulator threshold of the Euclidean item graph's tensor-core pass
// (pyarrowspace_b200/csrc/l2_bound.cuh), exported for tests/test_l2_item_graph_cpu.py.
// Build: g++ -O2 -ffp-contract=off -fno-fast-math -shared -fPIC.
#include "../../pyarrowspace_b200/csrc/l2_bound.cuh"

extern "C" float l2_score(float A, float B, float acc) { return asp_l2::score(A, B, acc); }
extern "C" float l2_threshold(float A, float lo, float hi, float theta) { return asp_l2::threshold(A, lo, hi, theta); }
