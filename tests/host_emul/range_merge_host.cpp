// CPU walk of the cross-shard range merge of pyarrowspace_b200/csrc/range.cuh (test infrastructure:
// tests/test_range_search_cpu.py): the offset tables asp_range_merge builds on the host and range_merge_kernel, every
// thread index walked in an order that differs from the GPU's only where threads are independent; plus the sort key.
// Build: g++ -O2 -ffp-contract=off -shared -fPIC.
#include <vector>

#include "../../pyarrowspace_b200/csrc/range.cuh"

extern "C" void range_merge_emulate(int parts, int64_t nq, const int64_t *counts, const int64_t *idx, const double *score,
                                    int64_t *out_idx, double *out_score)
{
    std::vector<int64_t> part_off((size_t)parts * (nq + 1)), out_off((size_t)nq + 1);
    const int64_t total = asp_range::merge_tables(parts, nq, counts, part_off.data(), out_off.data());
    const int64_t threads = 3 * 256;                         // range_merge_kernel: grid-stride, a grid smaller than the work
    for (int64_t tid = threads - 1; tid >= 0; --tid)
        for (int64_t t = tid; t < total; t += threads)
            asp_range::merge_elem(t, parts, nq, part_off.data(), out_off.data(), idx, score, out_idx, out_score);
}

extern "C" uint64_t range_desc_key(double s) { return asp_range::desc_key(s); }
extern "C" double range_key_score(uint64_t k) { return asp_range::key_score(k); }
