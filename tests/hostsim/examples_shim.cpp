// TEST-ONLY host build of the example-buffer helpers (cn_chess_ai_b200/csrc/xq_examples.cuh, xq_examples_*), compiled with
// -ffp-contract=off like search_shim.cpp: the cleaned result and the z sign, the policy-target division, the view of a stored action, the
// sample-index draw and the commit offsets of the scan.  Never loaded by the product package.
#include <cstdint>
#include <cstring>

#include "../../cn_chess_ai_b200/csrc/xq_examples.cuh"

using namespace xq;

extern "C" {
float ex_shim_z(float result_red, int player) { return ex_z(result_red, player); }
float ex_shim_policy(uint32_t visits, uint32_t total) { return ex_policy(visits, total); }
int ex_shim_view_index(int action, int player, int view) { return ex_view_index(action, player, view); }
void ex_shim_sample_index(uint64_t seed, uint32_t counter, int64_t size, int64_t batch, int64_t* out) {
    for (int64_t i = 0; i < batch; ++i) out[i] = ex_sample_index(seed, i, counter, size);
}
int64_t ex_shim_commit_offsets(int64_t n, int threads, const uint8_t* ended, const uint32_t* staged, int64_t base, int64_t* off) {
    return ex_commit_offsets(n, threads, ended, staged, base, off);
}
int64_t ex_shim_find_env(const int64_t* off, int64_t n, int64_t pos) { return ex_find_env(off, n, pos); }
}
