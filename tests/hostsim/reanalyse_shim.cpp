// TEST-ONLY host build of the reanalyse status rule (cn_chess_ai_b200/csrc/xq_examples.cuh: ex_refresh_status, and ex_refresh_statuses,
// the claim and refresh kernels restated on the host).  Never loaded by the product package.
#include <cstdint>

#include "../../cn_chess_ai_b200/csrc/xq_examples.cuh"

using namespace xq;

extern "C" {
void ex_shim_refresh_statuses(int64_t m, const int64_t* index, int64_t size, const uint8_t* stale, const uint32_t* total, uint32_t* claim,
                              uint8_t* status) {
    ex_refresh_statuses(m, index, size, stale, total, claim, status);
}
uint8_t ex_shim_refresh_status(int64_t idx, int64_t size, uint32_t claim, uint32_t t, int stale, uint32_t total) {
    return ex_refresh_status(idx, size, claim, t, stale != 0, total);
}
}
