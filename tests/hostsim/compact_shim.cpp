// TEST-ONLY host build of the compact action lists (xq_env_legal_actions_device, xq_search_leaf_actions_device) from the helpers of
// cn_chess_ai_b200/csrc/xq_policy.cuh, board by board, as actions_lane_kernel / actions_generic_kernel (xq_policy.cu) emit them: the
// register-resident generator's list, or all_actions for the boards it refuses.  Never loaded by the product package.
#include <cstdint>
#include <cstring>

#include "../../cn_chess_ai_b200/csrc/xq_policy.cuh"

namespace {
using namespace xq;
struct RecBoard {
    const uint32_t* w;
    int get(int s) const { return (w[s >> 3] >> ((s & 7) * 4)) & 15; }
};
const uint32_t* host_geo() {
    static uint32_t g[kGeoWords];
    static bool init = false;
    if (!init) { for (int i = 0; i < kGeoWords; ++i) g[i] = geo_entry(i >> 7, i & 127); init = true; }
    return g;
}
}  // namespace

extern "C" {
// actions int32 [n][128] (policy indices in the frame of `view`, -1 past the count), counts u8 [n], path[i] = 0 generator, 1 generic
void cs_actions(const xq_env_rec* recs, long n, int view, int32_t* actions, uint8_t* counts, uint8_t* path) {
    for (long i = 0; i < n; ++i) {
        int32_t* row = actions + i * XQ_COMPACT_ACTIONS;
        const int player = recs[i].player;
        const bool flip = policy_flip(player, view);
        uint32_t w[12], vm[kViewWords];
        uint8_t slot[32];
        std::memcpy(w, recs[i].sq, 48);
        LaneGen g;
        int cnt = 0;
        if (policy_lane_gen(w, player, vm, slot, 1, host_geo(), g)) {
            path[i] = 0;
            cnt = policy_lane_emit(g, player, [&](int idx, int from, int to) { if (idx < XQ_COMPACT_ACTIONS) row[idx] = policy_index(from, to, flip); });
            cnt = cnt < XQ_COMPACT_ACTIONS ? cnt : XQ_COMPACT_ACTIONS;
        } else {
            path[i] = 1;
            if (player <= 1)
                all_actions(RecBoard{recs[i].sq}, player, [&](int from, int to) { if (cnt < XQ_COMPACT_ACTIONS) row[cnt++] = policy_index(from, to, flip); });
        }
        counts[i] = (uint8_t)cnt;
        for (int k = cnt; k < XQ_COMPACT_ACTIONS; ++k) row[k] = -1;
    }
}
}  // extern "C"
