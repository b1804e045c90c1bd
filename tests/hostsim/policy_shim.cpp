// TEST-ONLY host build of the external-policy helpers (cn_chess_ai_b200/csrc/xq_policy.cuh), board by board, as the kernels of
// xq_policy.cu run them: the register-resident generator with its mask emission and its choice over the staged score row, and the
// generic path (all_actions in list order) for the boards the generator does not take.  Never loaded by the product package.
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
// the generic kernels' enumeration: a player byte > 1 owns no piece
template <class F>
void generic_actions(const xq_env_rec& r, F&& f) {
    if (r.player <= 1) all_actions(RecBoard{r.sq}, r.player, f);
}
}  // namespace

extern "C" {
// mask_lane_kernel / mask_generic_kernel: packed rows [n][254]; path[i] = 0 generator, 1 generic
void ps_mask(const xq_env_rec* recs, long n, int view, uint32_t* mask, uint8_t* path) {
    for (long i = 0; i < n; ++i) {
        uint32_t* row = mask + i * XQ_MASK_WORDS;
        std::memset(row, 0, 4 * XQ_MASK_WORDS);
        const int player = recs[i].player;
        const bool flip = policy_flip(player, view);
        auto set = [&](int from, int to) { const int k = policy_index(from, to, flip); row[k >> 5] |= 1u << (k & 31); };
        uint32_t w[12], vm[kViewWords];
        uint8_t slot[32];
        std::memcpy(w, recs[i].sq, 48);
        LaneGen g;
        if (policy_lane_gen(w, player, vm, slot, 1, host_geo(), g)) {
            path[i] = 0;
            policy_lane_emit(g, player, [&](int, int from, int to) { set(from, to); });
        } else {
            path[i] = 1;
            generic_actions(recs[i], set);
        }
    }
}

// the choice of policy_step_lane_kernel / policy_step_generic_kernel (nothing is applied): out_idx = policy index of the played action
// (-1 = none), out_logp; scores f32 [n][8100] (may be null for GIVEN), given int64 [n] (GIVEN); force_generic: every board on the generic path
void ps_choose(const xq_env_rec* recs, long n, const float* scores, int view, int pick, float t, uint64_t seed, uint64_t env_id0,
               const int64_t* given, int force_generic, int64_t* out_idx, float* out_logp, uint8_t* path) {
    for (long i = 0; i < n; ++i) {
        const int player = recs[i].player;
        const bool flip = policy_flip(player, view);
        const float* sc = scores ? scores + i * XQ_POLICY_ACTIONS : nullptr;
        const int64_t gi = pick == XQ_PICK_GIVEN ? given[i] : -1;
        const float u = pick == XQ_PICK_SAMPLE ? policy_uniform(rng(seed, env_id0 + (uint64_t)i, recs[i].ctr)) : 0.f;
        PolicyBest best{-INFINITY, -1};
        int given_k = -1, cnt = 0, from = 0, to = 0;
        uint32_t w[12], vm[kViewWords];
        uint8_t slot[32];
        std::memcpy(w, recs[i].sq, 48);
        LaneGen g;
        PolicyChoice c;
        if (!force_generic && policy_lane_gen(w, player, vm, slot, 1, host_geo(), g)) {
            path[i] = 0;
            float row[XQ_MAX_ACTIONS];
            cnt = policy_lane_emit(g, player, [&](int idx, int f, int tt) {
                const int pi = policy_index(f, tt, flip);
                if (sc) row[idx] = sc[pi];
                given_k = pi == gi ? idx : given_k;
            });
            auto each = [&](auto&& f) { for (int k = 0; k < cnt; ++k) f(policy_clean(row[k])); };
            if (sc) { int k = 0; each([&](float l) { best.offer(l, k++); }); }
            c = policy_choose(each, cnt, best, given_k, pick, sc != nullptr, true, t, u);
            if (c.k >= 0) { const uint32_t mv = lane_select_kth(g.own_sq, player, g.sdesc, g.cw, g.dw, (uint32_t)c.k, (uint32_t)cnt); from = mv & 0xFF; to = (mv >> 8) & 0xFF; }
        } else {
            path[i] = 1;
            generic_actions(recs[i], [&](int f, int tt) {
                const int pi = policy_index(f, tt, flip);
                if (sc) best.offer(policy_clean(sc[pi]), cnt);
                given_k = pi == gi ? cnt : given_k;
                ++cnt;
            });
            c = policy_choose([&](auto&& f) { generic_actions(recs[i], [&](int ff, int tt) { f(policy_clean(sc[policy_index(ff, tt, flip)])); }); },
                              cnt, best, given_k, pick, sc != nullptr, true, t, u);
            int j = 0;
            if (c.k >= 0) generic_actions(recs[i], [&](int ff, int tt) { if (j == c.k) { from = ff; to = tt; } ++j; });
        }
        out_idx[i] = c.k >= 0 ? policy_index(from, to, flip) : -1;
        out_logp[i] = c.logp;
    }
}
}
