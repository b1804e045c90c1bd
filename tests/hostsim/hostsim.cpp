// TEST-ONLY host build of the device rules header (cn_chess_ai_b200/csrc/xq_rules.cuh).
// It lets the CPU-only test suite diff the exact source the CUDA kernels compile against
// the oracle on millions of positions before any GPU time is spent.  This library lives
// under tests/ and is never loaded by the product package: the product has no CPU path.
#include <cstdint>
#include <cstring>
#include "../../cn_chess_ai_b200/csrc/xq_rules.cuh"
#include "../../cn_chess_ai_b200/csrc/xq_bitboard.cuh"
#include "../../cn_chess_ai_b200/csrc/xq_rollout_team.cuh"
#include "../../cn_chess_ai_b200/csrc/xq_rollout_lane.cuh"
#include "../../cn_chess_ai_b200/csrc/xq_act_team.cuh"
#include "../../include/xq.h"

namespace {
struct RecBoard {
    const uint32_t* w;
    int get(int s) const { return (w[s >> 3] >> ((s & 7) * 4)) & 15; }
};
}

// ---- the team rollout kernel's ply (xq_rollout_team.cuh), one board at a time: the 4 threads of a board run phase by phase ----
namespace {
using namespace xq;
template <int T>
int team_rollout_host(xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace, xq_env_stats* stats) {
    constexpr int S = 16 / T;
    int nonstd = 0;
    for (long env = 0; env < n; ++env) {
        TeamShared<1> sh;
        team_tables_init(sh, 0, 1);
        uint8_t slot[32];
        for (int i = 0; i < 32; ++i) slot[i] = kDeadSq;
        uint32_t w[12];
        std::memcpy(w, recs[env].sq, 48);
        Bits90 red, black, occT;
        if (!team_unpack_record(w, red, black, occT, [&](int s, int q) { slot[s] = (uint8_t)q; })) { ++nonstd; continue; }
        TeamRole R[T];
        TeamState st[T];
        TeamPly pl[T];
        TeamBook bk{0, 0, 1480, 1480, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        bk.red = recs[env].red_score; bk.black = recs[env].black_score;
        bk.mat_red = bk.mat_black = 0;
        for (int i = 0; i < 16; ++i) {
            if (slot[i] != kDeadSq) bk.mat_red += piece_score(slot_type(i));
            if (slot[16 + i] != kDeadSq) bk.mat_black += piece_score(slot_type(i));
        }
        const bool finished = recs[env].move_count >= XQ_MAX_MOVES || slot[8] == kDeadSq || slot[24] == kDeadSq;
        if (finished) { bk.red = bk.black = 0; bk.mat_red = bk.mat_black = 1480; }
        for (int r = 0; r < T; ++r) {
            R[r] = team_role<T>(r);
            team_reset(R[r], st[r]);
            st[r].ctr = recs[env].ctr;
            if (finished) continue;
            uint32_t wr = 0, wb = 0;
            for (int i = 0; i < 4; ++i) {
                const int s = (int)((R[r].slots >> (8 * i)) & 0xFFu);
                wr |= (uint32_t)(i < S ? slot[s] : kDeadSq) << (8 * i);
                wb |= (uint32_t)(i < S ? slot[16 + s] : kDeadSq) << (8 * i);
            }
            st[r].occT = occT; st[r].move_count = recs[env].move_count; st[r].player = recs[env].player;
            const bool redp = recs[env].player == 0;
            st[r].sq_own = redp ? wr : wb; st[r].sq_opp = redp ? wb : wr;
            st[r].own = redp ? red : black; st[r].opp = redp ? black : red;
            st[r].gen_own = redp ? slot[8] : slot[24]; st[r].gen_opp = redp ? slot[24] : slot[8];
        }
        const uint64_t base = seed + (env_id0 + (uint64_t)env) * 0x9E3779B97F4A7C15ull;
        const uint32_t ctr0 = st[0].ctr;
        for (int r = 0; r < T; ++r) team_rng_chunk<T, 1>(R[r], sh, 0, 0, base, ctr0);
        // the rollout kernel's teams of 4 read their bitboards through the memory view; the one-ply kernels (below) keep them in registers
        TeamViewMem<1> vmem;
        uint32_t* const view = T == 4 ? vmem.w : nullptr;
        if (view) for (int r = 0; r < T; ++r) team_view_put<1>(R[r], st[r], view, 0);
        for (int p = 0; p < n_plies; ++p) {
            if ((p & 15) == 0) for (int r = 0; r < T; ++r) team_rng_chunk<T, 1>(R[r], sh, 0, (p >> 4) + 1, base, ctr0);
            for (int r = 0; r < T; ++r) team_phase_a<T, 1>(R[r], st[r], pl[r], sh, 0, p, view);
            team_finalize<1>(bk, sh, 0, trace, n, env);
            for (int r = 0; r < T; ++r) team_phase_b<T, 1>(R[r], st[r], pl[r], sh, 0, p);
            for (int r = 0; r < T; ++r) team_phase_c<1>(R[r], st[r], pl[r], sh, bk, 0, p, view);
        }
        team_finalize<1>(bk, sh, 0, trace, n, env);
        // store
        for (int r = 0; r < T; ++r) {
            const uint32_t wr = st[r].player == 0 ? st[r].sq_own : st[r].sq_opp, wb = st[r].player == 0 ? st[r].sq_opp : st[r].sq_own;
            for (int i = 0; i < S; ++i) {
                const int s = (int)((R[r].slots >> (8 * i)) & 0xFFu);
                slot[s] = (uint8_t)(wr >> (8 * i)); slot[16 + s] = (uint8_t)(wb >> (8 * i));
            }
        }
        uint32_t words[12] = {0};
        for (int i = 0; i < 32; ++i)
            if (slot[i] != kDeadSq) words[slot[i] >> 3] |= (uint32_t)(slot_type(i & 15) + (i >= 16 ? 7 : 0)) << (4 * (slot[i] & 7));
        std::memcpy(recs[env].sq, words, 48);
        recs[env].move_count = (uint16_t)st[0].move_count; recs[env].player = (uint8_t)st[0].player;
        recs[env].red_score = bk.red; recs[env].black_score = bk.black; recs[env].ctr = st[0].ctr;
        if (stats) {
            stats->steps += bk.a_steps; stats->games += bk.a_games; stats->red_wins += bk.a_red; stats->black_wins += bk.a_black;
            stats->cap_games += bk.a_capg; stats->captures += bk.a_caps; stats->reward_sum += bk.a_reward; stats->legal_sum += bk.a_legal;
        }
    }
    return nonstd;
}
}

// ---- the board-per-thread rollout kernel's ply (xq_rollout_lane.cuh), one board at a time ----
namespace {
const uint32_t* host_geo() {
    static uint32_t g[xq::kGeoWords];
    static bool init = false;
    if (!init) { for (int i = 0; i < xq::kGeoWords; ++i) g[i] = xq::geo_entry(i >> 7, i & 127); init = true; }
    return g;
}
int lane_rollout_host(xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace, xq_env_stats* stats) {
    int nonstd = 0;
    uint32_t magic[XQ_MAX_ACTIONS + 1] = {0};
    for (int d = 1; d <= XQ_MAX_ACTIONS; ++d) magic[d] = team_mod_magic((uint32_t)d);
    for (long env = 0; env < n; ++env) {
        uint8_t slot[32];
        for (int i = 0; i < 32; ++i) slot[i] = kDeadSq;
        uint32_t w[12];
        std::memcpy(w, recs[env].sq, 48);
        Bits90 red, black, occT;
        uint32_t scratch[12];
        if (!team_unpack_record_m(w, scratch, 1, red, black, occT, [&](int s, int q) { slot[s] = (uint8_t)q; })) { ++nonstd; continue; }
        LaneState st;
        LaneStats a{0, 0, 0, 0, 0, 0, 0, 0};
        lane_load(st, [&](int s) { return (int)slot[s]; }, red, black, occT, recs[env].move_count, recs[env].player, recs[env].red_score,
                  recs[env].black_score, recs[env].ctr);
        const uint64_t base = seed + (env_id0 + (uint64_t)env) * 0x9E3779B97F4A7C15ull;
        uint32_t vm[kViewWords];
        view_init(vm, 1);
        view_store(vm, 1, st.own, st.opp, st.occT);
        for (int p = 0; p < n_plies; ++p) lane_ply(st, a, base, magic, host_geo(), vm, 1, trace ? trace + ((long)p * n + env) : nullptr);
        uint32_t words[12], words2[12];
        lane_store_words(st, words2);
        lane_store_words_mem(st, vm, 1, words);
        if (std::memcmp(words, words2, 48) != 0) return -1;      // the two forms of the record builder must agree
        std::memcpy(recs[env].sq, words, 48);
        recs[env].move_count = (uint16_t)st.move_count; recs[env].player = (uint8_t)st.player;
        recs[env].red_score = st.red; recs[env].black_score = st.black; recs[env].ctr = st.ctr;
        if (stats) {
            stats->steps += a.steps; stats->games += a.games; stats->red_wins += a.red; stats->black_wins += a.black;
            stats->cap_games += a.capg; stats->captures += a.caps; stats->reward_sum += a.reward; stats->legal_sum += a.legal;
        }
    }
    return nonstd;
}
}

// ---- DQN::selectAction through the team act phases (xq_act_team.cuh), one board at a time ----
namespace {
int act_team_host(const xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, const float* q90, uint32_t eps_thr, uint16_t* actions) {
    int nonstd = 0;
    for (long env = 0; env < n; ++env) {
        actions[env] = XQ_ACTION_NONE;
        TeamShared<1> sh;
        ActShared<1> as;
        team_tables_init(sh, 0, 1);
        for (int t = 0; t < kQStride; ++t) as.qt[t * 2] = q90[env * kQStride + t];
        uint8_t slot[32];
        for (int i = 0; i < 32; ++i) slot[i] = kDeadSq;
        uint32_t w[12];
        std::memcpy(w, recs[env].sq, 48);
        Bits90 red, black, occT;
        if (!team_unpack_record(w, red, black, occT, [&](int s, int q) { slot[s] = (uint8_t)q; })) { ++nonstd; continue; }
        TeamRole R[4];
        TeamState st[4];
        TeamPly pl[4];
        uint32_t kbest[4][4];
        for (int r = 0; r < 4; ++r) {
            R[r] = team_role<4>(r);
            uint32_t wr = 0, wb = 0;
            for (int i = 0; i < 4; ++i) {
                const int s = (int)((R[r].slots >> (8 * i)) & 0xFFu);
                wr |= (uint32_t)slot[s] << (8 * i);
                wb |= (uint32_t)slot[16 + s] << (8 * i);
            }
            const bool redp = recs[env].player == 0;
            st[r].occT = occT; st[r].move_count = recs[env].move_count; st[r].player = recs[env].player; st[r].ctr = recs[env].ctr;
            st[r].sq_own = redp ? wr : wb; st[r].sq_opp = redp ? wb : wr;
            st[r].own = redp ? red : black; st[r].opp = redp ? black : red;
            st[r].gen_own = redp ? slot[8] : slot[24]; st[r].gen_opp = redp ? slot[24] : slot[8];
        }
        for (int r = 0; r < 4; ++r) { team_phase_a<4, 1>(R[r], st[r], pl[r], sh, 0, 0); act_best<1>(R[r], st[r], pl[r], as, 0, kbest[r]); }
        const uint64_t x = rng(seed, env_id0 + (uint64_t)env, recs[env].ctr);
        uint32_t tot = 0;
        for (int r = 0; r < 4; ++r) tot = act_select<1>(R[r], st[r], pl[r], sh, as, 0, kbest[r], x, eps_thr);
        if (tot > 0) { const uint32_t mv = sh.move[0]; actions[env] = XQ_ACTION(mv & 0xFFu, (mv >> 8) & 0xFFu); }
    }
    return nonstd;
}
}

extern "C" {
int hs_act_team(const xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, const float* q90, uint32_t eps_thr, uint16_t* actions) {
    return act_team_host(recs, n, env_id0, seed, q90, eps_thr, actions);
}
// the register-resident list kernel's generator + emission (legal_moves_lane_kernel); returns the number of non-standard boards (skipped)
int hs_lane_all_actions(const xq_env_rec* recs, long n, uint8_t* counts, uint16_t* actions) {
    int nonstd = 0;
    for (long i = 0; i < n; ++i) {
        uint16_t* out = actions + i * XQ_MAX_ACTIONS;
        for (int k = 0; k < XQ_MAX_ACTIONS; ++k) out[k] = XQ_ACTION_NONE;
        counts[i] = 0xFF;
        uint8_t slot[32];
        for (int k = 0; k < 32; ++k) slot[k] = xq::kDeadSq;
        uint32_t w[12];
        std::memcpy(w, recs[i].sq, 48);
        xq::Bits90 red, black, occT;
        uint32_t scratch[12];
        if (!xq::team_unpack_record_m(w, scratch, 1, red, black, occT, [&](int s, int q) { slot[s] = (uint8_t)q; })) { ++nonstd; continue; }
        {   // the one-loop unpack places the pieces exactly like the per-word form
            uint8_t slot2[32];
            for (int k = 0; k < 32; ++k) slot2[k] = xq::kDeadSq;
            xq::Bits90 r2, b2, o2;
            if (!xq::team_unpack_record(w, r2, b2, o2, [&](int s, int q) { slot2[s] = (uint8_t)q; }) || std::memcmp(slot, slot2, 32) != 0 ||
                r2.w0 != red.w0 || r2.w2 != red.w2 || b2.w1 != black.w1 || o2.w0 != occT.w0 || o2.w1 != occT.w1 || o2.w2 != occT.w2) return -1;
        }
        const int player = recs[i].player;
        uint32_t own_sq[4] = {0, 0, 0, 0};
        for (int pos = 0; pos < 16; ++pos) own_sq[pos >> 2] |= (uint32_t)slot[(player ? 16 : 0) + xq::lane_pos_slot(pos)] << (8 * (pos & 3));
        uint32_t sdesc[4], cw[4], dw[4];
        uint32_t vm[xq::kViewWords];
        xq::view_init(vm, 1);
        xq::view_store(vm, 1, player ? black : red, player ? red : black, occT);
        xq::lane_movegen(own_sq, xq::MemView{vm, 1}, player, host_geo(), sdesc, cw, dw);
        counts[i] = (uint8_t)xq::lane_emit_actions(own_sq, player, sdesc, cw, dw, [&](int idx, int a, bool live) { if (live) out[idx] = (uint16_t)a; });
    }
    return nonstd;
}
// the team list kernel's phases (legal_moves_team_kernel: team_phase_a + team_emit_actions), the 4 threads of a board one after the other
int hs_team_all_actions(const xq_env_rec* recs, long n, uint8_t* counts, uint16_t* actions) {
    using namespace xq;
    int nonstd = 0;
    for (long env = 0; env < n; ++env) {
        uint16_t* out = actions + env * XQ_MAX_ACTIONS;
        for (int k = 0; k < XQ_MAX_ACTIONS; ++k) out[k] = XQ_ACTION_NONE;
        counts[env] = 0xFF;
        TeamShared<1> sh;
        team_tables_init(sh, 0, 1);
        uint8_t slot[32];
        for (int i = 0; i < 32; ++i) slot[i] = kDeadSq;
        uint32_t w[12];
        std::memcpy(w, recs[env].sq, 48);
        // the kernel unpacks the two colours in two warps (team_unpack_side)
        Bits90 bb[2], oT[2];
        bool ok = true;
        for (int side = 0; side < 2; ++side) ok &= team_unpack_side(w, side, bb[side], oT[side], [&](int s, int q) { slot[side * 16 + s] = (uint8_t)q; });
        if (!ok) { ++nonstd; continue; }
        TeamRole R[4];
        TeamState st[4];
        TeamPly pl[4];
        for (int r = 0; r < 4; ++r) {
            R[r] = team_role<4>(r);
            team_reset(R[r], st[r]);
            uint32_t wr = 0, wb = 0;
            for (int i = 0; i < 4; ++i) {
                const int s = (int)((R[r].slots >> (8 * i)) & 0xFFu);
                wr |= (uint32_t)slot[s] << (8 * i);
                wb |= (uint32_t)slot[16 + s] << (8 * i);
            }
            const bool redp = recs[env].player == 0;
            st[r].occT = Bits90{oT[0].w0 | oT[1].w0, oT[0].w1 | oT[1].w1, oT[0].w2 | oT[1].w2};
            st[r].move_count = recs[env].move_count; st[r].player = recs[env].player; st[r].ctr = recs[env].ctr;
            st[r].sq_own = redp ? wr : wb; st[r].sq_opp = redp ? wb : wr;
            st[r].own = redp ? bb[0] : bb[1]; st[r].opp = redp ? bb[1] : bb[0];
        }
        for (int r = 0; r < 4; ++r) team_phase_a<4, 1>(R[r], st[r], pl[r], sh, 0, 0);
        uint32_t tot = 0;
        for (int r = 0; r < 4; ++r) tot = team_emit_actions<1>(R[r], st[r], pl[r], sh, 0, [&](int idx, int a) { out[idx] = (uint16_t)a; });
        counts[env] = (uint8_t)tot;
    }
    return nonstd;
}
// DQN::selectAction through the board-per-thread functions of xq_rollout_lane.cuh: same contract as hs_act_team
int hs_act_lane(const xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, const float* q90, uint32_t eps_thr, uint16_t* actions) {
    int nonstd = 0;
    uint32_t magic[XQ_MAX_ACTIONS + 1] = {0};
    for (int d = 1; d <= XQ_MAX_ACTIONS; ++d) magic[d] = xq::team_mod_magic((uint32_t)d);
    for (long i = 0; i < n; ++i) {
        actions[i] = XQ_ACTION_NONE;
        uint8_t slot[32];
        for (int k = 0; k < 32; ++k) slot[k] = xq::kDeadSq;
        uint32_t w[12];
        std::memcpy(w, recs[i].sq, 48);
        xq::Bits90 red, black, occT;
        if (!xq::team_unpack_record(w, red, black, occT, [&](int s, int q) { slot[s] = (uint8_t)q; })) { ++nonstd; continue; }
        const int player = recs[i].player;
        uint32_t own_sq[4] = {0, 0, 0, 0};
        for (int pos = 0; pos < 16; ++pos) own_sq[pos >> 2] |= (uint32_t)slot[(player ? 16 : 0) + xq::lane_pos_slot(pos)] << (8 * (pos & 3));
        uint32_t sdesc[4], cw[4], dw[4], tot = 0;
        uint32_t vm[xq::kViewWords];
        xq::view_init(vm, 1);
        xq::view_store(vm, 1, player ? black : red, player ? red : black, occT);
        xq::lane_movegen(own_sq, xq::MemView{vm, 1}, player, host_geo(), sdesc, cw, dw);
        for (int k = 0; k < 4; ++k) tot = xq::dp4a_u(cw[k], 0x01010101u, tot);
        if (tot == 0) continue;
        const uint64_t x = xq::rng(seed, env_id0 + (uint64_t)i, recs[i].ctr);
        const uint32_t coin31 = (uint32_t)(x & 0x7FFFFFFFu), idx31 = (uint32_t)(x >> 33);
        const float* q = q90 + i * 96;
        const uint32_t mv = coin31 < eps_thr ? xq::lane_select_kth(own_sq, player, sdesc, cw, dw, xq::team_mod(idx31, tot, magic[tot]), tot)
                                             : xq::lane_select_greedy(own_sq, player, sdesc, cw, dw, [&](int to) { return q[to]; });
        actions[i] = XQ_ACTION(mv & 0xFFu, (mv >> 8) & 0xFFu);
    }
    return nonstd;
}
int hs_lane_rollout(xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace, xq_env_stats* stats) {
    return lane_rollout_host(recs, n, env_id0, seed, n_plies, trace, stats);
}
// whole fused rollout through the team kernel's phases; returns the number of boards it does not handle (non-standard piece sets),
// or -1 for a team size other than 4, the only one the rollout kernel runs
int hs_team_rollout(int team, xq_env_rec* recs, long n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace, xq_env_stats* stats) {
    return team == 4 ? team_rollout_host<4>(recs, n, env_id0, seed, n_plies, trace, stats) : -1;
}
// opt-in strict legality (xq_rules.cuh: leaves_general_safe): the reference-ordered list filtered
void hs_all_actions_strict(const xq_env_rec* recs, long n, uint8_t* counts, uint16_t* actions) {
    struct MutBoard {
        uint32_t w[12];
        int get(int s) const { return (w[s >> 3] >> ((s & 7) * 4)) & 15; }
        void set(int s, int code) { w[s >> 3] = (w[s >> 3] & ~(15u << ((s & 7) * 4))) | ((uint32_t)code << ((s & 7) * 4)); }
    };
    for (long i = 0; i < n; ++i) {
        MutBoard b;
        std::memcpy(b.w, recs[i].sq, 48);
        uint16_t* out = actions + i * XQ_MAX_ACTIONS;
        for (int k = 0; k < XQ_MAX_ACTIONS; ++k) out[k] = XQ_ACTION_NONE;
        uint16_t all[XQ_MAX_ACTIONS];
        int cnt = 0, kept = 0;
        const MutBoard& cb = b;
        xq::all_actions(cb, recs[i].player, [&](int from, int to) { if (cnt < XQ_MAX_ACTIONS) all[cnt++] = XQ_ACTION(from, to); });
        for (int k = 0; k < cnt; ++k)
            if (xq::leaves_general_safe(b, recs[i].player, XQ_ACTION_FROM(all[k]), XQ_ACTION_TO(all[k]))) out[kept++] = all[k];
        counts[i] = (uint8_t)kept;
    }
}
void hs_all_actions(const xq_env_rec* recs, long n, uint8_t* counts, uint16_t* actions) {
    for (long i = 0; i < n; ++i) {
        RecBoard b{recs[i].sq};
        uint16_t* out = actions + i * XQ_MAX_ACTIONS;
        for (int k = 0; k < XQ_MAX_ACTIONS; ++k) out[k] = XQ_ACTION_NONE;
        int cnt = 0;
        xq::all_actions(b, recs[i].player, [&](int from, int to) { if (cnt < XQ_MAX_ACTIONS) out[cnt++] = XQ_ACTION(from, to); });
        counts[i] = (uint8_t)cnt;
    }
}
int hs_valid_moves(const xq_env_rec* rec, int row, int col, uint8_t* to) {
    RecBoard b{rec->sq};
    int n = 0;
    if (!xq::inside(row, col)) return 0;
    int code = b.get(row * 9 + col);
    if (code) xq::gen_piece(b, row, col, code, [&](int t) { to[n++] = (uint8_t)t; });
    return n;
}
int hs_is_valid_move(const xq_env_rec* rec, int fr, int fc, int tr, int tc) {
    RecBoard b{rec->sq};
    return xq::is_valid_move(b, fr, fc, tr, tc) ? 1 : 0;
}
// bitboard count + k-th decode (xq_bitboard.cuh), enumerated piece by piece in square order
void hs_bb_all_actions(const xq_env_rec* recs, long n, uint8_t* counts, uint16_t* actions) {
    for (long i = 0; i < n; ++i) {
        RecBoard b{recs[i].sq};
        const int player = recs[i].player;
        xq::Pos P{{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
        for (int s = 0; s < 90; ++s) {
            const int code = b.get(s);
            if (!code) continue;
            P.occ.set(s); P.occT.set(xq::cm_index(s / 9, s % 9));
            if ((code >= 8) == (player == 1)) P.own.set(s);
        }
        uint16_t* out = actions + i * XQ_MAX_ACTIONS;
        for (int k = 0; k < XQ_MAX_ACTIONS; ++k) out[k] = XQ_ACTION_NONE;
        int cnt = 0;
        for (int s = 0; s < 90; ++s) {
            const int code = b.get(s);
            if (!code || (code >= 8) != (player == 1)) continue;
            int dummy = -1;
            const int c = xq::piece_moves_dyn(xq::type_of(code), P, s, player, -1, &dummy);
            for (int j = 0; j < c; ++j) {
                int to = -1;
                xq::piece_moves_dyn(xq::type_of(code), P, s, player, j, &to);
                if (cnt < XQ_MAX_ACTIONS) out[cnt++] = XQ_ACTION(s, to);
            }
        }
        counts[i] = (uint8_t)cnt;
    }
}
// step_kernel's board summary (summarize_words, xq_bitboard.cuh): out[i] = {mat_red, mat_black, lowest square of the Red General or 127, same for Black}
void hs_summarize_words(const xq_env_rec* recs, long n, int* out) {
    for (long i = 0; i < n; ++i) {
        uint32_t w[12];
        std::memcpy(w, recs[i].sq, 48);
        const xq::WordSummary s = xq::summarize_words(w);
        out[4 * i] = s.mat_red; out[4 * i + 1] = s.mat_black; out[4 * i + 2] = s.gen_red; out[4 * i + 3] = s.gen_black;
    }
}
int hs_reward(int material_diff, int move_count) { return xq::reward_from_material(material_diff, move_count); }
int hs_piece_score(int type) { return xq::piece_score(type); }
uint64_t hs_rng(uint64_t seed, uint64_t env, uint32_t ctr) { return xq::rng(seed, env, ctr); }
}

// ---- the scale and the entries of the acting path's fixed-point layer-0 table (xq_act_quant.cuh) ----
#include "../../cn_chess_ai_b200/csrc/xq_act_quant.cuh"
extern "C" int hs_act_quant(const float* w, long n, int32_t* q_out) {
    uint32_t m = 0;
    for (long i = 0; i < n; ++i) { uint32_t b; std::memcpy(&b, &w[i], 4); b &= 0x7FFFFFFFu; if (b > m) m = b; }      // act_quant_max_kernel
    const int k = xq::act_quant_shift(m);
    for (long i = 0; i < n; ++i) q_out[i] = xq::act_quantize(w[i], k);                                             // act_quant_kernel
    return k;
}
