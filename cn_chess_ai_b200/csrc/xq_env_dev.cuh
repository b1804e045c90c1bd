// xq_env_dev.cuh -- device helpers shared by the thread-per-board kernels (xq_env.cu, xq_selfplay.cu), the board steps of the policy
// and search kernels (xq_policy.cu, xq_search.cu) and the root check of the search and example kernels (xq_search.cu, xq_examples.cu).
#pragma once
#include "xq_common.cuh"
#include "xq_bitboard.cuh"

namespace xq {

constexpr int kThreads = 128;          // thread-per-board kernels: boards per CTA
constexpr int kListStride = 65;        // words per thread of the staged action list (64 + 1 pad)

// ------------------------------------------------------------------------------------------
// Board summary: material per colour, general presence, first general in index order
// (ChessBoard::checkGameOver :286-309, getWinner :312-320, ChessAI::evaluateBoard :311-342).
struct Summary {
    int mat_red, mat_black;
    int winner;          // colour of the first General in square order, NOCOLOR if none
    bool red_alive, black_alive;
};

template <class B>
__device__ __forceinline__ Summary summarize(const B& b) {
    Summary s{0, 0, NOCOLOR, false, false};
    for (int w = 0; w < 12; ++w) {
        uint32_t word = b.base[w * b.stride];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int code = (word >> (4 * i)) & 15;
            if (code == 0) continue;
            const int sc = piece_score(type_of(code));
            if (code >= 8) s.mat_black += sc; else s.mat_red += sc;
            if (code == GENERAL) { s.red_alive = true; if (s.winner == NOCOLOR) s.winner = RED; }
            if (code == GENERAL + 7) { s.black_alive = true; if (s.winner == NOCOLOR) s.winner = BLACK; }
        }
    }
    return s;
}

__device__ __forceinline__ void reset_board(SmemBoard& b) {
#pragma unroll
    for (int w = 0; w < 12; ++w) b.base[w * b.stride] = kOpening[w];
}

struct Meta {
    int move_count, player, red_score, black_score;
    uint32_t ctr;
    uint8_t flags;
    __device__ __forceinline__ void load(const xq_env_rec* r) {
        const uint4 m = reinterpret_cast<const uint4*>(r)[3];
        move_count = m.x & 0xFFFF; player = (m.x >> 16) & 0xFF; flags = (uint8_t)(m.x >> 24);
        red_score = (int)m.y; black_score = (int)m.z; ctr = m.w;
    }
    __device__ __forceinline__ void store(xq_env_rec* r) const {
        reinterpret_cast<uint4*>(r)[3] = make_uint4((uint32_t)(move_count & 0xFFFF) | ((uint32_t)player << 16) | ((uint32_t)flags << 24),
                                                    (uint32_t)red_score, (uint32_t)black_score, ctr);
    }
    __device__ __forceinline__ void reset() { move_count = 0; player = RED; red_score = 0; black_score = 0; }
};

// ChessBoard::movePiece after validation (src/chessboard.cpp:43-63); returns the captured code
__device__ __forceinline__ int apply_move(SmemBoard& b, Meta& m, int from, int to) {
    const int cap = b.get(to);
    b.set(to, b.get(from));
    b.set(from, 0);
    if (cap != 0) {
        const int sc = piece_score(type_of(cap));
        if (cap >= 8) m.red_score += sc; else m.black_score += sc;   // captured Black => Red scores (:53-57)
    }
    m.move_count++;
    m.player ^= 1;
    return cap;
}

// step_kernel (xq_env.cu) after its validation: movePiece + evaluateBoard + checkGameOver + getWinner, the optional reset, the outputs
// (the policy step of xq_policy.cu and the search's play of xq_search.cu)
__device__ __forceinline__ void policy_apply(SmemBoard& b, Meta& m, xq_env_rec* __restrict__ envs, int64_t env, bool ok, int from, int to, int auto_reset,
                                             int32_t* reward, uint8_t* done, uint8_t* winner, uint8_t* captured, uint8_t* valid) {
    const int mover = m.player;
    int cap = 0;
    if (ok) { cap = apply_move(b, m, from, to); m.ctr++; }
    uint32_t wd[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) wd[i] = b.base[i * b.stride];
    const WordSummary s = summarize_words(wd);
    const int diff = mover == RED ? s.mat_red - s.mat_black : s.mat_black - s.mat_red;
    const bool over = m.move_count >= XQ_MAX_MOVES || s.gen_red == 127 || s.gen_black == 127;
    const int win = (s.gen_red == 127 && s.gen_black == 127) ? NOCOLOR : (s.gen_red < s.gen_black ? RED : BLACK);
    if (reward) reward[env] = reward_from_material(diff, m.move_count);
    if (done) done[env] = over ? 1 : 0;
    if (winner) winner[env] = (uint8_t)win;
    if (captured) captured[env] = (uint8_t)cap;
    if (valid) valid[env] = ok ? 1 : 0;
    if (over && auto_reset) { reset_board(b); m.reset(); }
    if (ok || (over && auto_reset)) { b.store(envs + env); m.store(envs + env); }
}

// one warp: whether a search root's 64-byte record is no longer its env's, on every lane.  Lanes 0-3 compare a 16-byte word each and hand
// it back in keep[lane] when keep is given.
__device__ __forceinline__ bool root_stale_warp(const xq_env_rec* root, const xq_env_rec* env, int lane, uint4* keep = nullptr) {
    bool diff = false;
    if (lane < 4) {
        const uint4 rv = reinterpret_cast<const uint4*>(root)[lane], ev = reinterpret_cast<const uint4*>(env)[lane];
        diff = rv.x != ev.x || rv.y != ev.y || rv.z != ev.z || rv.w != ev.w;
        if (keep) keep[lane] = rv;
    }
    return __any_sync(0xFFFFFFFFu, diff);
}


}  // namespace xq
