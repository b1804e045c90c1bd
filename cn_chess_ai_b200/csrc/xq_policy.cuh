// xq_policy.cuh -- device helpers of the external-policy interface (xq_policy.cu; include/xq.h: xq_env_observe_device,
// xq_env_legal_mask_device, xq_env_policy_step_device): policy indices and views, the register-resident generator of one board, and
// the choice of an action from a policy's scores (greedy, sampled, given).
//
// Host-compilable: tests/hostsim/policy_shim.cpp runs the same functions board by board against the oracle before any GPU time.
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "../../include/xq.h"
#include "xq_rollout_lane.cuh"

namespace xq {

// a player byte other than 0 / 1 has no pieces of its colour (ChessAI::getAllValidActions compares colours): the view leaves it alone
XQ_HD bool policy_flip(int player, int view) { return view == XQ_VIEW_SIDE_TO_MOVE && player == BLACK; }
// policy index of the absolute action (from, to) in the frame of the view (flip: rotated by 180 degrees, s -> 89 - s)
XQ_HD int policy_index(int from, int to, bool flip) { return flip ? (89 - from) * 90 + (89 - to) : from * 90 + to; }
// NaN never wins (it counts as -inf); +inf is clamped so that a softmax over it stays defined
XQ_HD float policy_clean(float v) { return v != v ? -INFINITY : (v > FLT_MAX ? FLT_MAX : v); }
// bf16 -> f32 is exact: the 16 bits are the high half of the f32
XQ_HD float bf16_bits_to_float(uint16_t b) {
    const uint32_t u = (uint32_t)b << 16;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}

// The legal actions of one board through the register-resident generator of the list kernel (legal_moves_lane_kernel): unpack the record
// words into the piece slots (slot[32 * stride], [slot][thread]) and the thread's view memory (vm, kViewWords words at `stride`), then
// lane_movegen.  false: the board goes to the generic kernel (a non-standard piece set, or a player byte > 1 -- the geometry table is
// indexed by colour and has two entries).
struct LaneGen {
    uint32_t own_sq[4], sdesc[4], cw[4], dw[4];
};
XQ_HD bool policy_lane_gen(const uint32_t (&w)[12], int player, uint32_t* vm, uint8_t* slot, int stride, const uint32_t* geo, LaneGen& g) {
    if ((unsigned)player > 1u) return false;
    for (int i = 0; i < 32; ++i) slot[i * stride] = kDeadSq;
    Bits90 red, black, occT;
    if (!team_unpack_record_m(w, vm, stride, red, black, occT, [&](int s, int q) { slot[s * stride] = (uint8_t)q; })) return false;
#pragma unroll
    for (int i = 0; i < 4; ++i) g.own_sq[i] = 0;
#pragma unroll
    for (int pos = 0; pos < 16; ++pos) g.own_sq[pos >> 2] |= (uint32_t)slot[((player ? 16 : 0) + lane_pos_slot(pos)) * stride] << (8 * (pos & 3));
    view_init(vm, stride);
    view_store(vm, stride, player ? black : red, player ? red : black, occT);
    lane_movegen(g.own_sq, MemView{vm, stride}, player, geo, g.sdesc, g.cw, g.dw);
    return true;
}
// f(list index, from, to) for every legal action, in slot order (lane_emit_actions); returns the list size
template <class F>
XQ_HD int policy_lane_emit(const LaneGen& g, int player, F&& f) {
    return lane_emit_actions(g.own_sq, player, g.sdesc, g.cw, g.dw, [&](int idx, int a, bool live) { if (live) f(idx, (int)XQ_ACTION_FROM(a), (int)XQ_ACTION_TO(a)); });
}

// The first maximum in list order, fed in any order: a larger score, or an equal one at a smaller list index
struct PolicyBest {
    float m;
    int k;
    XQ_HD void offer(float v, int idx) {
        const bool take = k < 0 || v > m || (v == m && idx < k);
        m = take ? v : m; k = take ? idx : k;
    }
};

struct PolicyChoice {
    int k;         // list index of the played action, -1 = none
    float logp;    // NaN where not defined
};
// The choice among the n legal actions.  each(f) calls f(l) with the cleaned score of every legal action in reference list order (it is
// only called when scores exist); best = PolicyBest over the same scores; given_k = list index of the given action (-1: rejected);
// u = the uniform draw of SAMPLE; want_logp: compute logp (GREEDY / GIVEN skip the sums without it).  GREEDY = best.k; SAMPLE = the first
// k whose running sum of exp((l - m) / t) exceeds u * S; logp of the played action = (l_k - m) / t - log S.  A board whose every score is
// -inf plays its first action and has no logp.
template <class EACH>
XQ_HD PolicyChoice policy_choose(EACH&& each, int n, const PolicyBest& best, int given_k, int pick, bool scores, bool want_logp, float t, float u) {
    PolicyChoice c{-1, NAN};
    if (n == 0) return c;
    c.k = pick == XQ_PICK_GIVEN ? given_k : (pick == XQ_PICK_GREEDY ? best.k : 0);
    if (!scores || c.k < 0 || best.m == -INFINITY || (pick != XQ_PICK_SAMPLE && !want_logp)) return c;
    const float m = best.m;
    float s = 0.f, lk = m;
    int i = 0;
    each([&](float l) {
        s += expf((l - m) / t);
        lk = i == c.k ? l : lk;
        ++i;
    });
    if (pick == XQ_PICK_SAMPLE) {
        const float thr = u * s;
        float run = 0.f, last = m;
        int pk = -1;
        i = 0;
        each([&](float l) {
            run += expf((l - m) / t);
            const bool hit = pk < 0 && run > thr;
            pk = hit ? i : pk; lk = hit ? l : lk; last = l;
            ++i;
        });
        if (pk < 0) { pk = n - 1; lk = last; }
        c.k = pk;
    }
    c.logp = (lk - m) / t - logf(s);
    return c;
}
// u of SAMPLE: 24 high bits of the env's draw
XQ_HD float policy_uniform(uint64_t x) { return (float)(uint32_t)(x >> 40) * 5.9604644775390625e-8f; }

}  // namespace xq
