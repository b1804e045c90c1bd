// xq_examples.cuh -- host-compilable helpers of the self-play example buffer (xq_examples.cu; include/xq.h: xq_examples_*): the game
// result and its sign per example, the policy target of one edge, the view of a stored action, the sample-index draw, the commit
// offsets of the ended envs' staged examples, and the status rule of a reanalyse refresh.
//
// tests/hostsim/examples_shim.cpp compiles this header with -ffp-contract=off so that numpy restates every value bit for bit.
#pragma once
#include <stdint.h>

#include "xq_search.cuh"

namespace xq {

constexpr int kExampleBytes = 864;
constexpr int kExampleVecs = kExampleBytes / 16;      // 16-byte words of one example

// the caller's result (Red's side) as the search backup cleans values: NaN -> 0, then clamped to [-1, 1]
XQ_HD float ex_result(float result_red) { return search_clean_value(result_red); }
// z of an example whose record has `player` to move: the cleaned result if Red is to move, its negation otherwise
XQ_HD float ex_z(float result_red, int player) {
    const float r = ex_result(result_red);
    return player == RED ? r : -r;
}
// the policy target of an edge: visits / total as one f32 division of the two counts converted to f32; 0 when the root has no visit
XQ_HD float ex_policy(uint32_t visits, uint32_t total) { return total ? s_div((float)visits, (float)total) : 0.f; }
// policy index of an absolute stored action (from * 90 + to) in the frame of `view` for a record with `player` to move
XQ_HD int ex_view_index(int action, int player, int view) { return policy_flip(player, view) ? XQ_POLICY_ACTIONS - 1 - action : action; }
// ring slot of sample i (xq_replay_sample's rule); -1 for an empty ring
XQ_HD int64_t ex_sample_index(uint64_t seed, int64_t i, uint32_t counter, int64_t size) {
    return size > 0 ? (int64_t)((rng(seed, (uint64_t)i, counter) >> 1) % (uint64_t)size) : -1;
}

// ---- commit offsets ----
// The commit kernel runs one CTA of `threads` threads; thread t owns the contiguous envs [lo, hi) of ex_segment and sums their counts
// (ended ? staged : 0); the segment sums are scanned exclusively across the threads, and each thread then writes its envs' offsets in env
// order.  off[e] = base + the counts of the ended envs below e: the commit number of env e's first example.
XQ_HD void ex_segment(int64_t n, int threads, int t, int64_t& lo, int64_t& hi) {
    const int64_t per = (n + threads - 1) / threads;
    lo = (int64_t)t * per < n ? (int64_t)t * per : n;
    hi = lo + per < n ? lo + per : n;
}
XQ_HD uint32_t ex_count(uint8_t ended, uint32_t staged) { return ended ? staged : 0u; }

// host restatement of the kernel's three phases for the CPU suite; returns the total committed
inline int64_t ex_commit_offsets(int64_t n, int threads, const uint8_t* ended, const uint32_t* staged, int64_t base, int64_t* off) {
    int64_t run = base;
    for (int t = 0; t < threads; ++t) {         // the exclusive scan of the segment sums is the running total in thread order
        int64_t lo, hi;
        ex_segment(n, threads, t, lo, hi);
        for (int64_t e = lo; e < hi; ++e) { off[e] = run; run += ex_count(ended[e], staged[e]); }
    }
    return run - base;
}

// the ended env holding commit number pos: the last env e with off[e] <= pos (envs without examples share their successor's offset, and
// the last of a run of equal offsets is the one that has examples)
XQ_HD int64_t ex_find_env(const int64_t* off, int64_t n, int64_t pos) {
    int64_t lo = 0, hi = n;                     // first e with off[e] > pos, in [lo, hi]
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (off[mid] <= pos) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

// ---- reanalyse (xq_examples_refresh_device) ----
constexpr uint32_t kNoClaim = 0xFFFFFFFFu;      // a slot's claim word outside a refresh call
// whether ring slot idx holds a committed example (size = committed examples held)
XQ_HD bool ex_slot_held(int64_t idx, int64_t size) { return idx >= 0 && idx < size; }
// the status of row t, which refreshes slot idx: claim = the slot's claim word once every row of the call has claimed it (the smallest
// row whose index is idx), stale = the slot's record differs from the root's, total = the root's visits (or weights) summed.  The checks
// run in this order: NO_SLOT, DUPLICATE, STALE, UNSEARCHED; a row that passes all of them is REFRESHED (include/xq.h: XQ_REFRESH*).
XQ_HD uint8_t ex_refresh_status(int64_t idx, int64_t size, uint32_t claim, uint32_t t, bool stale, uint32_t total) {
    if (!ex_slot_held(idx, size)) return XQ_REFRESH_NO_SLOT;
    if (claim != t) return XQ_REFRESH_DUPLICATE;
    if (stale) return XQ_REFRESH_STALE;
    return total ? XQ_REFRESHED : XQ_REFRESH_UNSEARCHED;
}

// host restatement of the claim and refresh kernels for the CPU suite: every row claims its slot with the smallest row (atomicMin over
// claim[], kNoClaim on entry), each row takes its status, and the winner of a slot restores its claim word
inline void ex_refresh_statuses(int64_t m, const int64_t* index, int64_t size, const uint8_t* stale, const uint32_t* total, uint32_t* claim,
                                uint8_t* status) {
    for (int64_t t = 0; t < m; ++t)
        if (ex_slot_held(index[t], size) && (uint32_t)t < claim[index[t]]) claim[index[t]] = (uint32_t)t;
    for (int64_t t = 0; t < m; ++t) {
        const int64_t idx = index[t];
        const bool held = ex_slot_held(idx, size);
        const uint32_t c = held ? claim[idx] : kNoClaim;
        status[t] = ex_refresh_status(idx, size, c, (uint32_t)t, stale[t] != 0, total[t]);
        if (held && c == (uint32_t)t) claim[idx] = kNoClaim;
    }
}

}  // namespace xq
