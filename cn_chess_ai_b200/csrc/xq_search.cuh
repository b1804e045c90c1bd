// xq_search.cuh -- host-compilable helpers of the batched tree search (xq_search.cu; include/xq.h: xq_search_*): the PUCT score of an
// edge and its arg-max order, the priors of a freshly expanded node, the root-noise mix, the value cleaning, the backup along a path, and
// the membership and renumbering of a tree re-rooted after a move (xq_search_advance).
//
// The arithmetic is spelled with explicitly rounded operations (__fmul_rn and friends on the device; plain operators on the host, where
// tests/hostsim/search_shim.cpp is compiled with -ffp-contract=off) so that no multiply-add is contracted and numpy can restate every
// score bit for bit.
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "xq_bitboard.cuh"
#include "xq_policy.cuh"

namespace xq {

constexpr int kSearchEdges = XQ_MAX_ACTIONS;      // edge slots per node: the first 128 actions in list order

XQ_HD float s_add(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
XQ_HD float s_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
XQ_HD float s_div(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}
XQ_HD float s_sqrt(float a) {
#if defined(__CUDA_ARCH__)
    return __fsqrt_rn(a);
#else
    return sqrtf(a);
#endif
}

// Q + U of one edge: Q = N > 0 ? W / N : fpu, U = ((c_puct * P) * sqrt_n) / (1 + N), sqrt_n = sqrt(N_node) of the parent
XQ_HD float search_puct(float p, int n, float w, float c_puct, float fpu, float sqrt_n) {
    const float q = n > 0 ? s_div(w, (float)n) : fpu;
    const float u = s_div(s_mul(s_mul(c_puct, p), sqrt_n), (float)(1 + n));
    return s_add(q, u);
}
XQ_HD float search_sqrt_visits(int n_node) { return s_sqrt((float)n_node); }
// the arg-max order of selection: a larger score, or an equal one at a smaller list index (strict >, DQN::selectAction)
XQ_HD bool search_better(float a, int ia, float b, int ib) { return ib < 0 || a > b || (a == b && ia < ib); }

// Priors of a node from the cleaned scores of its legal actions: P_k = exp((l_k - m) / t) / S, S summed in list order -- the arithmetic
// of policy_choose's sum.  each(f) calls f(l) in list order; m = the maximum (PolicyBest); every score -inf: 1 / n.  out(k, P_k).
template <class EACH, class OUT>
XQ_HD void search_priors(EACH&& each, int n, float m, float t, OUT&& out) {
    if (n <= 0) return;
    if (m == -INFINITY) {
        for (int k = 0; k < n; ++k) out(k, 1.f / (float)n);
        return;
    }
    float s = 0.f;
    each([&](float l) { s += expf((l - m) / t); });
    int k = 0;
    each([&](float l) { out(k, expf((l - m) / t) / s); ++k; });
}
// the root's Dirichlet mix: (1 - eps) * P + eps * noise
XQ_HD float search_mix(float p, float noise, float eps) { return s_add(s_mul(s_add(1.f, -eps), p), s_mul(eps, noise)); }

// the caller's value: NaN -> 0, then clamped to [-1, 1]
XQ_HD float search_clean_value(float v) { return v != v ? 0.f : (v < -1.f ? -1.f : (v > 1.f ? 1.f : v)); }

// Backup of one simulation in one tree (node-local indices): the leaf's value v is from its side to move; walking up, v <- -v, the edge
// from the parent gets N += 1 and W += v, every node on the path (leaf and root included) N_node += 1.  Edges of node j at j * 128 + e.
XQ_HD void search_backup(int leaf, float value, const int32_t* parent, const uint8_t* parent_edge, int32_t* node_visits, int32_t* edge_n,
                         float* edge_w) {
    float v = search_clean_value(value);
    int j = leaf;
    node_visits[j] += 1;
    while (j > 0) {
        const int p = parent[j];
        const int64_t e = (int64_t)p * kSearchEdges + parent_edge[j];
        v = -v;
        edge_n[e] += 1;
        edge_w[e] = s_add(edge_w[e], v);
        node_visits[p] += 1;
        j = p;
    }
}

// ---- advance: re-rooting a tree at node m (0, or a child of the root) in place ----
// Membership: keep[j] = j == m || (j > m && keep[parent[j]]), decidable in increasing index order because parent[j] < j.  It is held as a
// bitmap of 32-node words with a prefix count per word (prefix[w] = kept nodes in words < w); a kept node's new index is
// prefix[j >> 5] + the kept nodes below it in its word, never larger than j, so moving the kept nodes in increasing old index (each batch
// read completely before it is written) overwrites only slots already read.

// node j of the word that starts at `base`, its parent p: the parent's bit from `bits` (an earlier word, complete) or from `word` (this
// word as far as it is known; iterated to its fixed point by search_keep_word)
XQ_HD bool search_kept(int j, int m, int p, int base, const uint32_t* bits, uint32_t word) {
    if (j == m) return true;
    if (j < m || p < m) return false;
    const uint32_t w = p >= base ? word >> (p - base) : bits[p >> 5] >> (p & 31);
    return (w & 1u) != 0;
}

// the kept bits of nodes base .. base + 31 (< count) as the advance kernel's warp finds them: every lane evaluates search_kept against
// the word of the last round (a ballot) until the word stops changing.  keep only grows and parents come first, so this ends at the
// membership itself after at most 33 rounds.  Host restatement of the lanes for the CPU suite.
XQ_HD uint32_t search_keep_word(int base, int count, int m, const int32_t* parent, const uint32_t* bits) {
    uint32_t word = 0;
    for (;;) {
        uint32_t next = 0;
        for (int l = 0; l < 32; ++l) {
            const int j = base + l;
            if (j < count && search_kept(j, m, parent[j], base, bits, word)) next |= 1u << l;
        }
        if (next == word) return word;
        word = next;
    }
}

// bits and prefix of words (m >> 5) .. (count - 1) >> 5 (the words below hold no kept node and are not written); returns the kept count
XQ_HD int search_membership(int count, int m, const int32_t* parent, uint32_t* bits, int32_t* prefix) {
    int kept = 0;
    for (int w = m >> 5; w <= (count - 1) >> 5; ++w) {
        bits[w] = search_keep_word(w << 5, count, m, parent, bits);
        prefix[w] = kept;
        kept += popc32(bits[w]);
    }
    return kept;
}

// the new index of kept node j
XQ_HD int search_new_index(const uint32_t* bits, const int32_t* prefix, int j) {
    return prefix[j >> 5] + popc32(bits[j >> 5] & ((1u << (j & 31)) - 1u));
}

}  // namespace xq
