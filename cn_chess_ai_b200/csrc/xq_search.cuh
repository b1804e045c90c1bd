// xq_search.cuh -- host-compilable helpers of the batched tree search (xq_search.cu; include/xq.h: xq_search_*): the PUCT score of an
// edge (with virtual loss: search_puct_vl) and its arg-max order, the in-flight counting of a multi-leaf selection, the priors of a
// freshly expanded node, the root-noise mix, the value cleaning, the backup along a path, and the membership and renumbering of a tree
// re-rooted after a move (xq_search_advance), the visit-count choice of the move to play (xq_search_play_device) and the Dirichlet draw
// of the root noise (xq_search_root_noise_device).
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
// Q + U with virtual loss (xq_search_select_leaves_device): c = the earlier descents of this selection through the edge, vl the virtual
// loss; N' = N + c, W' = c > 0 ? W - vl * c : W, Q = N' > 0 ? W' / N' : fpu, U = ((c_puct * P) * sqrt_n) / (1 + N'), sqrt_n =
// sqrt(N_node + c_node) of the parent.  At c = 0 this is search_puct bit for bit.
XQ_HD float search_puct_vl(float p, int n, float w, int c, float vl, float c_puct, float fpu, float sqrt_n) {
    const int nv = n + c;
    const float wv = c > 0 ? s_add(w, -s_mul(vl, (float)c)) : w;
    const float q = nv > 0 ? s_div(wv, (float)nv) : fpu;
    const float u = s_div(s_mul(s_mul(c_puct, p), sqrt_n), (float)(1 + nv));
    return s_add(q, u);
}
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

// ---- multi-leaf selection: the in-flight counts of descent k (xq_search_select_leaves_device) ----
// The earlier descents k' < k of the selection are lanes of the select-leaves warp.  Each keeps the list index of the edge it took at every
// depth (path[d][k'], d = plies below the root) and an "alive" bit: its path has taken the same edges as descent k so far, i.e. it went
// through descent k's current node (a tree: a node is its edge sequence from the root).  At an expanded, non-terminal node at depth d,
// c_e = the alive lanes whose edge at d is e, and c_node = the alive lanes; an alive lane stays alive if its edge at d is the one descent
// k takes.  Host restatement of the lanes: alive and counts for one node; returns the new alive mask after descent k took edge `taken`.
XQ_HD uint32_t search_inflight_node(uint32_t alive, const uint8_t* path_d, int taken, int32_t* counts, int* c_node) {
    uint32_t next = 0;
    *c_node = 0;
    for (int l = 0; l < 32; ++l) {
        if (!(alive >> l & 1u)) continue;
        counts[path_d[l]] += 1;
        *c_node += 1;
        if (path_d[l] == taken) next |= 1u << l;
    }
    return next;
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

// ---- play: the move from the root's visit counts (xq_search_play_device) ----
// weight of a root edge with n visits, nmax the root's largest count (> 0): n exactly at tau == 1 (every weight and sum an integer below
// 2^24, exact in f32); otherwise exp(log(n / nmax) / tau), 0 for n == 0
XQ_HD float search_play_weight(int n, int nmax, float tau) {
    if (tau == 1.f) return (float)n;
    return n > 0 ? expf(s_div(logf(s_div((float)n, (float)nmax)), tau)) : 0.f;
}
// the sampled edge among n: S = the weights w(k) summed in list order, the first k whose running sum exceeds u * S, else (rounding) the last
// edge with a positive weight; -1 if none has one
template <class W>
XQ_HD int search_play_sample(W&& w, int n, float u) {
    float s = 0.f;
    for (int k = 0; k < n; ++k) s = s_add(s, w(k));
    const float thr = s_mul(u, s);
    float run = 0.f;
    int last = -1;
    for (int k = 0; k < n; ++k) {
        const float x = w(k);
        run = s_add(run, x);
        if (run > thr) return k;
        last = x > 0.f ? k : last;
    }
    return last;
}

// ---- root noise: Dirichlet(alpha) over a root's edges (xq_search_root_noise_device) ----
// Word j of edge k: xq_rng(base, k, j), base = xq_rng(seed, global env id, root ctr).  A uniform from the 24-bit field f at bit `lo` is
// (f + 1) * 2^-24 in (0, 1] (exact in f32, never 0, so every log is finite).  Word 0: the boost uniform Ub (bits 40..63).  Candidate i
// (i = 0 .. 31): word 1 + 2i gives a Box-Muller normal z = sqrt(-2 log u1) * cos(2 pi u2) (u1 bits 40..63, u2 bits 16..39), word 2 + 2i the
// acceptance uniform Ua (bits 40..63).  Marsaglia-Tsang at shape a = alpha + 1: d = a - 1/3, c = 1 / sqrt(9 d), v = (1 + c z)^3, accepted
// when v > 0 and log Ua < ((0.5 z^2 + d) - d v) + d log v.  After 32 rejected candidates the last one with v > 0 is used (v = 1 if none
// had); at a rejection rate below 5 % per candidate this never happens in practice.  Gamma(alpha) = d v Ub^(1 / alpha), kept in log space.
constexpr int kGammaTries = 32;
XQ_HD float search_u24(uint64_t x, int lo) { return s_mul(s_add((float)((uint32_t)(x >> lo) & 0xFFFFFFu), 1.f), 5.9604644775390625e-8f); }
// log of the Gamma(alpha) draw of edge k: log(d v) + log(Ub) / alpha
XQ_HD float search_log_gamma(uint64_t base, int k, float alpha) {
    const float d = s_add(s_add(alpha, 1.f), -1.f / 3.f);
    const float c = s_div(1.f, s_sqrt(s_mul(9.f, d)));
    float v = 1.f;
    for (int i = 0; i < kGammaTries; ++i) {
        const uint64_t xn = rng(base, (uint64_t)k, (uint32_t)(1 + 2 * i));
        const float z = s_mul(s_sqrt(s_mul(-2.f, logf(search_u24(xn, 40)))), cosf(s_mul(6.28318548f, search_u24(xn, 16))));
        const float t = s_add(1.f, s_mul(c, z));
        const float cand = s_mul(s_mul(t, t), t);
        if (!(cand > 0.f)) continue;
        v = cand;
        const float ua = search_u24(rng(base, (uint64_t)k, (uint32_t)(2 + 2 * i)), 40);
        if (logf(ua) < s_add(s_add(s_add(s_mul(0.5f, s_mul(z, z)), d), -s_mul(d, v)), s_mul(d, logf(v)))) break;
    }
    return s_add(logf(s_mul(d, v)), s_div(logf(search_u24(rng(base, (uint64_t)k, 0u), 40)), alpha));
}
// exp(lg - m) of one edge, m the largest lg of the root (all -inf: 1 for every edge, so that eta stays defined)
XQ_HD float search_noise_exp(float lg, float m) { return m == -INFINITY ? 1.f : expf(s_add(lg, -m)); }
// eta[0 .. n) of one root (n >= 1): eta_k = exp(lg_k - max) / S, S summed in list order.  Host restatement of the noise kernel.
XQ_HD void search_dirichlet(uint64_t base, int n, float alpha, float* eta) {
    float m = -INFINITY;
    for (int k = 0; k < n; ++k) { eta[k] = search_log_gamma(base, k, alpha); m = fmaxf(m, eta[k]); }
    float s = 0.f;
    for (int k = 0; k < n; ++k) { eta[k] = search_noise_exp(eta[k], m); s = s_add(s, eta[k]); }
    for (int k = 0; k < n; ++k) eta[k] = s_div(eta[k], s);
}

}  // namespace xq
