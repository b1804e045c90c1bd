// xq_search.cuh -- host-compilable helpers of the batched tree search (xq_search.cu; include/xq.h: xq_search_*): the PUCT score of an
// edge and its arg-max order, the priors of a freshly expanded node, the root-noise mix, the value cleaning and the backup along a path.
//
// The arithmetic is spelled with explicitly rounded operations (__fmul_rn and friends on the device; plain operators on the host, where
// tests/hostsim/search_shim.cpp is compiled with -ffp-contract=off) so that no multiply-add is contracted and numpy can restate every
// score bit for bit.
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>

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

}  // namespace xq
