// TEST-ONLY host build of the tree-search helpers (cn_chess_ai_b200/csrc/xq_search.cuh), compiled with -ffp-contract=off so that the
// host arithmetic is the device's explicitly rounded one: PUCT scores, the selection order (sequentially and as the select kernel's
// 32-lane warp reduction), the priors of an expansion, the root-noise mix and the backup.  Never loaded by the product package.
#include <cstdint>

#include "../../cn_chess_ai_b200/csrc/xq_search.cuh"

using namespace xq;

extern "C" {
// Q + U of n edges of a node visited n_node times
void ss_puct(const float* p, const int32_t* nv, const float* w, int n, float c_puct, float fpu, int n_node, float* out) {
    const float sq = search_sqrt_visits(n_node);
    for (int k = 0; k < n; ++k) out[k] = search_puct(p[k], nv[k], w[k], c_puct, fpu, sq);
}

// the selected edge: lanes take k = lane, lane + 32, ... in order, then a butterfly over the 32 lanes (search_select_kernel)
int ss_select_warp(const float* p, const int32_t* nv, const float* w, int n, float c_puct, float fpu, int n_node) {
    const float sq = search_sqrt_visits(n_node);
    float bs[32];
    int bk[32];
    for (int lane = 0; lane < 32; ++lane) {
        bs[lane] = 0.f; bk[lane] = -1;
        for (int k = lane; k < n; k += 32) {
            const float v = search_puct(p[k], nv[k], w[k], c_puct, fpu, sq);
            if (search_better(v, k, bs[lane], bk[lane])) { bs[lane] = v; bk[lane] = k; }
        }
    }
    for (int off = 16; off > 0; off >>= 1) {
        float ns[32];
        int nk[32];
        for (int lane = 0; lane < 32; ++lane) {
            const int o = lane ^ off;
            ns[lane] = bs[lane]; nk[lane] = bk[lane];
            if (bk[o] >= 0 && search_better(bs[o], bk[o], bs[lane], bk[lane])) { ns[lane] = bs[o]; nk[lane] = bk[o]; }
        }
        for (int lane = 0; lane < 32; ++lane) { bs[lane] = ns[lane]; bk[lane] = nk[lane]; }
    }
    return bk[0];
}

// priors of one node from the raw scores of its n legal actions in list order (cleaned as the kernels clean them); noise (may be null):
// the root's mix with noise[k]
void ss_priors(const float* raw, int n, float t, const float* noise, float eps, float* out) {
    auto each = [&](auto&& f) { for (int k = 0; k < n; ++k) f(policy_clean(raw[k])); };
    PolicyBest best{-INFINITY, -1};
    int i = 0;
    each([&](float l) { best.offer(l, i++); });
    search_priors(each, n, best.m, t, [&](int k, float p) { out[k] = noise ? search_mix(p, noise[k], eps) : p; });
}

float ss_clean_value(float v) { return search_clean_value(v); }

void ss_backup(int leaf, float value, const int32_t* parent, const uint8_t* parent_edge, int32_t* node_visits, int32_t* edge_n, float* edge_w) {
    search_backup(leaf, value, parent, parent_edge, node_visits, edge_n, edge_w);
}
}
