// TEST-ONLY host build of the multi-leaf selection helpers (cn_chess_ai_b200/csrc/xq_search.cuh), compiled with -ffp-contract=off so
// that the host arithmetic is the device's explicitly rounded one: the virtual-loss score, the plain score it reduces to, and the select
// kernel's per-node in-flight counting.  Never loaded by the product package.
#include <cstdint>

#include "../../cn_chess_ai_b200/csrc/xq_search.cuh"

using namespace xq;

extern "C" {
// Q + U with virtual loss of n edges, c[k] in-flight descents through edge k, c_node through the node
void sl_puct_vl(const float* p, const int32_t* nv, const float* w, const int32_t* c, int n, float vl, float c_puct, float fpu, int n_node,
                int c_node, float* out) {
    const float sq = search_sqrt_visits(n_node + c_node);
    for (int k = 0; k < n; ++k) out[k] = search_puct_vl(p[k], nv[k], w[k], c[k], vl, c_puct, fpu, sq);
}

void sl_puct(const float* p, const int32_t* nv, const float* w, int n, float c_puct, float fpu, int n_node, float* out) {
    const float sq = search_sqrt_visits(n_node);
    for (int k = 0; k < n; ++k) out[k] = search_puct(p[k], nv[k], w[k], c_puct, fpu, sq);
}

// descent k over the edge paths of descents 0 .. k (path[d * 32 + k'], the edge descent k' took at depth d; descent k's own edges in
// column k), `depth` nodes deep: the in-flight counts at every node of its path as the select kernel builds them, counts[d * 128 + e]
// and c_node[d]
void sl_inflight(const uint8_t* path, int k, int depth, int32_t* counts, int32_t* c_node) {
    uint32_t alive = k >= 32 ? 0xFFFFFFFFu : (1u << k) - 1u;
    for (int d = 0; d < depth; ++d) {
        int cj = 0;
        alive = search_inflight_node(alive, path + d * 32, path[d * 32 + k], counts + d * kSearchEdges, &cj);
        c_node[d] = cj;
    }
}
}
