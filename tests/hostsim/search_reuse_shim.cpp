// TEST-ONLY host build of the re-rooting helpers of the tree search (cn_chess_ai_b200/csrc/xq_search.cuh, xq_search_advance), compiled
// with -ffp-contract=off like search_shim.cpp: the membership bitmap and prefix counts, the new indices, and the in-place move of
// search_advance_kernel (kept nodes in increasing old index, a batch of nodes read completely before it is written), node arrays and
// edge rows included, with the root-noise mix.  Never loaded by the product package.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../cn_chess_ai_b200/csrc/xq_search.cuh"

using namespace xq;

extern "C" {
// bits / prefix [(count + 31) / 32] (words below m >> 5 zeroed); returns the kept count
int sr_membership(int count, int m, const int32_t* parent, uint32_t* bits, int32_t* prefix) {
    const int words = (count + 31) >> 5;
    memset(bits, 0, 4 * (size_t)words);
    memset(prefix, 0, 4 * (size_t)words);
    return search_membership(count, m, parent, bits, prefix);
}

int sr_new_index(const uint32_t* bits, const int32_t* prefix, int j) { return search_new_index(bits, prefix, j); }

// The kernel's step 4 on one tree of `count` nodes with edge rows of 128 slots, in place, `batch` nodes per round: each round reads its
// nodes' fields and edge rows completely, then writes them to their new slots.  order[r] = the old index of the r-th node read (the
// caller checks the order and that no slot is written before it is read).  m > 0; noise (may be null) indexed by the action, [8100].
// Returns the number of nodes moved.
int sr_move(int count, int m, int batch, int32_t* parent, uint8_t* pedge, int32_t* visits, int32_t* reward, int32_t* depth, uint8_t* nedges,
            uint8_t* expanded, float* P, int32_t* N, float* W, int32_t* child, int16_t* act, const float* noise, float eps, int32_t* order) {
    const int words = (count + 31) >> 5;
    std::vector<uint32_t> bits(words, 0u);
    std::vector<int32_t> prefix(words, 0);
    search_membership(count, m, parent, bits.data(), prefix.data());
    const int dm = depth[m];
    int moved = 0;
    int w = m >> 5;
    uint32_t rest = bits[w];
    const int last = (count - 1) >> 5;
    struct Node { int j, parent, visits, reward, depth; uint8_t pedge, nedges, expanded; float P[kSearchEdges], W[kSearchEdges];
                  int32_t N[kSearchEdges], C[kSearchEdges]; int16_t A[kSearchEdges]; };
    std::vector<Node> nb(batch);
    for (;;) {
        int got = 0;
        for (int b = 0; b < batch; ++b) {
            while (rest == 0 && w < last) rest = bits[++w];
            nb[b].j = rest ? (w << 5) + ffs32(rest) - 1 : -1;
            rest &= rest - 1;
            got += nb[b].j >= 0;
        }
        if (!got) break;
        for (int b = 0; b < batch; ++b) {
            Node& x = nb[b];
            if (x.j < 0) continue;
            order[moved++] = x.j;
            x.parent = parent[x.j]; x.visits = visits[x.j]; x.reward = reward[x.j]; x.depth = depth[x.j];
            x.pedge = pedge[x.j]; x.nedges = nedges[x.j]; x.expanded = expanded[x.j];
            const int ne = x.expanded ? x.nedges : 0;
            for (int k = 0; k < ne; ++k) {
                const int64_t e = (int64_t)x.j * kSearchEdges + k;
                x.P[k] = P[e]; x.N[k] = N[e]; x.W[k] = W[e]; x.C[k] = child[e]; x.A[k] = act[e];
            }
        }
        for (int b = 0; b < batch; ++b) {
            const Node& x = nb[b];
            if (x.j < 0) continue;
            const bool root = x.j == m;
            const int g = search_new_index(bits.data(), prefix.data(), x.j);
            parent[g] = root ? -1 : search_new_index(bits.data(), prefix.data(), x.parent);
            pedge[g] = root ? 0 : x.pedge;
            visits[g] = x.visits; reward[g] = root ? 0 : x.reward; depth[g] = x.depth - dm;
            nedges[g] = x.nedges; expanded[g] = x.expanded;
            const int ne = x.expanded ? x.nedges : 0;
            for (int k = 0; k < ne; ++k) {
                const int64_t e = (int64_t)g * kSearchEdges + k;
                P[e] = root && noise ? search_mix(x.P[k], noise[x.A[k]], eps) : x.P[k];
                N[e] = x.N[k]; W[e] = x.W[k]; act[e] = x.A[k];
                child[e] = x.C[k] >= 0 ? search_new_index(bits.data(), prefix.data(), x.C[k]) : -1;
            }
        }
    }
    return moved;
}

float sr_mix(float p, float noise, float eps) { return search_mix(p, noise, eps); }
}
