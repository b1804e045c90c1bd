// xq_search.cu -- device-resident batched tree search for an external policy/value network: one PUCT tree per env of an env handle
// (include/xq.h: xq_search_*).  Between two network calls everything stays on the device.
//
// Layout (one slab of cap = max_simulations + 1 nodes per tree, node j of tree t at g = t * cap + j; helpers in xq_search.cuh):
//   nodes, structure of arrays over g: the board (xq_env_rec), parent, parent edge, N_node, reward and depth, edge count, expanded flag,
//     terminal status (0 / 1 General captured / 2 move cap / 3 no legal action) and winner;
//   edges, structure of arrays over g * 128 + k (k = reference list index): prior P, visit count N, value sum W, child node (-1 none),
//     action from * 90 + to (absolute).  A warp reads the P / N / W / child of one node with coalesced loads.
// search_select_kernel: one warp per tree, PUCT arg-max as a warp reduction keyed (score, -index); a new child is made with apply_move +
//   summarize_words on the nibble board, as policy_apply does; the leaf record goes to the leaf buffer.
// search_expand_lane_kernel: one thread per tree, the structure of policy_step_lane_kernel: the generator stages the legal scores into
//   a [list index][thread] shared row, the priors are taken over that row in list order, the backup walks the parent pointers.
//   Boards the generator refuses go to search_expand_generic_kernel (all_actions, thread per board).
// search_select_leaves_kernel: one warp per tree, the L descents of a multi-leaf selection in order with virtual loss (in-flight counts
//   from the earlier descents' edges, kept per depth in shared memory); search_expand_slots_kernel / search_expand_generic_slots_kernel:
//   one thread per (tree, slot) for the expansions, the backups of a tree in slot order by the thread of its slot 0.
// search_root_kernel: one CTA per tree, the dense visit row built in shared memory and written with 16-byte stores.
// search_advance_kernel: one warp per tree, re-roots the tree at the played child in place (membership bitmap in shared memory).
// search_play_kernel: one warp per tree, the move from the root's visit counts and the env's step with it.
// search_noise_kernel: one warp per tree, Dirichlet noise drawn over the root's edges and mixed into its priors.
#include <string.h>

#include <new>
#include <vector>

#include "xq_common.cuh"
#include "xq_env_dev.cuh"
#include "xq_bitboard.cuh"
#include "xq_search.cuh"

namespace xq {

cudaError_t launch_observe(const xq_env_rec* recs, int64_t n, void* planes, int dtype, int view, int32_t* aux, cudaStream_t stream);

constexpr int kSelWarps = 4;       // trees per CTA of the select kernel
constexpr int kExpBoards = 32;     // trees per CTA of the lane expand kernel
constexpr int kRootThreads = 256;

struct SearchDev {
    int64_t n; int cap;
    xq_env_rec* rec;
    int32_t *parent, *visits, *reward, *depth;
    uint8_t *pedge, *nedges, *expanded, *term, *winner;
    float *P, *W; int32_t *N, *child; int16_t* act;
    int32_t *count, *leaf; xq_env_rec* leaf_rec; uint8_t* nonstd;
};

// status of a board that a step has produced: a General missing (1) before the move cap (2), the order of xq_game_event.reason;
// winner = getWinner (the first General in square order), as policy_apply reports it
__device__ __forceinline__ void search_status(const WordSummary& s, int move_count, uint8_t& term, uint8_t& winner) {
    term = (s.gen_red == 127 || s.gen_black == 127) ? 1 : (move_count >= XQ_MAX_MOVES ? 2 : 0);
    winner = (uint8_t)((s.gen_red == 127 && s.gen_black == 127) ? NOCOLOR : (s.gen_red < s.gen_black ? RED : BLACK));
}

// tree t emptied down to a root holding the env's record `env` (xq_search_reset; xq_search_advance for a tree it does not keep)
__device__ __forceinline__ void search_reset_tree(const SearchDev& d, int64_t t, const xq_env_rec* env) {
    const int64_t g = t * d.cap;
    const uint4* src = reinterpret_cast<const uint4*>(env);
    uint4* dst = reinterpret_cast<uint4*>(d.rec + g);
    uint32_t wd[12];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint4 v = src[i];
        dst[i] = v;
        if (i < 3) { wd[4 * i] = v.x; wd[4 * i + 1] = v.y; wd[4 * i + 2] = v.z; wd[4 * i + 3] = v.w; }
    }
    Meta m; m.load(env);
    uint8_t term, win;
    search_status(summarize_words(wd), m.move_count, term, win);
    d.parent[g] = -1; d.pedge[g] = 0; d.visits[g] = 0; d.reward[g] = 0; d.depth[g] = 0;
    d.nedges[g] = 0; d.expanded[g] = 0; d.term[g] = term; d.winner[g] = win;
    d.count[t] = 1;
}

__global__ void __launch_bounds__(256) search_reset_kernel(SearchDev d, const xq_env_rec* __restrict__ envs) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.n) return;
    search_reset_tree(d, t, envs + t);
}

// Re-rooting at the env's record (xq_search_advance), one warp per tree:
//   1. the match m: the root, else the root's child whose 64-byte record equals the env's (the lanes split the children);
//   2. m > 0: the membership bitmap and per-word prefix counts in shared memory (search_kept / search_membership of xq_search.cuh), one
//      32-node word per round, each word a ballot iterated to its fixed point;
//   3. no match, or more than cap - min_free kept nodes: the tree is rebuilt as search_reset_kernel builds it;
//   4. m > 0: the kept nodes move to their new slots kAdvBatch at a time in increasing old index, the whole batch read before any of it
//      is written (new index <= old index, so only slots already read are overwritten); the lanes split a node's edge slots.  Parents and
//      children are renumbered through the bitmap, depths lowered by m's; m becomes the root.  The root noise is mixed into a kept,
//      expanded root's priors (in place when m == 0).
constexpr int kAdvWarps = 4;       // trees per CTA of the advance kernel
constexpr int kAdvBatch = 2;       // nodes a warp moves per round
constexpr int kAdvSlots = kSearchEdges / 32;

__global__ void __launch_bounds__(32 * kAdvWarps) search_advance_kernel(SearchDev d, const xq_env_rec* __restrict__ envs, int min_free,
                                                                       const float* __restrict__ noise, float eps, int view,
                                                                       int32_t* __restrict__ kept_out) {
    extern __shared__ uint32_t s_adv[];          // per warp: bits[words], then prefix[words]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * kAdvWarps + warp;
    if (t >= d.n) return;
    const int words = (d.cap + 31) >> 5;
    uint32_t* bits = s_adv + (size_t)warp * 2 * words;
    int32_t* prefix = reinterpret_cast<int32_t*>(bits + words);
    const int64_t g0 = t * d.cap, eb0 = g0 * kSearchEdges;
    const int count = d.count[t];
    uint4 e[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) e[i] = reinterpret_cast<const uint4*>(envs + t)[i];
    auto same = [&](int64_t g) {
        const uint4* r = reinterpret_cast<const uint4*>(d.rec + g);
        bool eq = true;
#pragma unroll
        for (int i = 0; i < 4; ++i) { const uint4 v = r[i]; eq = eq && v.x == e[i].x && v.y == e[i].y && v.z == e[i].z && v.w == e[i].w; }
        return eq;
    };
    // 1. the match
    int m = -1;
    if (same(g0)) {
        m = 0;
    } else if (d.expanded[g0]) {
        const int ne = d.nedges[g0];
        unsigned cand = 0xFFFFFFFFu;
        for (int k = lane; k < ne; k += 32) {
            const int c = d.child[eb0 + k];
            if (c >= 0 && (unsigned)c < cand && same(g0 + c)) cand = (unsigned)c;
        }
        cand = __reduce_min_sync(0xFFFFFFFFu, cand);
        if (cand != 0xFFFFFFFFu) m = (int)cand;
    }
    // 2. the membership
    int kept = count;
    const int last = (count - 1) >> 5;
    if (m > 0) {
        kept = 0;
        for (int w = m >> 5; w <= last; ++w) {
            const int base = w << 5, j = base + lane;
            const int p = j < count ? d.parent[g0 + j] : -1;
            uint32_t word = 0;
            for (;;) {
                const uint32_t next = __ballot_sync(0xFFFFFFFFu, j < count && search_kept(j, m, p, base, bits, word));
                if (next == word) break;
                word = next;
            }
            if (lane == 0) { bits[w] = word; prefix[w] = kept; }
            kept += popc32(word);
            __syncwarp();
        }
    }
    // 3. a tree that is not kept
    if (m < 0 || kept > d.cap - min_free) {
        if (lane == 0) {
            search_reset_tree(d, t, envs + t);
            if (kept_out) kept_out[t] = 0;
        }
        return;
    }
    // 4. the move, and the root noise
    const float* nz = noise ? noise + t * XQ_POLICY_ACTIONS : nullptr;
    const bool flip = policy_flip(d.rec[g0 + m].player, view);
    auto mix = [&](float p, int a) { return search_mix(p, nz[flip ? XQ_POLICY_ACTIONS - 1 - a : a], eps); };
    if (m == 0) {
        if (nz && d.expanded[g0]) {
            const int ne = d.nedges[g0];
            for (int k = lane; k < ne; k += 32) d.P[eb0 + k] = mix(d.P[eb0 + k], d.act[eb0 + k]);
        }
    } else {
        const int dm = d.depth[g0 + m];
        int w = m >> 5;
        uint32_t rest = bits[w];
        for (;;) {
            int js[kAdvBatch];
#pragma unroll
            for (int b = 0; b < kAdvBatch; ++b) {
                while (rest == 0 && w < last) rest = bits[++w];
                js[b] = rest ? (w << 5) + ffs32(rest) - 1 : -1;
                rest &= rest - 1;
            }
            if (js[0] < 0) break;
            // read the batch
            int parent[kAdvBatch], visits[kAdvBatch], reward[kAdvBatch], depth[kAdvBatch], ne[kAdvBatch];
            uint8_t pedge[kAdvBatch], nedges[kAdvBatch], expanded[kAdvBatch], term[kAdvBatch], winner[kAdvBatch];
            uint4 rec[kAdvBatch];
            float P[kAdvBatch][kAdvSlots], W[kAdvBatch][kAdvSlots];
            int N[kAdvBatch][kAdvSlots], C[kAdvBatch][kAdvSlots];
            int16_t A[kAdvBatch][kAdvSlots];
#pragma unroll
            for (int b = 0; b < kAdvBatch; ++b) {
                if (js[b] < 0) continue;
                const int64_t g = g0 + js[b], eb = g * kSearchEdges;
                parent[b] = d.parent[g]; visits[b] = d.visits[g]; reward[b] = d.reward[g]; depth[b] = d.depth[g];
                pedge[b] = d.pedge[g]; expanded[b] = d.expanded[g]; term[b] = d.term[g]; winner[b] = d.winner[g];
                nedges[b] = d.nedges[g];
                ne[b] = expanded[b] ? nedges[b] : 0;        // only the edge slots of an expanded node hold edges
                if (lane < 4) rec[b] = reinterpret_cast<const uint4*>(d.rec + g)[lane];
#pragma unroll
                for (int i = 0; i < kAdvSlots; ++i) {
                    const int k = lane + 32 * i;
                    if (k < ne[b]) { P[b][i] = d.P[eb + k]; N[b][i] = d.N[eb + k]; W[b][i] = d.W[eb + k]; C[b][i] = d.child[eb + k]; A[b][i] = d.act[eb + k]; }
                }
            }
            __syncwarp();
            // write it to the new slots
#pragma unroll
            for (int b = 0; b < kAdvBatch; ++b) {
                if (js[b] < 0) continue;
                const bool root = js[b] == m;
                const int64_t g = g0 + search_new_index(bits, prefix, js[b]), eb = g * kSearchEdges;
                if (lane == 0) {
                    d.parent[g] = root ? -1 : search_new_index(bits, prefix, parent[b]);
                    d.pedge[g] = root ? 0 : pedge[b];
                    d.visits[g] = visits[b]; d.reward[g] = root ? 0 : reward[b]; d.depth[g] = depth[b] - dm;
                    d.nedges[g] = nedges[b]; d.expanded[g] = expanded[b]; d.term[g] = term[b]; d.winner[g] = winner[b];
                }
                if (lane < 4) reinterpret_cast<uint4*>(d.rec + g)[lane] = rec[b];
#pragma unroll
                for (int i = 0; i < kAdvSlots; ++i) {
                    const int k = lane + 32 * i;
                    if (k < ne[b]) {
                        d.P[eb + k] = root && nz ? mix(P[b][i], A[b][i]) : P[b][i];
                        d.N[eb + k] = N[b][i]; d.W[eb + k] = W[b][i]; d.act[eb + k] = A[b][i];
                        d.child[eb + k] = C[b][i] >= 0 ? search_new_index(bits, prefix, C[b][i]) : -1;
                    }
                }
            }
        }
    }
    // 5. the kept count
    if (lane == 0) {
        d.count[t] = kept;
        if (kept_out) kept_out[t] = kept;
    }
}

// node nw of tree t as the child of `node` through edge bk: the parent's record after the action, exactly as xq_env_step_device
// (auto_reset = 0) makes it (one thread; sb a 12-word shared board)
__device__ __forceinline__ void search_make_child(const SearchDev& d, int64_t t, int64_t g0, int node, int bk, int nw, uint32_t* sb) {
    const int64_t g = g0 + node, eb = g * kSearchEdges;
    const int a = d.act[eb + bk];
    const int64_t gn = g0 + nw;
    SmemBoard b{sb, 1};
    b.load(d.rec + g);
    Meta m; m.load(d.rec + g);
    const int mover = m.player;
    apply_move(b, m, a / 90, a % 90);
    m.ctr++;
    uint32_t wd[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) wd[i] = b.base[i];
    const WordSummary s = summarize_words(wd);
    uint8_t term, win;
    search_status(s, m.move_count, term, win);
    const int diff = mover == RED ? s.mat_red - s.mat_black : s.mat_black - s.mat_red;
    b.store(d.rec + gn); m.store(d.rec + gn);
    d.parent[gn] = node; d.pedge[gn] = (uint8_t)bk; d.visits[gn] = 0; d.reward[gn] = reward_from_material(diff, m.move_count);
    d.depth[gn] = d.depth[g] + 1; d.nedges[gn] = 0; d.expanded[gn] = 0; d.term[gn] = term; d.winner[gn] = win;
    d.child[eb + bk] = nw;
    d.count[t] = nw + 1;
}

__global__ void __launch_bounds__(32 * kSelWarps) search_select_kernel(SearchDev d, float c_puct, float fpu, uint8_t* __restrict__ status,
                                                                      uint8_t* __restrict__ winner, int32_t* __restrict__ reward,
                                                                      int32_t* __restrict__ depth) {
    __shared__ uint32_t s_b[kSelWarps][12];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * kSelWarps + warp;
    if (t >= d.n) return;
    const int64_t g0 = t * d.cap;
    int node = 0, leaf;
    for (;;) {
        const int64_t g = g0 + node;
        if (!d.expanded[g] || d.term[g]) { leaf = node; break; }
        const int ne = d.nedges[g];
        const float sq = search_sqrt_visits(d.visits[g]);
        const int64_t eb = g * kSearchEdges;
        float bs = 0.f;
        int bk = -1;
        for (int k = lane; k < ne; k += 32) {
            const float v = search_puct(d.P[eb + k], d.N[eb + k], d.W[eb + k], c_puct, fpu, sq);
            if (search_better(v, k, bs, bk)) { bs = v; bk = k; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float os = __shfl_xor_sync(0xFFFFFFFFu, bs, off);
            const int ok = __shfl_xor_sync(0xFFFFFFFFu, bk, off);
            if (ok >= 0 && search_better(os, ok, bs, bk)) { bs = os; bk = ok; }
        }
        bk = __shfl_sync(0xFFFFFFFFu, bk, 0);
        const int child = d.child[eb + bk];
        if (child >= 0) { node = child; continue; }
        const int nw = d.count[t];
        if (lane == 0) search_make_child(d, t, g0, node, bk, nw, s_b[warp]);
        leaf = nw;
        break;
    }
    __syncwarp();
    if (lane < 4) {
        const int64_t g = g0 + leaf;
        reinterpret_cast<uint4*>(d.leaf_rec + t)[lane] = reinterpret_cast<const uint4*>(d.rec + g)[lane];
        if (lane == 0) {
            d.leaf[t] = leaf;
            if (status) status[t] = d.term[g];
            if (winner) winner[t] = d.winner[g];
            if (reward) reward[t] = d.reward[g];
            if (depth) depth[t] = d.depth[g];
        }
    }
}

// Multi-leaf selection (xq_search_select_leaves_device), one warp per tree: the L descents k = 0 .. L - 1 in order, each by the rules of
// search_select_kernel with the scores of search_puct_vl.  Lane k' stands for descent k' once it has ended: it holds that descent's leaf
// and its alive bit (search_inflight_node); the list index of the edge each descent took at depth dep is s_path[dep][k'] (depth < 200:
// a node at move 200 is terminal).  At a node the alive lanes add their edge to the warp's count row s_cnt (integer atomics: the counts
// do not depend on the order), the scoring lanes read it, and the alive lanes clear their entries again.  The slab changes only by child
// creation, as in search_select_kernel.  A descent that ends at an open leaf (unexpanded, not terminal) an earlier one ended at is a
// duplicate: status 4, leaf index -1 for the expand kernel.
constexpr int kSelLeavesWarps = 4;      // trees per CTA of the multi-leaf select kernel

__global__ void __launch_bounds__(32 * kSelLeavesWarps) search_select_leaves_kernel(SearchDev d, int L, float c_puct, float fpu, float vl,
                                                                                    uint8_t* __restrict__ status, uint8_t* __restrict__ winner,
                                                                                    int32_t* __restrict__ reward, int32_t* __restrict__ depth) {
    __shared__ uint32_t s_b[kSelLeavesWarps][12];
    __shared__ uint8_t s_path[kSelLeavesWarps][XQ_MAX_MOVES][32];
    __shared__ int32_t s_cnt[kSelLeavesWarps][kSearchEdges];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * kSelLeavesWarps + warp;
    if (t >= d.n) return;
    for (int e = lane; e < kSearchEdges; e += 32) s_cnt[warp][e] = 0;
    __syncwarp();
    const int64_t g0 = t * d.cap;
    int mine = -1;                      // lane k: the leaf of descent k
    for (int k = 0; k < L; ++k) {
        bool alive = lane < k;
        int node = 0, dep = 0, leaf;
        for (;;) {
            const int64_t g = g0 + node;
            if (!d.expanded[g] || d.term[g]) { leaf = node; break; }
            const int ne = d.nedges[g];
            const int cj = popc32(__ballot_sync(0xFFFFFFFFu, alive));
            if (alive) atomicAdd(&s_cnt[warp][s_path[warp][dep][lane]], 1);
            __syncwarp();
            const float sq = search_sqrt_visits(d.visits[g] + cj);
            const int64_t eb = g * kSearchEdges;
            float bs = 0.f;
            int bk = -1;
            for (int e = lane; e < ne; e += 32) {
                const float v = search_puct_vl(d.P[eb + e], d.N[eb + e], d.W[eb + e], s_cnt[warp][e], vl, c_puct, fpu, sq);
                if (search_better(v, e, bs, bk)) { bs = v; bk = e; }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float os = __shfl_xor_sync(0xFFFFFFFFu, bs, off);
                const int ok = __shfl_xor_sync(0xFFFFFFFFu, bk, off);
                if (ok >= 0 && search_better(os, ok, bs, bk)) { bs = os; bk = ok; }
            }
            bk = __shfl_sync(0xFFFFFFFFu, bk, 0);
            __syncwarp();
            if (alive) {
                const int e = s_path[warp][dep][lane];
                s_cnt[warp][e] = 0;
                alive = e == bk;
            }
            if (lane == 0) s_path[warp][dep][k] = (uint8_t)bk;
            __syncwarp();
            ++dep;
            const int child = d.child[eb + bk];
            if (child >= 0) { node = child; continue; }
            const int nw = d.count[t];
            if (lane == 0) search_make_child(d, t, g0, node, bk, nw, s_b[warp]);
            leaf = nw;
            break;
        }
        __syncwarp();
        const int64_t g = g0 + leaf, i = t * L + k;
        const bool open = !d.expanded[g] && !d.term[g];
        const bool dup = __any_sync(0xFFFFFFFFu, lane < k && mine == leaf) && open;
        if (lane == k) mine = leaf;
        if (lane < 4) {
            reinterpret_cast<uint4*>(d.leaf_rec + i)[lane] = reinterpret_cast<const uint4*>(d.rec + g)[lane];
            if (lane == 0) {
                d.leaf[i] = dup ? -1 : leaf;
                if (status) status[i] = dup ? 4 : d.term[g];
                if (winner) winner[i] = d.winner[g];
                if (reward) reward[i] = d.reward[g];
                if (depth) depth[i] = d.depth[g];
            }
        }
    }
}

template <int SDT>
__device__ __forceinline__ float search_score(const void* p, int64_t i) {
    return SDT == XQ_DTYPE_BF16 ? bf16_bits_to_float(__ldg(static_cast<const unsigned short*>(p) + i)) : __ldg(static_cast<const float*>(p) + i);
}

struct ExpandArgs {
    const void* scores; float t; int view; const float* values; const float* noise; float eps;
};

// the edges of a new node from the list-ordered cleaned scores (each), their maximum m and count n; the root mixes in the noise
template <class EACH>
__device__ __forceinline__ void search_write_edges(const SearchDev& d, const ExpandArgs& a, int64_t t, int64_t g, bool root, bool flip, EACH&& each,
                                                   int n, float m) {
    const int64_t eb = g * kSearchEdges;
    const float* nz = root && a.noise ? a.noise + t * XQ_POLICY_ACTIONS : nullptr;
    search_priors(each, n, m, a.t, [&](int k, float p) {
        if (nz) { const int ai = d.act[eb + k]; p = search_mix(p, nz[flip ? XQ_POLICY_ACTIONS - 1 - ai : ai], a.eps); }
        d.P[eb + k] = p; d.N[eb + k] = 0; d.W[eb + k] = 0.f; d.child[eb + k] = -1;
    });
    d.nedges[g] = (uint8_t)n;
    d.expanded[g] = 1;
    if (n == 0) d.term[g] = 3;
}

// Expansion of leaf `leaf` of tree t from the leaf record and score row `slot` (slot = t at one leaf per tree), one thread: the structure
// of policy_step_lane_kernel (the generator stages the legal scores into the [list index][thread] shared row s_row).  Returns 1 when the
// generator refuses the board and the generic kernel has to expand it.
template <int SDT>
__device__ __forceinline__ uint8_t search_expand_lane(const SearchDev& d, const ExpandArgs& a, int64_t t, int64_t slot, int leaf, int tid,
                                                      uint8_t* s_slot, const uint32_t* s_geo, uint32_t* s_view, float* s_row) {
    const int64_t g = t * d.cap + leaf;
    uint8_t generic = 0;
    if (!d.expanded[g] && d.term[g] == 0) {
        const uint4* rec = reinterpret_cast<const uint4*>(d.leaf_rec + slot);
        uint32_t w[12];
#pragma unroll
        for (int i = 0; i < 3; ++i) { const uint4 v = rec[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
        const int player = (int)((rec[3].x >> 16) & 0xFFu);
        LaneGen lg;
        if (policy_lane_gen(w, player, s_view + tid, s_slot + tid, kExpBoards, s_geo, lg)) {
            const bool flip = policy_flip(player, a.view);
            const void* sc = static_cast<const uint8_t*>(a.scores) + slot * XQ_POLICY_ACTIONS * (SDT == XQ_DTYPE_BF16 ? 2 : 4);
            const int64_t eb = g * kSearchEdges;
            const int cnt = policy_lane_emit(lg, player, [&](int idx, int from, int to) {
                s_row[idx * kExpBoards + tid] = search_score<SDT>(sc, policy_index(from, to, flip));
                d.act[eb + idx] = (int16_t)(from * 90 + to);
            });
            auto each = [&](auto&& f) { for (int k = 0; k < cnt; ++k) f(policy_clean(s_row[k * kExpBoards + tid])); };
            PolicyBest best{-INFINITY, -1};
            int k = 0;
            each([&](float l) { best.offer(l, k++); });
            search_write_edges(d, a, t, g, leaf == 0, flip, each, cnt, best.m);
        } else {
            generic = 1;
        }
    }
    return generic;
}

template <int SDT>
__global__ void __launch_bounds__(kExpBoards) search_expand_lane_kernel(SearchDev d, ExpandArgs a) {
    __shared__ uint8_t s_slot[32 * kExpBoards];
    __shared__ uint32_t s_geo[kGeoWords];
    __shared__ uint32_t s_view[kViewWords * kExpBoards];
    __shared__ float s_row[XQ_MAX_ACTIONS * kExpBoards];       // [list index][thread]: the raw scores of the legal actions
    const int tid = threadIdx.x;
    const int64_t t = (int64_t)blockIdx.x * kExpBoards + tid;
    for (int i = tid; i < kGeoWords; i += kExpBoards) s_geo[i] = geo_word(i);
    __syncthreads();
    if (t >= d.n) return;
    const int leaf = d.leaf[t];
    const int64_t g0 = t * d.cap;
    // the generic kernel expands a refused board; the backup below does not touch the new node's edges
    d.nonstd[t] = search_expand_lane<SDT>(d, a, t, t, leaf, tid, s_slot, s_geo, s_view, s_row);
    search_backup(leaf, a.values[t], d.parent + g0, d.pedge + g0, d.visits + g0, d.N + g0 * kSearchEdges, d.W + g0 * kSearchEdges);
}

// Expansion and backup after a multi-leaf selection of L slots per tree (slot i = t * L + k), one thread per slot: each status-0 slot
// expands its leaf as search_expand_lane_kernel does (its score row i, the noise row t at the root); the thread of slot 0 then backs up
// the tree's non-duplicate slots in slot order.  Expansions write only edges of unexpanded leaves, backups only edges of expanded
// ancestors and N_node, so the two need no ordering between threads and the result is that of "expand, then back up in slot order".
template <int SDT>
__global__ void __launch_bounds__(kExpBoards) search_expand_slots_kernel(SearchDev d, ExpandArgs a, int L) {
    __shared__ uint8_t s_slot[32 * kExpBoards];
    __shared__ uint32_t s_geo[kGeoWords];
    __shared__ uint32_t s_view[kViewWords * kExpBoards];
    __shared__ float s_row[XQ_MAX_ACTIONS * kExpBoards];
    const int tid = threadIdx.x;
    const int64_t i = (int64_t)blockIdx.x * kExpBoards + tid;
    for (int j = tid; j < kGeoWords; j += kExpBoards) s_geo[j] = geo_word(j);
    __syncthreads();
    if (i >= d.n * L) return;
    const int64_t t = i / L;
    const int leaf = d.leaf[i];          // -1: a duplicate slot
    d.nonstd[i] = leaf >= 0 ? search_expand_lane<SDT>(d, a, t, i, leaf, tid, s_slot, s_geo, s_view, s_row) : 0;
    if (i != t * L) return;
    const int64_t g0 = t * d.cap;
    for (int k = 0; k < L; ++k) {
        const int lf = d.leaf[i + k];
        if (lf >= 0) search_backup(lf, a.values[i + k], d.parent + g0, d.pedge + g0, d.visits + g0, d.N + g0 * kSearchEdges, d.W + g0 * kSearchEdges);
    }
}

// Expansion of a board the generator refuses (all_actions, one thread): leaf `leaf` of tree t from the record and score row of slot i
template <int SDT>
__device__ __forceinline__ void search_expand_generic(const SearchDev& d, const ExpandArgs& a, int64_t t, int64_t i, int leaf, uint32_t* sb) {
    const int64_t g = t * d.cap + leaf, eb = g * kSearchEdges;
    SmemBoard b{sb, kThreads};
    b.load(d.leaf_rec + i);
    Meta mt; mt.load(d.leaf_rec + i);
    const int player = mt.player;
    const bool flip = policy_flip(player, a.view);
    const void* sc = static_cast<const uint8_t*>(a.scores) + i * XQ_POLICY_ACTIONS * (SDT == XQ_DTYPE_BF16 ? 2 : 4);
    // the first 128 actions in list order; a player byte > 1 owns no piece
    auto each_action = [&](auto&& f) {
        int c = 0;
        if ((unsigned)player <= 1u) all_actions(b, player, [&](int from, int to) { if (c < kSearchEdges) f(from, to); ++c; });
    };
    PolicyBest best{-INFINITY, -1};
    int cnt = 0;
    each_action([&](int from, int to) {
        best.offer(policy_clean(search_score<SDT>(sc, policy_index(from, to, flip))), cnt);
        d.act[eb + cnt] = (int16_t)(from * 90 + to);
        ++cnt;
    });
    search_write_edges(d, a, t, g, leaf == 0, flip,
                       [&](auto&& f) { each_action([&](int from, int to) { f(policy_clean(search_score<SDT>(sc, policy_index(from, to, flip)))); }); },
                       cnt, best.m);
}

template <int SDT>
__global__ void __launch_bounds__(kThreads) search_expand_generic_kernel(SearchDev d, ExpandArgs a) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= d.n || !d.nonstd[t]) return;
    search_expand_generic<SDT>(d, a, t, t, d.leaf[t], s_board + threadIdx.x);
}

// the slots of a multi-leaf selection that search_expand_slots_kernel left to the generic generator
template <int SDT>
__global__ void __launch_bounds__(kThreads) search_expand_generic_slots_kernel(SearchDev d, ExpandArgs a, int L) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= d.n * L || !d.nonstd[i]) return;
    search_expand_generic<SDT>(d, a, i / L, i, d.leaf[i], s_board + threadIdx.x);
}

__global__ void __launch_bounds__(kRootThreads) search_root_kernel(SearchDev d, int view, int32_t* __restrict__ visits, float* __restrict__ q,
                                                                  int64_t* __restrict__ best) {
    __shared__ __align__(16) int32_t s_v[XQ_POLICY_ACTIONS];
    const int tid = threadIdx.x;
    const int64_t t = blockIdx.x, g = t * d.cap, eb = g * kSearchEdges;
    const int ne = d.expanded[g] ? d.nedges[g] : 0;
    const bool flip = policy_flip(d.rec[g].player, view);
    if (visits) {
        for (int i = tid; i < XQ_POLICY_ACTIONS / 4; i += kRootThreads) reinterpret_cast<int4*>(s_v)[i] = make_int4(0, 0, 0, 0);
        __syncthreads();
        for (int k = tid; k < ne; k += kRootThreads) { const int ai = d.act[eb + k]; s_v[flip ? XQ_POLICY_ACTIONS - 1 - ai : ai] = d.N[eb + k]; }
        __syncthreads();
        int4* dst = reinterpret_cast<int4*>(visits + t * XQ_POLICY_ACTIONS);
        for (int i = tid; i < XQ_POLICY_ACTIONS / 4; i += kRootThreads) dst[i] = reinterpret_cast<const int4*>(s_v)[i];
    }
    if (tid == 0) {
        // sums in list order; the most-visited edge, first in list order, none while no edge is visited
        int sn = 0, bn = 0, bk = -1;
        float sw = 0.f;
        for (int k = 0; k < ne; ++k) {
            const int nk = d.N[eb + k];
            sn += nk;
            sw = s_add(sw, d.W[eb + k]);
            if (nk > bn) { bn = nk; bk = k; }
        }
        if (q) q[t] = sn > 0 ? s_div(sw, (float)sn) : NAN;
        if (best) {
            const int ai = bk >= 0 ? d.act[eb + bk] : -1;
            best[t] = bk < 0 ? -1 : (flip ? XQ_POLICY_ACTIONS - 1 - ai : ai);
        }
    }
}

// The move of every tree from its root's visit counts (xq_search_play_device), one warp per tree: the lanes compare the root record with
// the env's and read the root's N row coalesced (edge k = lane + 32 i); the maximum and the total come from warp reductions.  Greedy: the
// first edge with the maximum (a min-reduction over the lanes' first hits).  Sampled: the lanes write the weights to shared memory and lane 0
// walks them in list order (search_play_sample).  Lane 0 then steps the env with the edge's action exactly as xq_env_policy_step_device
// (policy_apply on a 12-word shared-memory board); a stale or unvisited root steps with no action.
constexpr int kPlayWarps = 4;      // trees per CTA of the play and noise kernels

struct PlayArgs {
    xq_env_rec* envs; uint64_t env_id0, seed;
    float tau; int sample_plies, view, auto_reset;
    int64_t* actions; int32_t* reward; uint8_t *done, *winner, *captured, *valid;
};

__global__ void __launch_bounds__(32 * kPlayWarps) search_play_kernel(SearchDev d, PlayArgs a) {
    __shared__ uint32_t s_b[kPlayWarps][12];
    __shared__ float s_w[kPlayWarps][kSearchEdges];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * kPlayWarps + warp;
    if (t >= d.n) return;
    const int64_t g0 = t * d.cap, eb0 = g0 * kSearchEdges;
    bool diff = false;
    if (lane < 4) {
        const uint4 rv = reinterpret_cast<const uint4*>(d.rec + g0)[lane], ev = reinterpret_cast<const uint4*>(a.envs + t)[lane];
        diff = rv.x != ev.x || rv.y != ev.y || rv.z != ev.z || rv.w != ev.w;
    }
    const bool stale = __any_sync(0xFFFFFFFFu, diff);
    const int ne = !stale && d.expanded[g0] ? d.nedges[g0] : 0;
    int nv[kSearchEdges / 32];
    int nmax = 0;
#pragma unroll
    for (int i = 0; i < kSearchEdges / 32; ++i) {
        const int k = lane + 32 * i;
        nv[i] = k < ne ? d.N[eb0 + k] : 0;
        nmax = max(nmax, nv[i]);
    }
    nmax = __reduce_max_sync(0xFFFFFFFFu, nmax);
    int kp = -1;
    if (nmax > 0) {
        const xq_env_rec& root = d.rec[g0];
        if (a.tau == 0.f || (int)root.move_count >= a.sample_plies) {
            int first = kSearchEdges;
#pragma unroll
            for (int i = kSearchEdges / 32 - 1; i >= 0; --i) first = nv[i] == nmax && lane + 32 * i < ne ? lane + 32 * i : first;
            kp = (int)__reduce_min_sync(0xFFFFFFFFu, (unsigned)first);
        } else {
#pragma unroll
            for (int i = 0; i < kSearchEdges / 32; ++i) {
                const int k = lane + 32 * i;
                if (k < ne) s_w[warp][k] = search_play_weight(nv[i], nmax, a.tau);
            }
            __syncwarp();
            if (lane == 0) kp = search_play_sample([&](int k) { return s_w[warp][k]; }, ne, policy_uniform(rng(a.seed, a.env_id0 + (uint64_t)t, root.ctr)));
        }
    }
    if (lane != 0) return;
    SmemBoard b{s_b[warp], 1};
    b.load(a.envs + t);
    Meta m; m.load(a.envs + t);
    const int ai = kp >= 0 ? d.act[eb0 + kp] : 0, from = ai / 90, to = ai % 90;
    if (a.actions) a.actions[t] = kp >= 0 ? policy_index(from, to, policy_flip(m.player, a.view)) : -1;
    policy_apply(b, m, a.envs, t, kp >= 0, from, to, a.auto_reset, a.reward, a.done, a.winner, a.captured, a.valid);
}

// Dirichlet(alpha) noise mixed into the priors of every expanded root with at least one edge (xq_search_root_noise_device), one warp per
// tree: the lanes draw the log-Gamma variates of edges k = lane + 32 i (search_log_gamma), the maximum is a shuffle reduction, the
// exponentials go through shared memory where lane 0 sums them in list order; every lane then divides its edges, writes eta and mixes it
// into the priors in place (search_mix).  The arithmetic is search_dirichlet's.
__global__ void __launch_bounds__(32 * kPlayWarps) search_noise_kernel(SearchDev d, float alpha, float eps, uint64_t seed, uint64_t env_id0,
                                                                      const uint8_t* __restrict__ mask, float* __restrict__ noise_out) {
    __shared__ float s_e[kPlayWarps][kSearchEdges];
    __shared__ float s_sum[kPlayWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * kPlayWarps + warp;
    if (t >= d.n) return;
    const int64_t g0 = t * d.cap, eb0 = g0 * kSearchEdges;
    const int ne = (!mask || mask[t]) && d.expanded[g0] ? d.nedges[g0] : 0;
    float* out = noise_out ? noise_out + t * kSearchEdges : nullptr;
    if (ne == 0) {
        if (out) for (int k = lane; k < kSearchEdges; k += 32) out[k] = 0.f;
        return;
    }
    const uint64_t base = rng(seed, env_id0 + (uint64_t)t, d.rec[g0].ctr);
    float lg[kSearchEdges / 32];
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < kSearchEdges / 32; ++i) {
        const int k = lane + 32 * i;
        lg[i] = k < ne ? search_log_gamma(base, k, alpha) : -INFINITY;
        m = fmaxf(m, lg[i]);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, off));
#pragma unroll
    for (int i = 0; i < kSearchEdges / 32; ++i) {
        const int k = lane + 32 * i;
        if (k < ne) s_e[warp][k] = search_noise_exp(lg[i], m);
    }
    __syncwarp();
    if (lane == 0) {
        float s = 0.f;
        for (int k = 0; k < ne; ++k) s = s_add(s, s_e[warp][k]);
        s_sum[warp] = s;
    }
    __syncwarp();
    const float s = s_sum[warp];
#pragma unroll
    for (int i = 0; i < kSearchEdges / 32; ++i) {
        const int k = lane + 32 * i;
        const float eta = k < ne ? s_div(s_e[warp][k], s) : 0.f;
        if (k < ne) d.P[eb0 + k] = search_mix(d.P[eb0 + k], eta, eps);
        if (out) out[k] = eta;
    }
}

}  // namespace xq

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace xq;

struct xq_search_s {
    xq_env_t env = nullptr;
    int device = 0;
    int max_sims = 0;
    int max_leaves = 1;
    int leaves = 1;                // slots per tree of the last selection
    int sims = 0;
    int phase = 0;                 // 0 never reset, 1 ready for select, 2 selected (observe / leaves / expand_backup)
    bool maybe_nonstd = false;     // the env had injected boards at the reset: leaves may need the generic kernel
    void* slab = nullptr;
    SearchDev d{};
};

namespace {
constexpr size_t kNodeBytes = sizeof(xq_env_rec) + 4 * 4 + 5;                               // record, 4 int32, 5 bytes
constexpr size_t kEdgeBytes = 4 + 4 + 4 + 4 + 2;                                              // P, N, W, child, action
constexpr size_t kSlotBytes = sizeof(xq_env_rec) + 4 + 1;                                     // per leaf slot: leaf record, leaf, generic flag
constexpr size_t kTreeBytes = 4 + kSlotBytes;                                                  // node count and one slot
static_assert(kNodeBytes == 85 && kEdgeBytes == 18 && kSlotBytes == 69, "include/xq.h documents these sizes");

inline unsigned grid_of(int64_t n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }

int enter(xq_search_t s, EnvInfo* E, const char* fn) {
    if (!s) return fail(XQ_ERR_INVALID, "%s: null handle", fn);
    if (int rc = env_info(s->env, E)) return rc;
    XQ_CUDA(cudaSetDevice(E->device));
    return XQ_OK;
}
bool valid_view(int v) { return v == XQ_VIEW_ABSOLUTE || v == XQ_VIEW_SIDE_TO_MOVE; }
}  // namespace

int xq::search_roots(xq_search_t s, SearchRoots* out) {
    if (!s) return fail(XQ_ERR_INVALID, "null search handle");
    const SearchDev& d = s->d;
    *out = SearchRoots{s->env, s->phase, d.n, d.cap, d.rec, d.nedges, d.expanded, d.N, d.W, d.act};
    return XQ_OK;
}

extern "C" {

int xq_search_create(xq_env_t env, int max_simulations, xq_search_t* out) { return xq_search_create_ex(env, max_simulations, 1, out); }

int xq_search_create_ex(xq_env_t env, int max_simulations, int max_leaves, xq_search_t* out) {
    if (!out || !env) return fail(XQ_ERR_INVALID, "xq_search_create: null env or out");
    if (max_simulations < 1 || max_simulations > (1 << 24)) return fail(XQ_ERR_INVALID, "xq_search_create: max_simulations %d (1 .. 2^24)", max_simulations);
    if (max_leaves < 1 || max_leaves > XQ_SEARCH_MAX_LEAVES)
        return fail(XQ_ERR_INVALID, "xq_search_create_ex: max_leaves %d (1 .. %d)", max_leaves, XQ_SEARCH_MAX_LEAVES);
    EnvInfo E;
    if (int rc = env_info(env, &E)) return rc;
    XQ_CUDA(cudaSetDevice(E.device));
    xq_search_s* s = new (std::nothrow) xq_search_s();
    if (!s) return fail(XQ_ERR_NOMEM, "xq_search_create: out of host memory");
    s->env = env; s->device = E.device; s->max_sims = max_simulations; s->max_leaves = max_leaves;
    const int64_t n = E.n, cap = (int64_t)max_simulations + 1, nodes = n * cap, edges = nodes * kSearchEdges, slots = n * max_leaves;
    // one slab, every array 16-byte aligned
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_rec = take(sizeof(xq_env_rec) * nodes), o_parent = take(4 * nodes), o_visits = take(4 * nodes), o_reward = take(4 * nodes),
                 o_depth = take(4 * nodes), o_pedge = take(nodes), o_nedges = take(nodes), o_exp = take(nodes), o_term = take(nodes),
                 o_win = take(nodes), o_P = take(4 * edges), o_N = take(4 * edges), o_W = take(4 * edges), o_child = take(4 * edges),
                 o_act = take(2 * edges), o_count = take(4 * n), o_leaf = take(4 * slots), o_leafrec = take(sizeof(xq_env_rec) * slots), o_ns = take(slots);
    if (cudaMalloc(&s->slab, off) != cudaSuccess) {
        cudaGetLastError();
        delete s;
        return fail(XQ_ERR_NOMEM, "xq_search_create: %lld trees x %d simulations need %.1f GB of device memory", (long long)n, max_simulations, off / 1e9);
    }
    char* b = static_cast<char*>(s->slab);
    SearchDev& d = s->d;
    d.n = n; d.cap = (int)cap;
    d.rec = reinterpret_cast<xq_env_rec*>(b + o_rec);
    d.parent = reinterpret_cast<int32_t*>(b + o_parent); d.visits = reinterpret_cast<int32_t*>(b + o_visits);
    d.reward = reinterpret_cast<int32_t*>(b + o_reward); d.depth = reinterpret_cast<int32_t*>(b + o_depth);
    d.pedge = reinterpret_cast<uint8_t*>(b + o_pedge); d.nedges = reinterpret_cast<uint8_t*>(b + o_nedges);
    d.expanded = reinterpret_cast<uint8_t*>(b + o_exp); d.term = reinterpret_cast<uint8_t*>(b + o_term); d.winner = reinterpret_cast<uint8_t*>(b + o_win);
    d.P = reinterpret_cast<float*>(b + o_P); d.N = reinterpret_cast<int32_t*>(b + o_N); d.W = reinterpret_cast<float*>(b + o_W);
    d.child = reinterpret_cast<int32_t*>(b + o_child); d.act = reinterpret_cast<int16_t*>(b + o_act);
    d.count = reinterpret_cast<int32_t*>(b + o_count); d.leaf = reinterpret_cast<int32_t*>(b + o_leaf);
    d.leaf_rec = reinterpret_cast<xq_env_rec*>(b + o_leafrec); d.nonstd = reinterpret_cast<uint8_t*>(b + o_ns);
    *out = s;
    return XQ_OK;
}

int xq_search_destroy(xq_search_t s) {
    if (!s) return XQ_OK;
    cudaSetDevice(s->device);
    cudaFree(s->slab);             // synchronises with the work still queued on the env's stream
    delete s;
    return XQ_OK;
}

int xq_search_bytes_per_tree(int max_simulations, int64_t* bytes) { return xq_search_bytes_per_tree_ex(max_simulations, 1, bytes); }

int xq_search_bytes_per_tree_ex(int max_simulations, int max_leaves, int64_t* bytes) {
    if (!bytes || max_simulations < 1 || max_leaves < 1 || max_leaves > XQ_SEARCH_MAX_LEAVES)
        return fail(XQ_ERR_INVALID, "xq_search_bytes_per_tree: bad arguments");
    *bytes = (int64_t)(max_simulations + 1) * (int64_t)(kNodeBytes + kSearchEdges * kEdgeBytes) + (int64_t)kTreeBytes +
             (int64_t)(max_leaves - 1) * (int64_t)kSlotBytes;
    return XQ_OK;
}

int xq_search_reset(xq_search_t s) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_reset")) return rc;
    search_reset_kernel<<<grid_of(s->d.n, 256), 256, 0, E.stream>>>(s->d, E.d_envs);
    XQ_LAUNCH_CHECK();
    s->maybe_nonstd = E.maybe_nonstd;
    s->sims = 0;
    s->phase = 1;
    return XQ_OK;
}

int xq_search_advance(xq_search_t s, int min_free, const float* root_noise_dev, float noise_eps, int view, int32_t* kept_dev) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_advance")) return rc;
    if (s->max_sims > XQ_SEARCH_ADVANCE_MAX_SIMULATIONS)
        return fail(XQ_ERR_INVALID, "xq_search_advance: max_simulations %d (at most %d)", s->max_sims, XQ_SEARCH_ADVANCE_MAX_SIMULATIONS);
    if (min_free < 1 || min_free > s->max_sims) return fail(XQ_ERR_INVALID, "xq_search_advance: min_free %d (1 .. %d)", min_free, s->max_sims);
    if (!(noise_eps >= 0.f && noise_eps <= 1.f)) return fail(XQ_ERR_INVALID, "xq_search_advance: noise_eps must be in [0, 1]");
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_search_advance: view %d", view);
    if (s->phase == 0) return fail(XQ_ERR_STATE, "xq_search_advance: the search was never reset (xq_search_reset)");
    if (s->phase == 2) return fail(XQ_ERR_STATE, "xq_search_advance: the last selection was not expanded and backed up");
    // per warp (tree) the membership bitmap and one prefix count per 32-node word: cap / 4 bytes
    const size_t smem = (size_t)kAdvWarps * 2 * 4 * (size_t)((s->d.cap + 31) / 32);
    if (smem > 48 * 1024) XQ_CUDA(cudaFuncSetAttribute(search_advance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    search_advance_kernel<<<grid_of(s->d.n, kAdvWarps), 32 * kAdvWarps, smem, E.stream>>>(s->d, E.d_envs, min_free, root_noise_dev, noise_eps,
                                                                                         view, kept_dev);
    XQ_LAUNCH_CHECK();
    s->maybe_nonstd = s->maybe_nonstd || E.maybe_nonstd;      // kept boards descend from the old roots
    s->sims = s->max_sims - min_free;
    s->phase = 1;
    return XQ_OK;
}

int xq_search_select_device(xq_search_t s, float c_puct, float fpu, uint8_t* status_dev, uint8_t* winner_dev, int32_t* reward_dev,
                            int32_t* depth_dev) {
    return xq_search_select_leaves_device(s, 1, c_puct, fpu, 0.f, status_dev, winner_dev, reward_dev, depth_dev);
}

int xq_search_select_leaves_device(xq_search_t s, int leaves, float c_puct, float fpu, float virtual_loss, uint8_t* status_dev,
                                   uint8_t* winner_dev, int32_t* reward_dev, int32_t* depth_dev) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_select_device")) return rc;
    if (leaves < 1 || leaves > s->max_leaves) return fail(XQ_ERR_INVALID, "xq_search_select_leaves_device: leaves %d (1 .. %d)", leaves, s->max_leaves);
    if (!(c_puct >= 0.f && c_puct <= FLT_MAX)) return fail(XQ_ERR_INVALID, "xq_search_select_device: c_puct must be finite and >= 0");
    if (!(fpu >= -FLT_MAX && fpu <= FLT_MAX)) return fail(XQ_ERR_INVALID, "xq_search_select_device: fpu must be finite");
    if (!(virtual_loss >= 0.f && virtual_loss <= FLT_MAX))
        return fail(XQ_ERR_INVALID, "xq_search_select_leaves_device: virtual_loss must be finite and >= 0");
    if (s->phase == 0) return fail(XQ_ERR_STATE, "xq_search_select_device: the search was never reset (xq_search_reset)");
    if (s->phase == 2) return fail(XQ_ERR_STATE, "xq_search_select_device: the last selection was not expanded and backed up");
    if (s->sims + leaves > s->max_sims)
        return fail(XQ_ERR_STATE, "xq_search_select_device: %d simulations since the reset, %d more pass the capacity %d", s->sims, leaves, s->max_sims);
    if (leaves == 1)
        search_select_kernel<<<grid_of(s->d.n, kSelWarps), 32 * kSelWarps, 0, E.stream>>>(s->d, c_puct, fpu, status_dev, winner_dev, reward_dev, depth_dev);
    else
        search_select_leaves_kernel<<<grid_of(s->d.n, kSelLeavesWarps), 32 * kSelLeavesWarps, 0, E.stream>>>(s->d, leaves, c_puct, fpu, virtual_loss,
                                                                                                            status_dev, winner_dev, reward_dev, depth_dev);
    XQ_LAUNCH_CHECK();
    s->sims += leaves;
    s->leaves = leaves;
    s->phase = 2;
    return XQ_OK;
}

int xq_search_leaves_device(xq_search_t s, void** leaf_recs_dev) {
    if (!s || !leaf_recs_dev) return fail(XQ_ERR_INVALID, "xq_search_leaves_device: null argument");
    if (s->phase != 2) return fail(XQ_ERR_STATE, "xq_search_leaves_device: no selection since the last expand_backup / reset");
    *leaf_recs_dev = s->d.leaf_rec;
    return XQ_OK;
}

int xq_search_observe_leaves_device(xq_search_t s, void* planes_dev, int dtype, int view, int32_t* aux_dev) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_observe_leaves_device")) return rc;
    if (dtype < XQ_DTYPE_F32 || dtype > XQ_DTYPE_U8) return fail(XQ_ERR_INVALID, "xq_search_observe_leaves_device: dtype %d", dtype);
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_search_observe_leaves_device: view %d", view);
    if ((reinterpret_cast<uintptr_t>(planes_dev) & 15u) || (reinterpret_cast<uintptr_t>(aux_dev) & 15u))
        return fail(XQ_ERR_INVALID, "xq_search_observe_leaves_device: planes and aux must be 16-byte aligned");
    if (s->phase != 2) return fail(XQ_ERR_STATE, "xq_search_observe_leaves_device: no selection since the last expand_backup / reset");
    XQ_CUDA(launch_observe(s->d.leaf_rec, s->d.n * s->leaves, planes_dev, dtype, view, aux_dev, E.stream));
    return XQ_OK;
}

int xq_search_expand_backup_device(xq_search_t s, const void* scores_dev, int scores_dtype, float temperature, int view, const float* values_dev,
                                   const float* root_noise_dev, float noise_eps) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_expand_backup_device")) return rc;
    if (!scores_dev || !values_dev) return fail(XQ_ERR_INVALID, "xq_search_expand_backup_device: scores and values are required");
    if (scores_dtype != XQ_DTYPE_F32 && scores_dtype != XQ_DTYPE_BF16)
        return fail(XQ_ERR_INVALID, "xq_search_expand_backup_device: scores_dtype %d (f32 or bf16)", scores_dtype);
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_search_expand_backup_device: view %d", view);
    if (!(temperature > 0.f && temperature <= FLT_MAX)) return fail(XQ_ERR_INVALID, "xq_search_expand_backup_device: temperature must be finite and > 0");
    if (!(noise_eps >= 0.f && noise_eps <= 1.f)) return fail(XQ_ERR_INVALID, "xq_search_expand_backup_device: noise_eps must be in [0, 1]");
    if (s->phase != 2) return fail(XQ_ERR_STATE, "xq_search_expand_backup_device: no selection since the last expand_backup / reset");
    const ExpandArgs a{scores_dev, temperature, view, values_dev, root_noise_dev, noise_eps};
    const bool bf16 = scores_dtype == XQ_DTYPE_BF16;
    const int L = s->leaves;
    if (L > 1) {
        const int64_t slots = s->d.n * L;
        if (bf16) search_expand_slots_kernel<XQ_DTYPE_BF16><<<grid_of(slots, kExpBoards), kExpBoards, 0, E.stream>>>(s->d, a, L);
        else search_expand_slots_kernel<XQ_DTYPE_F32><<<grid_of(slots, kExpBoards), kExpBoards, 0, E.stream>>>(s->d, a, L);
        XQ_LAUNCH_CHECK();
        if (s->maybe_nonstd) {
            if (bf16) search_expand_generic_slots_kernel<XQ_DTYPE_BF16><<<grid_of(slots, kThreads), kThreads, 0, E.stream>>>(s->d, a, L);
            else search_expand_generic_slots_kernel<XQ_DTYPE_F32><<<grid_of(slots, kThreads), kThreads, 0, E.stream>>>(s->d, a, L);
            XQ_LAUNCH_CHECK();
        }
        s->phase = 1;
        return XQ_OK;
    }
    if (bf16) search_expand_lane_kernel<XQ_DTYPE_BF16><<<grid_of(s->d.n, kExpBoards), kExpBoards, 0, E.stream>>>(s->d, a);
    else search_expand_lane_kernel<XQ_DTYPE_F32><<<grid_of(s->d.n, kExpBoards), kExpBoards, 0, E.stream>>>(s->d, a);
    XQ_LAUNCH_CHECK();
    if (s->maybe_nonstd) {
        if (bf16) search_expand_generic_kernel<XQ_DTYPE_BF16><<<grid_of(s->d.n, kThreads), kThreads, 0, E.stream>>>(s->d, a);
        else search_expand_generic_kernel<XQ_DTYPE_F32><<<grid_of(s->d.n, kThreads), kThreads, 0, E.stream>>>(s->d, a);
        XQ_LAUNCH_CHECK();
    }
    s->phase = 1;
    return XQ_OK;
}

int xq_search_root_device(xq_search_t s, int view, int32_t* visits_dev, float* q_dev, int64_t* best_dev) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_root_device")) return rc;
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_search_root_device: view %d", view);
    if (reinterpret_cast<uintptr_t>(visits_dev) & 15u) return fail(XQ_ERR_INVALID, "xq_search_root_device: visits must be 16-byte aligned");
    if (s->phase == 0) return fail(XQ_ERR_STATE, "xq_search_root_device: the search was never reset (xq_search_reset)");
    search_root_kernel<<<(unsigned)s->d.n, kRootThreads, 0, E.stream>>>(s->d, view, visits_dev, q_dev, best_dev);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_search_play_device(xq_search_t s, float temperature, int sample_plies, int view, int auto_reset, int64_t* actions_dev, int32_t* reward_dev,
                          uint8_t* done_dev, uint8_t* winner_dev, uint8_t* captured_dev, uint8_t* valid_dev) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_play_device")) return rc;
    if (!(temperature >= 0.f && temperature <= FLT_MAX)) return fail(XQ_ERR_INVALID, "xq_search_play_device: temperature must be finite and >= 0");
    if (sample_plies < 0) return fail(XQ_ERR_INVALID, "xq_search_play_device: sample_plies %d < 0", sample_plies);
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_search_play_device: view %d", view);
    if (s->phase == 0) return fail(XQ_ERR_STATE, "xq_search_play_device: the search was never reset (xq_search_reset)");
    if (s->phase == 2) return fail(XQ_ERR_STATE, "xq_search_play_device: the last selection was not expanded and backed up");
    const PlayArgs a{E.d_envs, E.env_id0, E.seed, temperature, sample_plies, view, auto_reset,
                     actions_dev, reward_dev, done_dev, winner_dev, captured_dev, valid_dev};
    search_play_kernel<<<grid_of(s->d.n, kPlayWarps), 32 * kPlayWarps, 0, E.stream>>>(s->d, a);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_search_root_noise_device(xq_search_t s, float alpha, float eps, uint64_t seed, const uint8_t* mask_dev, float* noise_out_dev) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_root_noise_device")) return rc;
    if (!(alpha > 0.f && alpha <= FLT_MAX)) return fail(XQ_ERR_INVALID, "xq_search_root_noise_device: alpha must be finite and > 0");
    if (!(eps >= 0.f && eps <= 1.f)) return fail(XQ_ERR_INVALID, "xq_search_root_noise_device: eps must be in [0, 1]");
    if (s->phase == 0) return fail(XQ_ERR_STATE, "xq_search_root_noise_device: the search was never reset (xq_search_reset)");
    if (s->phase == 2) return fail(XQ_ERR_STATE, "xq_search_root_noise_device: the last selection was not expanded and backed up");
    search_noise_kernel<<<grid_of(s->d.n, kPlayWarps), 32 * kPlayWarps, 0, E.stream>>>(s->d, alpha, eps, seed, E.env_id0, mask_dev, noise_out_dev);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_search_get_tree(xq_search_t s, int64_t tree, xq_search_node* nodes_host, xq_search_edge* edges_host, int32_t* n_nodes) {
    EnvInfo E;
    if (int rc = enter(s, &E, "xq_search_get_tree")) return rc;
    if (tree < 0 || tree >= s->d.n) return fail(XQ_ERR_INVALID, "xq_search_get_tree: tree %lld of %lld", (long long)tree, (long long)s->d.n);
    if (!nodes_host || !n_nodes) return fail(XQ_ERR_INVALID, "xq_search_get_tree: nodes and n_nodes are required");
    if (s->phase == 0) return fail(XQ_ERR_STATE, "xq_search_get_tree: the search was never reset (xq_search_reset)");
    const SearchDev& d = s->d;
    const int64_t cap = d.cap, g0 = tree * cap;
    int32_t cnt = 0;
    XQ_CUDA(cudaMemcpyAsync(&cnt, d.count + tree, 4, cudaMemcpyDeviceToHost, E.stream));
    XQ_CUDA(cudaStreamSynchronize(E.stream));
    std::vector<xq_env_rec> rec(cnt);
    std::vector<int32_t> i32(4 * (size_t)cnt);
    std::vector<uint8_t> u8(5 * (size_t)cnt);
    XQ_CUDA(cudaMemcpyAsync(rec.data(), d.rec + g0, sizeof(xq_env_rec) * cnt, cudaMemcpyDeviceToHost, E.stream));
    int32_t* const i32src[4] = {d.parent, d.visits, d.reward, d.depth};
    uint8_t* const u8src[5] = {d.pedge, d.nedges, d.expanded, d.term, d.winner};
    for (int f = 0; f < 4; ++f) XQ_CUDA(cudaMemcpyAsync(i32.data() + f * cnt, i32src[f] + g0, 4 * (size_t)cnt, cudaMemcpyDeviceToHost, E.stream));
    for (int f = 0; f < 5; ++f) XQ_CUDA(cudaMemcpyAsync(u8.data() + f * cnt, u8src[f] + g0, (size_t)cnt, cudaMemcpyDeviceToHost, E.stream));
    const size_t ne = (size_t)cnt * kSearchEdges;
    std::vector<float> P(ne), W(ne);
    std::vector<int32_t> N(ne), C(ne);
    std::vector<int16_t> A(ne);
    if (edges_host) {
        const int64_t e0 = g0 * kSearchEdges;
        XQ_CUDA(cudaMemcpyAsync(P.data(), d.P + e0, 4 * ne, cudaMemcpyDeviceToHost, E.stream));
        XQ_CUDA(cudaMemcpyAsync(N.data(), d.N + e0, 4 * ne, cudaMemcpyDeviceToHost, E.stream));
        XQ_CUDA(cudaMemcpyAsync(W.data(), d.W + e0, 4 * ne, cudaMemcpyDeviceToHost, E.stream));
        XQ_CUDA(cudaMemcpyAsync(C.data(), d.child + e0, 4 * ne, cudaMemcpyDeviceToHost, E.stream));
        XQ_CUDA(cudaMemcpyAsync(A.data(), d.act + e0, 2 * ne, cudaMemcpyDeviceToHost, E.stream));
    }
    XQ_CUDA(cudaStreamSynchronize(E.stream));
    for (int32_t j = 0; j < cnt; ++j) {
        xq_search_node& o = nodes_host[j];
        memset(&o, 0, sizeof(o));
        o.rec = rec[j];
        o.parent = i32[j]; o.visits = i32[cnt + j]; o.reward = i32[2 * cnt + j]; o.depth = i32[3 * cnt + j];
        o.parent_edge = u8[j]; o.n_edges = u8[cnt + j]; o.expanded = u8[2 * cnt + j]; o.status = u8[3 * cnt + j]; o.winner = u8[4 * cnt + j];
        if (!edges_host) continue;
        for (int k = 0; k < kSearchEdges; ++k) {
            xq_search_edge& e = edges_host[(size_t)j * kSearchEdges + k];
            const size_t i = (size_t)j * kSearchEdges + k;
            if (o.expanded && k < o.n_edges) { e.action = A[i]; e.prior = P[i]; e.visits = N[i]; e.value_sum = W[i]; e.child = C[i]; }
            else { e.action = -1; e.prior = 0.f; e.visits = 0; e.value_sum = 0.f; e.child = -1; }
        }
    }
    *n_nodes = cnt;
    return XQ_OK;
}

}  // extern "C"
