// xq_policy.cu -- device-resident interface for a policy that is not the library's DQN (include/xq.h: xq_env_observe_device,
// xq_env_legal_mask_device, xq_env_legal_actions_device, xq_env_policy_step_device and its compact form).
//
// observe_kernel: the record -> [14][10][9] planes (f32 / bf16 / u8) + aux; write-bound, so a CTA stages 32 records in shared memory and
//   streams the 32 contiguous rows as one flat run of 16-byte stores (a row is 5,040 / 2,520 / 1,260 B: not a multiple of 16, the run is).
// mask_lane_kernel: the register-resident generator of the list kernel (policy_lane_gen = team_unpack_record_m + lane_movegen,
//   lane_emit_actions), each legal action setting one bit of the board's 254-word row in shared memory; the rows go out as one flat run of
//   16-byte stores, either as they are (packed) or expanded to one byte per index (dense: 8,100 B per board written once, no memset).
// policy_step_lane_kernel: the same generator; the score of each legal action is read once (only legal entries are touched) into a
//   [list index][thread] row of shared memory, the choice runs over that row in reference list order (policy_choose), the played
//   action is decoded with lane_select_kth and applied exactly as step_kernel (xq_env.cu) applies an xq_action.  The score rows are
//   dense ([n][8100], read at the policy index) or compact ([n][128], read at the list index): a template parameter of the step kernels.
// actions_lane_kernel: the same generator, the compact list of each board (policy indices in list order) staged per thread in shared
//   memory and written as one flat run of 16-byte stores; also over the leaf records of a search (launch_legal_actions).
// Boards the generator cannot take (a non-standard piece set, or a player byte > 1) are flagged and handled by the generic thread-per-board
// kernels on all_actions (xq_rules.cuh), with the same choice in list order.
#include "xq_common.cuh"
#include "xq_env_dev.cuh"
#include "xq_bitboard.cuh"
#include "xq_policy.cuh"

namespace xq {

constexpr int kPolBoards = 32;      // boards per CTA of the lane kernels (32 packed mask rows = 32.5 KB of shared memory)
constexpr int kObsBoards = 32;      // boards per CTA of observe_kernel
constexpr int kObsThreads = 256;

// ---- observation ------------------------------------------------------------------------------------------------------------------
// DT: XQ_DTYPE_F32 / BF16 / U8 -> bits of the value 1 and bits per element
template <int DT> struct ObsType;
template <> struct ObsType<XQ_DTYPE_F32> { static constexpr uint32_t one = 0x3F800000u; static constexpr int bits = 32; };
template <> struct ObsType<XQ_DTYPE_BF16> { static constexpr uint32_t one = 0x3F80u; static constexpr int bits = 16; };
template <> struct ObsType<XQ_DTYPE_U8> { static constexpr uint32_t one = 1u; static constexpr int bits = 8; };

template <int DT>
__global__ void __launch_bounds__(kObsThreads) observe_kernel(const xq_env_rec* __restrict__ envs, int64_t n, uint8_t* __restrict__ planes, int view,
                                                             int32_t* __restrict__ aux) {
    constexpr int V = 128 / ObsType<DT>::bits;                 // elements per 16-byte store
    constexpr int kRow = 14 * XQ_SQUARES;
    __shared__ uint32_t s_w[kObsBoards * 13];                  // 12 square words + (flip) per board
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * kObsBoards;
    const int live = (int)min((int64_t)kObsBoards, n - env0);
    if (tid < 4 * live) {
        const int e = tid >> 2, q = tid & 3;
        const uint4 v = reinterpret_cast<const uint4*>(envs + env0 + e)[q];
        if (q < 3) { s_w[e * 13 + 4 * q] = v.x; s_w[e * 13 + 4 * q + 1] = v.y; s_w[e * 13 + 4 * q + 2] = v.z; s_w[e * 13 + 4 * q + 3] = v.w; }
        else {
            const int player = (int)((v.x >> 16) & 0xFFu);
            s_w[e * 13 + 12] = policy_flip(player, view) ? 1u : 0u;
            if (aux) reinterpret_cast<int4*>(aux)[env0 + e] = make_int4(player, (int)(v.x & 0xFFFFu), (int)v.y, (int)v.z);
        }
    }
    __syncthreads();
    if (!planes) return;
    // element (board e, channel ch, square sp of the view): 1 iff the piece on the absolute square has code ch + 1 after the colour swap
    auto bit = [&](int e, int ch, int sp) -> uint32_t {
        const bool flip = s_w[e * 13 + 12] != 0;
        const int s = flip ? 89 - sp : sp;
        int code = (int)((s_w[e * 13 + (s >> 3)] >> (4 * (s & 7))) & 15u);
        code = (flip && (unsigned)(code - 1) < 14u) ? (code >= 8 ? code - 7 : code + 7) : code;
        return code == ch + 1 ? ObsType<DT>::one : 0u;
    };
    uint8_t* base = planes + env0 * kRow * (ObsType<DT>::bits / 8);
    const int total = live * kRow, nvec = total / V;
    for (int c = tid; c < nvec; c += kObsThreads) {            // 16-byte store c covers elements V c .. V c + V - 1 of the CTA's run
        const int f = c * V;
        int e = f / kRow, j = f - e * kRow;
        int ch = j / XQ_SQUARES, sp = j - ch * XQ_SQUARES;
        uint32_t o[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int i = 0; i < V; ++i) {
            o[i * ObsType<DT>::bits / 32] |= bit(e, ch, sp) << ((i * ObsType<DT>::bits) & 31);
            if (++sp == XQ_SQUARES) { sp = 0; if (++ch == 14) { ch = 0; ++e; } }
        }
        reinterpret_cast<uint4*>(base)[c] = make_uint4(o[0], o[1], o[2], o[3]);
    }
    for (int f = nvec * V + tid; f < total; f += kObsThreads) {  // the tail of the last CTA
        const int e = f / kRow, j = f - e * kRow, ch = j / XQ_SQUARES;
        const uint32_t v = bit(e, ch, j - ch * XQ_SQUARES);
        if (DT == XQ_DTYPE_F32) reinterpret_cast<uint32_t*>(base)[f] = v;
        else if (DT == XQ_DTYPE_BF16) reinterpret_cast<uint16_t*>(base)[f] = (uint16_t)v;
        else base[f] = (uint8_t)v;
    }
}

// ---- legal-action mask ------------------------------------------------------------------------------------------------------------
template <bool DENSE>
__global__ void __launch_bounds__(kPolBoards) mask_lane_kernel(const xq_env_rec* __restrict__ envs, int64_t n, uint8_t* __restrict__ out, int view,
                                                              uint8_t* __restrict__ nonstd) {
    __shared__ uint8_t s_slot[32 * kPolBoards];
    __shared__ uint32_t s_geo[kGeoWords];
    __shared__ uint32_t s_view[kViewWords * kPolBoards];
    __shared__ __align__(16) uint32_t s_mask[kPolBoards * XQ_MASK_WORDS];      // [board][word]: the CTA's rows as they lie in the packed output
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * kPolBoards, env = env0 + tid;
    for (int i = tid; i < kGeoWords; i += kPolBoards) s_geo[i] = geo_word(i);
    for (int i = tid; i < kPolBoards * XQ_MASK_WORDS / 4; i += kPolBoards) reinterpret_cast<uint4*>(s_mask)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    if (env < n) {
        const uint4* rec = reinterpret_cast<const uint4*>(envs + env);
        uint32_t w[12];
#pragma unroll
        for (int i = 0; i < 3; ++i) { const uint4 v = rec[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
        const int player = (int)((rec[3].x >> 16) & 0xFFu);
        LaneGen g;
        const bool ok = policy_lane_gen(w, player, s_view + tid, s_slot + tid, kPolBoards, s_geo, g);
        if (nonstd) nonstd[env] = ok ? 0 : 1;      // its row stays zero here; the generic kernel rewrites it
        if (ok) {
            const bool flip = policy_flip(player, view);
            uint32_t* row = s_mask + tid * XQ_MASK_WORDS;
            policy_lane_emit(g, player, [&](int, int from, int to) { const int i = policy_index(from, to, flip); row[i >> 5] |= 1u << (i & 31); });
        }
    }
    __syncthreads();
    const int live = (int)min((int64_t)kPolBoards, n - env0);
    if (!DENSE) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(out) + env0 * XQ_MASK_WORDS;
        const int words = live * XQ_MASK_WORDS, nvec = words / 4;
        for (int c = tid; c < nvec; c += kPolBoards) reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(s_mask)[c];
        for (int i = nvec * 4 + tid; i < words; i += kPolBoards) dst[i] = s_mask[i];
    } else {
        // output word ow = bytes 4 ow' .. of board ow / 2025: four consecutive indices i (i % 4 == 0) = four bits of one mask word, spread to bytes
        constexpr int kRowWords = XQ_POLICY_ACTIONS / 4;
        uint32_t* dst = reinterpret_cast<uint32_t*>(out + env0 * XQ_POLICY_ACTIONS);
        auto word = [&](int ow) -> uint32_t {
            const int e = ow / kRowWords, i = (ow - e * kRowWords) * 4;
            const uint32_t b = (s_mask[e * XQ_MASK_WORDS + (i >> 5)] >> (i & 31)) & 15u;
            return (b * 0x00204081u) & 0x01010101u;
        };
        const int words = live * kRowWords, nvec = words / 4;
        for (int c = tid; c < nvec; c += kPolBoards) reinterpret_cast<uint4*>(dst)[c] = make_uint4(word(4 * c), word(4 * c + 1), word(4 * c + 2), word(4 * c + 3));
        for (int i = nvec * 4 + tid; i < words; i += kPolBoards) dst[i] = word(i);
    }
}

// the boards the lane kernel flagged: the generic generator (all_actions), one thread per board, the whole row rewritten
__global__ void __launch_bounds__(kThreads) mask_generic_kernel(const xq_env_rec* __restrict__ envs, int64_t n, uint8_t* __restrict__ out, int packed,
                                                               int view, const uint8_t* __restrict__ only) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int64_t env = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (env >= n || !only[env]) return;
    SmemBoard b{s_board + threadIdx.x, kThreads};
    b.load(envs + env);
    Meta m; m.load(envs + env);
    const bool flip = policy_flip(m.player, view);
    if (packed) {
        uint32_t* row = reinterpret_cast<uint32_t*>(out) + env * XQ_MASK_WORDS;
        for (int i = 0; i < XQ_MASK_WORDS; ++i) row[i] = 0u;
        if ((unsigned)m.player <= 1u) all_actions(b, m.player, [&](int from, int to) { const int i = policy_index(from, to, flip); row[i >> 5] |= 1u << (i & 31); });
    } else {
        uint8_t* row = out + env * XQ_POLICY_ACTIONS;
        for (int i = 0; i < XQ_POLICY_ACTIONS / 4; ++i) reinterpret_cast<uint32_t*>(row)[i] = 0u;
        if ((unsigned)m.player <= 1u) all_actions(b, m.player, [&](int from, int to) { row[policy_index(from, to, flip)] = 1; });
    }
}

// ---- compact action lists ---------------------------------------------------------------------------------------------------------
// actions_lane_kernel: the generator's list of each board, entry k = its policy index, into a per-thread row of shared memory (row stride
// kActRow: odd, so the thread-major writes are conflict-free); the CTA's rows go out as one flat run of 16-byte stores, -1 past the count.
constexpr int kActRow = XQ_COMPACT_ACTIONS + 1;
__global__ void __launch_bounds__(kPolBoards) actions_lane_kernel(const xq_env_rec* __restrict__ recs, int64_t n, int32_t* __restrict__ actions,
                                                                 uint8_t* __restrict__ counts, int view, uint8_t* __restrict__ nonstd) {
    __shared__ uint8_t s_slot[32 * kPolBoards];
    __shared__ uint32_t s_geo[kGeoWords];
    __shared__ uint32_t s_view[kViewWords * kPolBoards];
    __shared__ int32_t s_list[kPolBoards * kActRow];
    __shared__ int s_cnt[kPolBoards];
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * kPolBoards, env = env0 + tid;
    for (int i = tid; i < kGeoWords; i += kPolBoards) s_geo[i] = geo_word(i);
    __syncthreads();
    int cnt = 0;
    if (env < n) {
        const uint4* rec = reinterpret_cast<const uint4*>(recs + env);
        uint32_t w[12];
#pragma unroll
        for (int i = 0; i < 3; ++i) { const uint4 v = rec[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
        const int player = (int)((rec[3].x >> 16) & 0xFFu);
        LaneGen g;
        const bool ok = policy_lane_gen(w, player, s_view + tid, s_slot + tid, kPolBoards, s_geo, g);
        nonstd[env] = ok ? 0 : 1;      // its row is written here as an empty list; the generic kernel rewrites it
        if (ok) {
            const bool flip = policy_flip(player, view);
            int32_t* row = s_list + tid * kActRow;
            cnt = policy_lane_emit(g, player, [&](int idx, int from, int to) { if (idx < XQ_COMPACT_ACTIONS) row[idx] = policy_index(from, to, flip); });
            cnt = min(cnt, XQ_COMPACT_ACTIONS);
        }
        if (counts) counts[env] = (uint8_t)cnt;
    }
    s_cnt[tid] = cnt;
    __syncthreads();
    const int live = (int)min((int64_t)kPolBoards, n - env0);
    int4* dst = reinterpret_cast<int4*>(actions + env0 * XQ_COMPACT_ACTIONS);
    for (int c = tid; c < live * (XQ_COMPACT_ACTIONS / 4); c += kPolBoards) {      // entries 4 (c % 32) .. + 3 of board c / 32
        const int e = c / (XQ_COMPACT_ACTIONS / 4), k = (c % (XQ_COMPACT_ACTIONS / 4)) * 4, ce = s_cnt[e];
        const int32_t* row = s_list + e * kActRow + k;
        dst[c] = make_int4(k < ce ? row[0] : -1, k + 1 < ce ? row[1] : -1, k + 2 < ce ? row[2] : -1, k + 3 < ce ? row[3] : -1);
    }
}

// the boards the lane kernel flagged: all_actions, one thread per board, the whole row rewritten
__global__ void __launch_bounds__(kThreads) actions_generic_kernel(const xq_env_rec* __restrict__ recs, int64_t n, int32_t* __restrict__ actions,
                                                                  uint8_t* __restrict__ counts, int view, const uint8_t* __restrict__ only) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int64_t env = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (env >= n || !only[env]) return;
    SmemBoard b{s_board + threadIdx.x, kThreads};
    b.load(recs + env);
    Meta m; m.load(recs + env);
    const bool flip = policy_flip(m.player, view);
    int32_t* row = actions + env * XQ_COMPACT_ACTIONS;
    int k = 0;
    if ((unsigned)m.player <= 1u)
        all_actions(b, m.player, [&](int from, int to) { if (k < XQ_COMPACT_ACTIONS) row[k++] = policy_index(from, to, flip); });
    if (counts) counts[env] = (uint8_t)k;
    for (int i = k; i < XQ_COMPACT_ACTIONS; ++i) row[i] = -1;
}

// the compact lists of any array of records (the envs of a handle, the leaves of a search); flags u8 [n] receives the lane kernel's
// refusals, and the generic kernel runs on them when `generic` (the records may hold boards the generator refuses)
cudaError_t launch_legal_actions(const xq_env_rec* recs, int64_t n, int32_t* actions, uint8_t* counts, int view, uint8_t* flags, bool generic,
                                 cudaStream_t stream) {
    actions_lane_kernel<<<grid_of(n, kPolBoards), kPolBoards, 0, stream>>>(recs, n, actions, counts, view, flags);
    ++g_launches;
    if (cudaError_t e = cudaGetLastError()) return e;
    if (generic) {
        actions_generic_kernel<<<grid_of(n, kThreads), kThreads, 0, stream>>>(recs, n, actions, counts, view, flags);
        ++g_launches;
    }
    return cudaGetLastError();
}

// ---- policy step ------------------------------------------------------------------------------------------------------------------
template <int SDT>
__device__ __forceinline__ float load_score(const void* p, int64_t i) {
    return SDT == XQ_DTYPE_BF16 ? bf16_bits_to_float(__ldg(static_cast<const unsigned short*>(p) + i)) : __ldg(static_cast<const float*>(p) + i);
}

struct PolicyArgs {
    xq_env_rec* envs; int64_t n; uint64_t env_id0, seed;
    const void* scores; int pick; float t; int view, auto_reset;
    int64_t* actions; float* logp; int32_t* reward; uint8_t *done, *winner, *captured, *valid;
};

template <int SDT, bool CMP>
__global__ void __launch_bounds__(kPolBoards) policy_step_lane_kernel(PolicyArgs a, uint8_t* __restrict__ nonstd) {
    __shared__ uint8_t s_slot[32 * kPolBoards];
    __shared__ uint32_t s_geo[kGeoWords];
    __shared__ uint32_t s_view[kViewWords * kPolBoards];       // the view memory of the generator, then the board of the apply step
    __shared__ float s_row[XQ_MAX_ACTIONS * kPolBoards];        // [list index][thread]: the cleaned scores of the legal actions
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * kPolBoards + tid;
    for (int i = tid; i < kGeoWords; i += kPolBoards) s_geo[i] = geo_word(i);
    __syncthreads();
    if (env >= a.n) return;
    const uint4* rec = reinterpret_cast<const uint4*>(a.envs + env);
    uint32_t w[12];
#pragma unroll
    for (int i = 0; i < 3; ++i) { const uint4 v = rec[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
    Meta mt; mt.load(a.envs + env);
    const int player = mt.player;
    LaneGen g;
    const bool ok = policy_lane_gen(w, player, s_view + tid, s_slot + tid, kPolBoards, s_geo, g);
    if (nonstd) nonstd[env] = ok ? 0 : 1;
    if (!ok) return;
    const bool flip = policy_flip(player, a.view);
    const void* sc = a.scores ? static_cast<const uint8_t*>(a.scores) + env * score_width<CMP>() * (SDT == XQ_DTYPE_BF16 ? 2 : 4) : nullptr;
    const int64_t given = a.pick == XQ_PICK_GIVEN ? a.actions[env] : -1;
    int given_k = -1;
    // the walk only stages the raw scores: its loads do not depend on each other and are in flight together (consuming each score in the
    // walk chained ~40 global-load latencies per board)
    const int cnt = policy_lane_emit(g, player, [&](int idx, int from, int to) {
        const int pi = policy_index(from, to, flip);
        if (sc) s_row[idx * kPolBoards + tid] = load_score<SDT>(sc, score_at<CMP>(idx, pi));
        given_k = pi == given ? idx : given_k;
    });
    auto each = [&](auto&& f) { for (int k = 0; k < cnt; ++k) f(policy_clean(s_row[k * kPolBoards + tid])); };
    PolicyBest best{-INFINITY, -1};
    if (sc) { int k = 0; each([&](float l) { best.offer(l, k++); }); }
    const float u = a.pick == XQ_PICK_SAMPLE ? policy_uniform(rng(a.seed, a.env_id0 + (uint64_t)env, mt.ctr)) : 0.f;
    const PolicyChoice c = policy_choose(each, cnt, best, given_k, a.pick, sc != nullptr, a.logp != nullptr, a.t, u);
    int from = 0, to = 0;
    if (c.k >= 0) { const uint32_t mv = lane_select_kth(g.own_sq, player, g.sdesc, g.cw, g.dw, (uint32_t)c.k, (uint32_t)cnt); from = (int)(mv & 0xFFu); to = (int)((mv >> 8) & 0xFFu); }
    if (a.pick != XQ_PICK_GIVEN && a.actions) a.actions[env] = c.k >= 0 ? policy_index(from, to, flip) : -1;
    if (a.logp) a.logp[env] = c.logp;
    SmemBoard b{s_view + tid, kPolBoards};
#pragma unroll
    for (int i = 0; i < 12; ++i) b.base[i * kPolBoards] = w[i];
    policy_apply(b, mt, a.envs, env, c.k >= 0, from, to, a.auto_reset, a.reward, a.done, a.winner, a.captured, a.valid);
}

// the boards the lane kernel flagged: all_actions enumerates the list in reference order (three or four times; rare boards); compact
// scores cover the first XQ_COMPACT_ACTIONS actions, and the choice is among those
template <int SDT, bool CMP>
__global__ void __launch_bounds__(kThreads) policy_step_generic_kernel(PolicyArgs a, const uint8_t* __restrict__ only) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int64_t env = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (env >= a.n || !only[env]) return;
    SmemBoard b{s_board + threadIdx.x, kThreads};
    b.load(a.envs + env);
    Meta mt; mt.load(a.envs + env);
    const int player = mt.player;
    const bool flip = policy_flip(player, a.view);
    const void* sc = a.scores ? static_cast<const uint8_t*>(a.scores) + env * score_width<CMP>() * (SDT == XQ_DTYPE_BF16 ? 2 : 4) : nullptr;
    const int64_t given = a.pick == XQ_PICK_GIVEN ? a.actions[env] : -1;
    auto each_action = [&](auto&& f) {      // f(list index, from, to); a player byte > 1 owns no piece
        int k = 0;
        if ((unsigned)player <= 1u) all_actions(b, player, [&](int from, int to) { if (!CMP || k < XQ_COMPACT_ACTIONS) f(k, from, to); ++k; });
    };
    PolicyBest best{-INFINITY, -1};
    int cnt = 0, given_k = -1;
    each_action([&](int k, int from, int to) {
        const int pi = policy_index(from, to, flip);
        if (sc) best.offer(policy_clean(load_score<SDT>(sc, score_at<CMP>(k, pi))), cnt);
        given_k = pi == given ? cnt : given_k;
        ++cnt;
    });
    const float u = a.pick == XQ_PICK_SAMPLE ? policy_uniform(rng(a.seed, a.env_id0 + (uint64_t)env, mt.ctr)) : 0.f;
    const PolicyChoice c = policy_choose(
        [&](auto&& f) { each_action([&](int k, int from, int to) { f(policy_clean(load_score<SDT>(sc, score_at<CMP>(k, policy_index(from, to, flip))))); }); },
        cnt, best, given_k, a.pick, sc != nullptr, a.logp != nullptr, a.t, u);
    int from = 0, to = 0, i = 0;
    if (c.k >= 0) each_action([&](int, int f, int t) { if (i == c.k) { from = f; to = t; } ++i; });
    if (a.pick != XQ_PICK_GIVEN && a.actions) a.actions[env] = c.k >= 0 ? policy_index(from, to, flip) : -1;
    if (a.logp) a.logp[env] = c.logp;
    policy_apply(b, mt, a.envs, env, c.k >= 0, from, to, a.auto_reset, a.reward, a.done, a.winner, a.captured, a.valid);
}

// observe_kernel on any array of records (xq_search.cu observes the leaves of its trees); planes 16-byte aligned, dtype checked by the caller
cudaError_t launch_observe(const xq_env_rec* recs, int64_t n, void* planes, int dtype, int view, int32_t* aux, cudaStream_t stream) {
    uint8_t* p = static_cast<uint8_t*>(planes);
    const unsigned grid = (unsigned)((n + kObsBoards - 1) / kObsBoards);
    if (dtype == XQ_DTYPE_F32) observe_kernel<XQ_DTYPE_F32><<<grid, kObsThreads, 0, stream>>>(recs, n, p, view, aux);
    else if (dtype == XQ_DTYPE_BF16) observe_kernel<XQ_DTYPE_BF16><<<grid, kObsThreads, 0, stream>>>(recs, n, p, view, aux);
    else observe_kernel<XQ_DTYPE_U8><<<grid, kObsThreads, 0, stream>>>(recs, n, p, view, aux);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace xq

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace xq;


extern "C" {

int xq_env_observe_device(xq_env_t h, void* planes_dev, int dtype, int view, int32_t* aux_dev) {
    EnvInfo E;
    if (int rc = env_info(h, &E)) return rc;
    if (dtype < XQ_DTYPE_F32 || dtype > XQ_DTYPE_U8) return fail(XQ_ERR_INVALID, "xq_env_observe_device: dtype %d", dtype);
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_env_observe_device: view %d", view);
    if (!aligned16(planes_dev) || !aligned16(aux_dev)) return fail(XQ_ERR_INVALID, "xq_env_observe_device: planes and aux must be 16-byte aligned");
    XQ_CUDA(cudaSetDevice(E.device));
    uint8_t* p = static_cast<uint8_t*>(planes_dev);
    const unsigned grid = grid_of(E.n, kObsBoards);
    if (dtype == XQ_DTYPE_F32) observe_kernel<XQ_DTYPE_F32><<<grid, kObsThreads, 0, E.stream>>>(E.d_envs, E.n, p, view, aux_dev);
    else if (dtype == XQ_DTYPE_BF16) observe_kernel<XQ_DTYPE_BF16><<<grid, kObsThreads, 0, E.stream>>>(E.d_envs, E.n, p, view, aux_dev);
    else observe_kernel<XQ_DTYPE_U8><<<grid, kObsThreads, 0, E.stream>>>(E.d_envs, E.n, p, view, aux_dev);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_env_legal_mask_device(xq_env_t h, void* mask_dev, int packed, int view) {
    EnvInfo E;
    if (int rc = env_info(h, &E)) return rc;
    if (!mask_dev || !aligned16(mask_dev)) return fail(XQ_ERR_INVALID, "xq_env_legal_mask_device: the mask must be a 16-byte aligned device buffer");
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_env_legal_mask_device: view %d", view);
    XQ_CUDA(cudaSetDevice(E.device));
    uint8_t* out = static_cast<uint8_t*>(mask_dev);
    if (packed) mask_lane_kernel<false><<<grid_of(E.n, kPolBoards), kPolBoards, 0, E.stream>>>(E.d_envs, E.n, out, view, E.d_nonstd);
    else mask_lane_kernel<true><<<grid_of(E.n, kPolBoards), kPolBoards, 0, E.stream>>>(E.d_envs, E.n, out, view, E.d_nonstd);
    XQ_LAUNCH_CHECK();
    if (E.maybe_nonstd) {      // injected boards (xq_env_set_boards) may have a piece set or a player byte the generator does not take
        mask_generic_kernel<<<grid_of(E.n, kThreads), kThreads, 0, E.stream>>>(E.d_envs, E.n, out, packed ? 1 : 0, view, E.d_nonstd);
        XQ_LAUNCH_CHECK();
    }
    return XQ_OK;
}

int xq_env_legal_actions_device(xq_env_t h, int view, int32_t* actions_dev, uint8_t* counts_dev) {
    EnvInfo E;
    if (int rc = env_info(h, &E)) return rc;
    if (!actions_dev || !aligned16(actions_dev)) return fail(XQ_ERR_INVALID, "xq_env_legal_actions_device: actions must be a 16-byte aligned device buffer");
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_env_legal_actions_device: view %d", view);
    XQ_CUDA(cudaSetDevice(E.device));
    XQ_CUDA(launch_legal_actions(E.d_envs, E.n, actions_dev, counts_dev, view, E.d_nonstd, E.maybe_nonstd, E.stream));
    return XQ_OK;
}

}  // extern "C"

namespace {
// the checks and launches of xq_env_policy_step_device and its compact form (CMP: the score rows are compact)
template <bool CMP>
int policy_step(const char* fn, xq_env_t h, const void* scores_dev, int scores_dtype, int pick, float temperature, int view, int auto_reset,
                int64_t* actions_dev, float* logp_dev, int32_t* reward_dev, uint8_t* done_dev, uint8_t* winner_dev, uint8_t* captured_dev,
                uint8_t* valid_dev) {
    EnvInfo E;
    if (int rc = env_info(h, &E)) return rc;
    if (pick < XQ_PICK_GREEDY || pick > XQ_PICK_GIVEN) return fail(XQ_ERR_INVALID, "%s: pick %d", fn, pick);
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "%s: view %d", fn, view);
    if (scores_dev && scores_dtype != XQ_DTYPE_F32 && scores_dtype != XQ_DTYPE_BF16)
        return fail(XQ_ERR_INVALID, "%s: scores_dtype %d (f32 or bf16)", fn, scores_dtype);
    if (CMP && !aligned16(scores_dev)) return fail(XQ_ERR_INVALID, "%s: compact scores must be 16-byte aligned", fn);
    if (pick != XQ_PICK_GIVEN && !scores_dev) return fail(XQ_ERR_INVALID, "%s: GREEDY and SAMPLE need scores", fn);
    if (pick == XQ_PICK_GIVEN && !actions_dev) return fail(XQ_ERR_INVALID, "%s: GIVEN needs actions", fn);
    if ((pick == XQ_PICK_SAMPLE || (logp_dev && scores_dev)) && !(temperature > 0.f && temperature <= FLT_MAX))
        return fail(XQ_ERR_INVALID, "%s: temperature must be finite and > 0", fn);
    XQ_CUDA(cudaSetDevice(E.device));
    const PolicyArgs a{E.d_envs, E.n, E.env_id0, E.seed, scores_dev, pick, temperature, view, auto_reset,
                       actions_dev, logp_dev, reward_dev, done_dev, winner_dev, captured_dev, valid_dev};
    const bool bf16 = scores_dev && scores_dtype == XQ_DTYPE_BF16;
    if (bf16) policy_step_lane_kernel<XQ_DTYPE_BF16, CMP><<<grid_of(E.n, kPolBoards), kPolBoards, 0, E.stream>>>(a, E.d_nonstd);
    else policy_step_lane_kernel<XQ_DTYPE_F32, CMP><<<grid_of(E.n, kPolBoards), kPolBoards, 0, E.stream>>>(a, E.d_nonstd);
    XQ_LAUNCH_CHECK();
    if (E.maybe_nonstd) {
        if (bf16) policy_step_generic_kernel<XQ_DTYPE_BF16, CMP><<<grid_of(E.n, kThreads), kThreads, 0, E.stream>>>(a, E.d_nonstd);
        else policy_step_generic_kernel<XQ_DTYPE_F32, CMP><<<grid_of(E.n, kThreads), kThreads, 0, E.stream>>>(a, E.d_nonstd);
        XQ_LAUNCH_CHECK();
    }
    return XQ_OK;
}
}  // namespace

extern "C" {

int xq_env_policy_step_device(xq_env_t h, const void* scores_dev, int scores_dtype, int pick, float temperature, int view, int auto_reset,
                              int64_t* actions_dev, float* logp_dev, int32_t* reward_dev, uint8_t* done_dev, uint8_t* winner_dev,
                              uint8_t* captured_dev, uint8_t* valid_dev) {
    return policy_step<false>("xq_env_policy_step_device", h, scores_dev, scores_dtype, pick, temperature, view, auto_reset, actions_dev, logp_dev,
                              reward_dev, done_dev, winner_dev, captured_dev, valid_dev);
}

int xq_env_policy_step_compact_device(xq_env_t h, const void* scores_dev, int scores_dtype, int pick, float temperature, int view, int auto_reset,
                                      int64_t* actions_dev, float* logp_dev, int32_t* reward_dev, uint8_t* done_dev, uint8_t* winner_dev,
                                      uint8_t* captured_dev, uint8_t* valid_dev) {
    return policy_step<true>("xq_env_policy_step_compact_device", h, scores_dev, scores_dtype, pick, temperature, view, auto_reset, actions_dev,
                             logp_dev, reward_dev, done_dev, winner_dev, captured_dev, valid_dev);
}

}  // extern "C"
