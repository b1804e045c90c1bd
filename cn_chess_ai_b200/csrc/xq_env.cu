// xq_env.cu -- batched Xiangqi environment on sm_100a: ordered legal-move generation, move
// application, terminal / winner / reward evaluation and the fused random-policy rollout.
//
// Data layout in HBM: one 64-byte xq_env_rec per environment (include/xq.h), AoS, 64-B aligned:
// a warp of the thread-per-board kernels touches 32 consecutive records = 2 KB contiguous.
// On chip each thread keeps its board as 12 nibble-packed words in shared memory, interleaved by
// thread (SmemBoard) so that data-dependent square lookups never bank-conflict, and the 16-byte
// meta in registers.  The rollout kernel loads a record once, plays n_plies plies entirely on
// chip and stores it once: per ply it touches HBM only for the optional 8-byte trace record.
//
// Reference functions replaced: ChessBoard::{getValidMoves,isValidMove,movePiece,checkGameOver,
// getWinner,reset} (src/chessboard.cpp), ChessAI::{getAllValidActions,evaluateBoard,
// getStateRepresentation} and the loop body of ChessAI::train (src/chessai.cpp:96-119).
#include <stdarg.h>
#include <string.h>

#include <new>
#include <vector>

#include <stdlib.h>

#include "xq_common.cuh"
#include <algorithm>

#include "xq_env_dev.cuh"
#include "xq_bitboard.cuh"

namespace xq {

std::string& last_error() { static thread_local std::string e; return e; }
unsigned long long g_launches = 0;
int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error() = buf;
    return code;
}


// ------------------------------------------------------------------------------------------
// K1: ordered legal-action lists (ChessAI::getAllValidActions for the side to move).
// The list is staged in shared memory (one padded row per thread) and written out with
// fully coalesced 4-byte stores: 256 B per env.
__global__ void __launch_bounds__(kThreads) legal_moves_kernel(const xq_env_rec* __restrict__ envs, int64_t n,
                                                              uint8_t* __restrict__ counts, uint32_t* __restrict__ actions,
                                                              const uint8_t* __restrict__ only /* boards the register-resident kernel flagged; null = all */) {
    __shared__ uint32_t s_board[12 * kThreads];
    __shared__ uint32_t s_list[kThreads * kListStride];
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * kThreads;
    const int64_t env = env0 + tid;
    uint16_t* my = reinterpret_cast<uint16_t*>(&s_list[tid * kListStride]);
    for (int i = 0; i < 64; ++i) s_list[tid * kListStride + i] = 0xFFFFFFFFu;
    if (env < n && (only == nullptr || only[env] != 0)) {
        SmemBoard b{s_board + tid, kThreads};
        b.load(envs + env);
        Meta m; m.load(envs + env);
        int cnt = 0;
        all_actions(b, m.player, [&](int from, int to) { if (cnt < XQ_MAX_ACTIONS) my[cnt++] = XQ_ACTION(from, to); });
        counts[env] = (uint8_t)cnt;
    }
    __syncthreads();
    const int64_t live = min((int64_t)kThreads, n - env0);
    for (int j = tid; j < live * 64; j += kThreads)
        if (only == nullptr || only[env0 + (j >> 6)] != 0) actions[env0 * 64 + j] = s_list[(j >> 6) * kListStride + (j & 63)];
}

// K1s: the same list filtered by the opt-in strict legality test (xq_rules.cuh: leaves_general_safe): self-check and
// flying-general rejection, which the reference does not have.  Every pseudo-legal action is tried on the shared-memory board.
__global__ void __launch_bounds__(kThreads) legal_moves_strict_kernel(const xq_env_rec* __restrict__ envs, int64_t n,
                                                                     uint8_t* __restrict__ counts, uint32_t* __restrict__ actions) {
    __shared__ uint32_t s_board[12 * kThreads];
    __shared__ uint32_t s_list[kThreads * kListStride];
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * kThreads;
    const int64_t env = env0 + tid;
    uint16_t* my = reinterpret_cast<uint16_t*>(&s_list[tid * kListStride]);
    if (env < n) {
        SmemBoard b{s_board + tid, kThreads};
        b.load(envs + env);
        Meta m; m.load(envs + env);
        int cnt = 0, kept = 0;
        all_actions(b, m.player, [&](int from, int to) { if (cnt < XQ_MAX_ACTIONS) my[cnt++] = XQ_ACTION(from, to); });
        for (int k = 0; k < cnt; ++k) {
            const int a = my[k];
            if (leaves_general_safe(b, m.player, XQ_ACTION_FROM(a), XQ_ACTION_TO(a))) my[kept++] = (uint16_t)a;
        }
        for (int k = kept; k < XQ_MAX_ACTIONS; ++k) my[k] = XQ_ACTION_NONE;
        counts[env] = (uint8_t)kept;
    }
    __syncthreads();
    const int64_t live = min((int64_t)kThreads, n - env0);
    for (int j = tid; j < live * 64; j += kThreads) actions[env0 * 64 + j] = s_list[(j >> 6) * kListStride + (j & 63)];
}

// K1b: ChessBoard::getValidMoves(row,col) for one square of every env
__global__ void __launch_bounds__(kThreads) valid_moves_kernel(const xq_env_rec* __restrict__ envs, int64_t n, int row, int col,
                                                              uint8_t* __restrict__ counts, uint8_t* __restrict__ to_out) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * kThreads + tid;
    if (env >= n) return;
    SmemBoard b{s_board + tid, kThreads};
    b.load(envs + env);
    int cnt = 0;
    uint8_t* out = to_out + env * 20;
    for (int i = 0; i < 20; ++i) out[i] = 0xFF;
    if (inside(row, col)) {
        const int code = b.get(row * 9 + col);
        if (code != 0) gen_piece(b, row, col, code, [&](int to) { if (cnt < 20) out[cnt] = (uint8_t)to; ++cnt; });
    }
    counts[env] = (uint8_t)cnt;
}

// K1c: ChessBoard::isValidMove for one (fr,fc,tr,tc) per env
__global__ void __launch_bounds__(kThreads) is_valid_kernel(const xq_env_rec* __restrict__ envs, int64_t n,
                                                           const int4* __restrict__ moves, uint8_t* __restrict__ valid) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * kThreads + tid;
    if (env >= n) return;
    SmemBoard b{s_board + tid, kThreads};
    b.load(envs + env);
    const int4 mv = moves[env];
    valid[env] = is_valid_move(b, mv.x, mv.y, mv.z, mv.w) ? 1 : 0;
}

// K2: one externally chosen action per env: movePiece + evaluateBoard + checkGameOver + getWinner
__global__ void __launch_bounds__(kThreads) step_kernel(xq_env_rec* __restrict__ envs, int64_t n, const uint16_t* __restrict__ actions,
                                                       int32_t* __restrict__ reward, uint8_t* __restrict__ done,
                                                       uint8_t* __restrict__ winner, uint8_t* __restrict__ captured,
                                                       uint8_t* __restrict__ valid, int auto_reset) {
    __shared__ uint32_t s_board[12 * kThreads];
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * kThreads + tid;
    if (env >= n) return;
    SmemBoard b{s_board + tid, kThreads};
    b.load(envs + env);
    Meta m; m.load(envs + env);
    const int a = actions[env];
    const int from = XQ_ACTION_FROM(a), to = XQ_ACTION_TO(a);
    const int mover = m.player;
    const bool ok = from < 90 && to < 90 && is_valid_move(b, from / 9, from % 9, to / 9, to % 9);
    int cap = 0;
    if (ok) { cap = apply_move(b, m, from, to); m.ctr++; }
    // material / Generals from the 12 packed words in registers (bit-plane SIMD, xq_bitboard.cuh) instead of a scan over the 90 squares
    uint32_t wd[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) wd[i] = b.base[i * b.stride];
    const WordSummary s = summarize_words(wd);
    const int diff = mover == RED ? s.mat_red - s.mat_black : s.mat_black - s.mat_red;
    const bool over = m.move_count >= XQ_MAX_MOVES || s.gen_red == 127 || s.gen_black == 127;
    const int win = (s.gen_red == 127 && s.gen_black == 127) ? NOCOLOR : (s.gen_red < s.gen_black ? RED : BLACK);      // first General in square order
    if (reward) reward[env] = reward_from_material(diff, m.move_count);
    if (done) done[env] = over ? 1 : 0;
    if (winner) winner[env] = (uint8_t)win;
    if (captured) captured[env] = (uint8_t)cap;
    if (valid) valid[env] = ok ? 1 : 0;
    if (over && auto_reset) { reset_board(b); m.reset(); }
    if (ok || (over && auto_reset)) { b.store(envs + env); m.store(envs + env); }
}

// K3: reset selected envs (ChessBoard::reset)
__global__ void reset_kernel(xq_env_rec* __restrict__ envs, int64_t n, const uint8_t* __restrict__ mask, int clear_ctr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one 16-byte quarter record per thread
    const int64_t env = i >> 2;
    const int q = (int)(i & 3);
    if (env >= n || (mask && !mask[env])) return;
    uint4* p = reinterpret_cast<uint4*>(envs + env) + q;
    if (q < 3) *p = make_uint4(kOpening[4 * q], kOpening[4 * q + 1], kOpening[4 * q + 2], kOpening[4 * q + 3]);
    else { const uint32_t ctr = clear_ctr ? 0u : p->w; *p = make_uint4(0u, 0u, 0u, ctr); }
}

// K4: one-hot state encoding (ChessAI::getStateRepresentation), 1260 doubles per env.
// One warp per env: lane writes are 8-byte and consecutive -> coalesced 256-B segments.
__global__ void __launch_bounds__(256) state_onehot_kernel(const xq_env_rec* __restrict__ envs, int64_t n, double* __restrict__ out) {
    const int64_t env = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (env >= n) return;
    const uint32_t w = lane < 12 ? envs[env].sq[lane] : 0u;
    double* o = out + env * XQ_STATE_SIZE;
    for (int i = lane; i < XQ_STATE_SIZE; i += 32) {
        const int s = i / 14, ch = i - s * 14;
        const uint32_t word = __shfl_sync(0xFFFFFFFFu, w, s >> 3);
        const int code = (word >> ((s & 7) * 4)) & 15;
        o[i] = (code == ch + 1) ? 1.0 : 0.0;
    }
}

// ------------------------------------------------------------------------------------------
// K5: fused random-policy rollout, v1: one thread per board, boards resident in shared memory
// for all n_plies plies.  Per ply: ordered list -> list[idx31 % n] -> apply -> reward ->
// terminal/winner -> reset on terminal.
struct StatsAcc {
    unsigned long long steps, games, red_wins, black_wins, cap_games, captures, legal_sum;
    long long reward_sum;
};

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

__global__ void __launch_bounds__(kThreads) rollout_random_kernel(xq_env_rec* __restrict__ envs, int64_t n, uint64_t env_id0,
                                                                 uint64_t seed, int n_plies, xq_trace_rec* __restrict__ trace,
                                                                 xq_env_stats* __restrict__ stats, const uint8_t* __restrict__ only,
                                                                 xq_env_rec* __restrict__ mirror /* mapped host copy of the final boards, or null */) {
    __shared__ uint32_t s_board[12 * kThreads];
    __shared__ uint32_t s_list[64 * kThreads];   // action list, u16 pairs, word-interleaved by thread
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * kThreads + tid;
    StatsAcc st{0, 0, 0, 0, 0, 0, 0, 0};
    if (env < n && (only == nullptr || only[env] != 0)) {   // `only`: boards the slot kernel could not map
        SmemBoard b{s_board + tid, kThreads};
        b.load(envs + env);
        Meta m; m.load(envs + env);
        Summary s = summarize(b);
        if (m.move_count >= XQ_MAX_MOVES || !(s.red_alive && s.black_alive)) {   // injected terminal board: chessai.cpp:90,96
            reset_board(b); m.reset(); s = summarize(b);
        }
        int mat_red = s.mat_red, mat_black = s.mat_black;
        uint16_t* list = reinterpret_cast<uint16_t*>(s_list);   // entry k of thread t: list[(k>>1)*2*kThreads + 2*t + (k&1)]
        for (int p = 0; p < n_plies; ++p) {
            int cnt = 0;
            all_actions(b, m.player, [&](int from, int to) {
                if (cnt < XQ_MAX_ACTIONS) { list[(cnt >> 1) * 2 * kThreads + 2 * tid + (cnt & 1)] = XQ_ACTION(from, to); ++cnt; }
            });
            xq_trace_rec tr;   // assembled in registers, stored as one 8-byte word pair
            if (cnt == 0) {   // chessai.cpp:100-103: no action ends the episode; the slot restarts
                tr.action = XQ_ACTION_NONE; tr.n_legal = 0; tr.flags = 1 | (NOCOLOR << 1); tr.reward = 0;
                reset_board(b); m.reset(); m.ctr++; mat_red = mat_black = 1480; st.games++;
            } else {
                const uint64_t x = rng(seed, env_id0 + (uint64_t)env, m.ctr);
                const int k = (int)((uint32_t)(x >> 33) % (uint32_t)cnt);
                const int a = list[(k >> 1) * 2 * kThreads + 2 * tid + (k & 1)];
                const int mover = m.player;
                const int cap = apply_move(b, m, XQ_ACTION_FROM(a), XQ_ACTION_TO(a));
                m.ctr++;
                if (cap != 0) { const int sc = piece_score(type_of(cap)); if (cap >= 8) mat_black -= sc; else mat_red -= sc; st.captures++; }
                const int reward = reward_from_material(mover == RED ? mat_red - mat_black : mat_black - mat_red, m.move_count);
                bool over = m.move_count >= XQ_MAX_MOVES;
                int win = NOCOLOR;
                if (over || type_of(cap) == GENERAL) {   // only now can the outcome change: rescan (rare)
                    const Summary e = summarize(b);
                    over = over || !(e.red_alive && e.black_alive);
                    win = e.winner;
                }
                tr.action = (uint16_t)a; tr.n_legal = (uint8_t)cnt; tr.reward = reward;
                tr.flags = (uint8_t)((over ? 1 : 0) | ((over ? win : NOCOLOR) << 1) | (cap << 4));
                st.steps++; st.legal_sum += cnt; st.reward_sum += reward;
                if (over) {
                    st.games++;
                    if (win == RED) st.red_wins++; else if (win == BLACK) st.black_wins++;
                    if (m.move_count < XQ_MAX_MOVES) st.cap_games++;
                    reset_board(b); m.reset(); mat_red = mat_black = 1480;
                }
            }
            if (trace)
                reinterpret_cast<uint2*>(trace)[(int64_t)p * n + env] =
                    make_uint2((uint32_t)tr.action | ((uint32_t)tr.n_legal << 16) | ((uint32_t)tr.flags << 24), (uint32_t)tr.reward);
        }
        b.store(envs + env);
        m.store(envs + env);
        if (mirror) { b.store(mirror + env); m.store(mirror + env); }
    }
    if (stats) {
        unsigned long long v[8] = {st.steps, st.games, st.red_wins, st.black_wins, st.cap_games, st.captures,
                                   (unsigned long long)st.reward_sum, st.legal_sum};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const unsigned long long r = warp_sum(v[i]);
            if ((tid & 31) == 0 && r != 0) atomicAdd(reinterpret_cast<unsigned long long*>(stats) + i, r);
        }
    }
}

}  // namespace xq

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace xq;

struct xq_env_s {
    int64_t n = 0;
    int device = 0;
    uint64_t seed = 0, env_id0 = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    xq_env_rec* d_envs = nullptr;
    xq_env_stats* d_stats = nullptr;
    // scratch for the host-pointer API
    uint8_t* d_u8[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // n bytes each
    uint16_t* d_actions = nullptr;    // n
    int32_t* d_i32 = nullptr;         // 4n
    uint32_t* d_lists = nullptr;      // n*64 words, allocated on first use
    xq_trace_rec* d_trace = nullptr; int64_t trace_cap = 0;
    double* d_state = nullptr;
    uint8_t* d_nonstd = nullptr;      // n flags written by the fused rollout and list kernels
    bool maybe_nonstd = false;        // set once boards were injected (xq_env_set_boards)
    // finished-game events of the self-play collector (xq_env_enable_game_events)
    xq_game_event* d_events = nullptr; unsigned long long* d_event_count = nullptr; int64_t event_cap = 0; uint32_t event_ply = 0;
    xq_game_event* h_events = nullptr; unsigned long long* h_event_count = nullptr; int64_t last_events = 0;      // pinned staging of the drain; size of the last drain
    // per-env scratch of the self-play collector (xq_selfplay.cu: Q(s) rows, chosen actions, auxiliary streams and events), released with the handle
    void* sp_scratch = nullptr; void (*sp_scratch_free)(void*) = nullptr;
    cudaEvent_t ev_io = nullptr; bool io_pending = false;      // xq_env_rollout_random_io_submit / _wait
    cudaStream_t io_in = nullptr, io_out = nullptr;            // its copy streams: boards in / results out move under the OTHER handle's kernel
    cudaEvent_t ev_in = nullptr, ev_run = nullptr, ev_prev = nullptr;
    bool async_dirty = false;                                   // asynchronous work on `stream` since the last synchronisation of the handle
};


namespace xq {
cudaError_t launch_rollout_team(xq_env_rec* envs, int64_t n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace,
                                xq_env_stats* stats, uint8_t* nonstd, cudaStream_t stream, const xq_env_rec* src, xq_env_rec* mirror);
cudaError_t launch_legal_moves_team(const xq_env_rec* envs, int64_t n, uint8_t* counts, uint32_t* actions, uint8_t* nonstd, cudaStream_t stream);
cudaError_t launch_rollout_lane(xq_env_rec* envs, int64_t n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace, xq_env_stats* stats,
                                uint8_t* nonstd, cudaStream_t stream, const xq_env_rec* src, xq_env_rec* mirror);
cudaError_t launch_legal_moves_lane(const xq_env_rec* envs, int64_t n, uint8_t* counts, uint32_t* actions, uint8_t* nonstd, cudaStream_t stream);
cudaError_t launch_pick_random(const xq_env_rec* envs, int64_t n, uint64_t env_id0, uint64_t seed, const uint8_t* counts, const uint16_t* lists, uint16_t* out,
                               cudaStream_t stream);
}
// ordered action lists of every env into h->d_u8[0] (counts) and h->d_lists ([n][128] u16): the register-resident kernel (xq_rollout_lane.cu)
// for every board with a standard piece set, then the generic thread-per-board kernel for the boards it flagged (only possible after
// xq_env_set_boards injected exotic positions).
static int launch_legal_moves(xq_env_s* h) {
    h->async_dirty = true;
    if (!h->d_lists) XQ_CUDA(cudaMalloc(&h->d_lists, sizeof(uint32_t) * 64 * h->n));
    // few envs: the team kernel (4 threads per board, a quarter of the per-thread chain); many: one thread per board.  XQ_LEGAL_TEAM=0|1 forces.
    // (read per call: the tests switch kernels inside one process)
    const char* te = getenv("XQ_LEGAL_TEAM");
    const int team_env = te ? atoi(te) : -1;
    const bool team = team_env >= 0 ? team_env != 0 : h->n <= 18944;      // 592 schedulers x 32: measured 12.3 against 14.4 us at 16,384 envs, 16.4 both at 24,576
    if (team) XQ_CUDA(launch_legal_moves_team(h->d_envs, h->n, h->d_u8[0], h->d_lists, h->d_nonstd, h->stream));
    else XQ_CUDA(launch_legal_moves_lane(h->d_envs, h->n, h->d_u8[0], h->d_lists, h->d_nonstd, h->stream));
    if (h->maybe_nonstd) {
        legal_moves_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, h->d_u8[0], h->d_lists, h->d_nonstd);
        XQ_LAUNCH_CHECK();
    }
    return XQ_OK;
}
// threads per board of the fused rollout kernel: 1 = rollout_lane_kernel (xq_rollout_lane.cu: the whole board in one thread's registers,
// no barrier, nothing replicated), the default above 9,472 envs (148 SMs x 64); 4 = rollout_team_kernel (xq_rollout_team.cu), the default below.
// XQ_ROLLOUT_TEAM=1|4 forces one (scripts/rollout_sweep.py re-measures the crossover).  Both are bit-identical.
// Measured on one B200 (steps/s, 200 / 200 / 100 / 32 plies per launch):   envs      4096     8192     16,384    65,536    1M
//   board per thread (1)                                                             2.98e9   5.94e9   1.17e10   1.61e10   1.83e10
//   team of 4 (4)                                                                    3.90e9   6.45e9   8.6e9     1.04e10   1.01e10
// Up to ~16k envs every warp sits alone on its scheduler and a launch lasts as long as ONE warp's plies: the team kernel's shorter
// per-thread ply (~700 instructions against ~1800) wins there; beyond that the kernels are issue-bound and the one that executes
// fewer instructions per env step (56 against 87 warp-instructions) wins.
static int rollout_team(int64_t n) {
    static const int forced = [] { const char* e = getenv("XQ_ROLLOUT_TEAM"); return e ? atoi(e) : 0; }();
    if (forced == 1 || forced == 4) return forced;
    return n <= 148 * 64 ? 4 : 1;      // up to two team CTAs (32 boards each) per SM; measured (env steps/s, team / lane): 4096 3.9e9 / 3.0e9, 8192 6.4e9 / 5.9e9, 10,240 6.6e9 / 7.4e9
}
// Fused rollout = lane or team kernel (xq_rollout_lane.cu, xq_rollout_team.cu) for every board with a standard piece set, then the generic
// thread-per-board kernel for the boards it flagged (only possible after xq_env_set_boards injected exotic positions).
// src / mirror (optional, xq_env_rollout_random_io with pinned host buffers): the kernels read the boards straight from MAPPED host memory and
// write the final boards to mapped host memory as well as to the device array -- no copy launches on the stream.  A board the first kernel leaves
// to the generic one is copied host -> device by the first kernel, so the generic kernel always starts from the device array.
static int launch_rollout(xq_env_s* h, int n_plies, xq_trace_rec* d_trace, const xq_env_rec* src = nullptr, xq_env_rec* mirror = nullptr) {
    if (n_plies >= (1 << 24)) return fail(XQ_ERR_INVALID, "rollout: n_plies must be < 2^24 per launch");
    h->async_dirty = true;
    if (rollout_team(h->n) == 1) XQ_CUDA(launch_rollout_lane(h->d_envs, h->n, h->env_id0, h->seed, n_plies, d_trace, h->d_stats, h->d_nonstd, h->stream, src, mirror));
    else XQ_CUDA(launch_rollout_team(h->d_envs, h->n, h->env_id0, h->seed, n_plies, d_trace, h->d_stats, h->d_nonstd, h->stream, src, mirror));
    if (h->maybe_nonstd) {
        rollout_random_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, h->env_id0, h->seed, n_plies, d_trace,
                                                                                    h->d_stats, h->d_nonstd, mirror);
        XQ_LAUNCH_CHECK();
    }
    return XQ_OK;
}
// device alias of a pinned, mapped, 16-byte aligned host buffer (cudaHostAlloc / cudaHostRegister under unified addressing), or null
static void* mapped_alias(const void* host) {
    if (!host || !aligned16(host)) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

namespace xq {
int env_info(xq_env_t h, EnvInfo* out) {
    if (!h || !out) return fail(XQ_ERR_INVALID, "env_info: null handle");
    h->async_dirty = true;      // the collector / trainer launch on the handle's stream and boards
    out->n = h->n; out->device = h->device; out->seed = h->seed; out->env_id0 = h->env_id0; out->stream = h->stream; out->d_envs = h->d_envs; out->d_stats = h->d_stats;
    out->d_events = h->d_events; out->d_event_count = h->d_event_count; out->event_cap = h->event_cap; out->event_ply = h->event_ply;
    out->d_nonstd = h->d_nonstd; out->maybe_nonstd = h->maybe_nonstd;
    return XQ_OK;
}
void env_advance_event_ply(xq_env_t h, uint32_t plies) { if (h) h->event_ply += plies; }
void env_boards_injected(xq_env_t h) { h->maybe_nonstd = true; }
void** env_scratch_slot(xq_env_t h, void (*free_fn)(void*)) { h->sp_scratch_free = free_fn; return &h->sp_scratch; }
}  // namespace xq

extern "C" {

const char* xq_last_error(void) { return last_error().c_str(); }
const char* xq_version(void) { return "xq-b200 0.1 (sm_100a)"; }
uint64_t xq_launch_count(void) { return g_launches; }
uint64_t xq_rng(uint64_t seed, uint64_t env_id, uint32_t ctr) { return rng(seed, env_id, ctr); }

uint32_t xq_eps_threshold(double eps) {
    const double rm = 2147483647.0;
    if (!(eps > 0.0)) return 0;
    if (eps > 1.0) return 0x80000000u;
    long long t = (long long)(eps * rm);
    while (t > 0 && !((double)(t - 1) / rm < eps)) --t;
    while (t <= 2147483647LL && ((double)t / rm < eps)) ++t;
    return (uint32_t)t;
}

int xq_device_count(int* count) {
    if (!count) return fail(XQ_ERR_INVALID, "xq_device_count: null pointer");
    XQ_CUDA(cudaGetDeviceCount(count));
    return XQ_OK;
}

int xq_env_destroy(xq_env_t h) {
    if (!h) return XQ_OK;
    cudaSetDevice(h->device);
    if (h->sp_scratch && h->sp_scratch_free) { cudaStreamSynchronize(h->stream); h->sp_scratch_free(h->sp_scratch); }
    if (h->io_pending && h->ev_io) cudaEventSynchronize(h->ev_io);      // a submission never waited for: its copies may still be in flight
    if (h->ev_io) cudaEventDestroy(h->ev_io);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_run) cudaEventDestroy(h->ev_run);
    if (h->ev_prev) cudaEventDestroy(h->ev_prev);
    if (h->io_in) cudaStreamDestroy(h->io_in);
    if (h->io_out) cudaStreamDestroy(h->io_out);
    cudaFree(h->d_envs); cudaFree(h->d_stats); cudaFree(h->d_actions); cudaFree(h->d_i32); cudaFree(h->d_lists);
    cudaFree(h->d_trace); cudaFree(h->d_state); cudaFree(h->d_nonstd); cudaFree(h->d_events); cudaFree(h->d_event_count); cudaFreeHost(h->h_events); cudaFreeHost(h->h_event_count);
    for (auto p : h->d_u8) cudaFree(p);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return XQ_OK;
}

int xq_env_create(int64_t n_envs, int device, uint64_t seed, uint64_t env_id0, xq_env_t* out) {
    if (!out || n_envs <= 0) return fail(XQ_ERR_INVALID, "xq_env_create: n_envs must be > 0 and out non-null");
    int ndev = 0;
    XQ_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(XQ_ERR_INVALID, "xq_env_create: device %d out of range (%d devices)", device, ndev);
    XQ_CUDA(cudaSetDevice(device));
    xq_env_s* h = new (std::nothrow) xq_env_s();
    if (!h) return fail(XQ_ERR_NOMEM, "xq_env_create: out of host memory");
    h->n = n_envs; h->device = device; h->seed = seed; h->env_id0 = env_id0;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    h->own_stream = (e == cudaSuccess);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_envs, sizeof(xq_env_rec) * n_envs);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_stats, sizeof(xq_env_stats));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_actions, sizeof(uint16_t) * n_envs);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_i32, sizeof(int32_t) * 4 * n_envs);
    for (auto& p : h->d_u8) if (e == cudaSuccess) e = cudaMalloc(&p, (size_t)n_envs);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_nonstd, (size_t)n_envs);
    if (e == cudaSuccess) e = cudaMemsetAsync(h->d_stats, 0, sizeof(xq_env_stats), h->stream);
    if (e != cudaSuccess) { xq_env_destroy(h); return fail(XQ_ERR_CUDA, "xq_env_create: %s", cudaGetErrorString(e)); }
    reset_kernel<<<grid_of(4 * n_envs, 256), 256, 0, h->stream>>>(h->d_envs, n_envs, nullptr, 1);
    ++g_launches;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { xq_env_destroy(h); return fail(XQ_ERR_CUDA, "xq_env_create: reset kernel: %s", cudaGetErrorString(e)); }
    *out = h;
    return XQ_OK;
}

#define XQ_ENV_ENTER_IO(h)                                                     \
    if (!(h)) return fail(XQ_ERR_INVALID, "%s: null handle", __func__);        \
    XQ_CUDA(cudaSetDevice((h)->device))
// between xq_env_rollout_random_io_submit and _wait the handle's boards and buffers are in flight on its copy streams: every other call is refused
#define XQ_ENV_ENTER(h)                                                        \
    XQ_ENV_ENTER_IO(h);                                                        \
    if ((h)->io_pending) return fail(XQ_ERR_STATE, "%s: a submission of this handle has not been waited for (xq_env_rollout_random_io_wait)", __func__)

int xq_env_count(xq_env_t h, int64_t* n) { if (!h || !n) return fail(XQ_ERR_INVALID, "xq_env_count: null"); *n = h->n; return XQ_OK; }

int xq_env_set_stream(xq_env_t h, void* s) {
    XQ_ENV_ENTER(h);
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    if (h->own_stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    h->stream = (cudaStream_t)s;
    return XQ_OK;
}
int xq_env_sync(xq_env_t h) { XQ_ENV_ENTER(h); XQ_CUDA(cudaStreamSynchronize(h->stream)); return XQ_OK; }
int xq_env_device_boards(xq_env_t h, void** p) { if (!h || !p) return fail(XQ_ERR_INVALID, "xq_env_device_boards: null"); h->async_dirty = true; *p = h->d_envs; return XQ_OK; }

int xq_env_reset(xq_env_t h, const uint8_t* mask_host) {
    XQ_ENV_ENTER(h);
    if (mask_host) XQ_CUDA(cudaMemcpyAsync(h->d_u8[0], mask_host, (size_t)h->n, cudaMemcpyHostToDevice, h->stream));
    reset_kernel<<<grid_of(4 * h->n, 256), 256, 0, h->stream>>>(h->d_envs, h->n, mask_host ? h->d_u8[0] : nullptr, 0);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_set_boards(xq_env_t h, const xq_env_rec* recs, int64_t first, int64_t n) {
    XQ_ENV_ENTER(h);
    if (!recs || first < 0 || n < 0 || first + n > h->n) return fail(XQ_ERR_INVALID, "xq_env_set_boards: range [%lld,+%lld) outside %lld envs", (long long)first, (long long)n, (long long)h->n);
    XQ_CUDA(cudaMemcpyAsync(h->d_envs + first, recs, sizeof(xq_env_rec) * n, cudaMemcpyHostToDevice, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    h->maybe_nonstd = true;
    return XQ_OK;
}
int xq_env_get_boards(xq_env_t h, xq_env_rec* recs, int64_t first, int64_t n) {
    XQ_ENV_ENTER(h);
    if (!recs || first < 0 || n < 0 || first + n > h->n) return fail(XQ_ERR_INVALID, "xq_env_get_boards: range [%lld,+%lld) outside %lld envs", (long long)first, (long long)n, (long long)h->n);
    XQ_CUDA(cudaMemcpyAsync(recs, h->d_envs + first, sizeof(xq_env_rec) * n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_legal_moves(xq_env_t h, uint8_t* counts_host, xq_action* actions_host) {
    XQ_ENV_ENTER(h);
    if (!counts_host || !actions_host) return fail(XQ_ERR_INVALID, "xq_env_legal_moves: null output");
    if (int rc = launch_legal_moves(h)) return rc;
    XQ_CUDA(cudaMemcpyAsync(counts_host, h->d_u8[0], (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaMemcpyAsync(actions_host, h->d_lists, sizeof(uint32_t) * 64 * h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_legal_moves_strict(xq_env_t h, uint8_t* counts_host, xq_action* actions_host) {
    XQ_ENV_ENTER(h);
    if (!counts_host || !actions_host) return fail(XQ_ERR_INVALID, "xq_env_legal_moves_strict: null output");
    if (!h->d_lists) XQ_CUDA(cudaMalloc(&h->d_lists, sizeof(uint32_t) * 64 * h->n));
    legal_moves_strict_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, h->d_u8[0], h->d_lists);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaMemcpyAsync(counts_host, h->d_u8[0], (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaMemcpyAsync(actions_host, h->d_lists, sizeof(uint32_t) * 64 * h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_valid_moves(xq_env_t h, int row, int col, uint8_t* counts_host, uint8_t* to_host) {
    XQ_ENV_ENTER(h);
    if (!counts_host || !to_host) return fail(XQ_ERR_INVALID, "xq_env_valid_moves: null output");
    if (!h->d_lists) XQ_CUDA(cudaMalloc(&h->d_lists, sizeof(uint32_t) * 64 * h->n));
    valid_moves_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, row, col, h->d_u8[0], reinterpret_cast<uint8_t*>(h->d_lists));
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaMemcpyAsync(counts_host, h->d_u8[0], (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaMemcpyAsync(to_host, h->d_lists, (size_t)20 * h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_is_valid_move(xq_env_t h, const int32_t* moves_host, uint8_t* valid_host) {
    XQ_ENV_ENTER(h);
    if (!moves_host || !valid_host) return fail(XQ_ERR_INVALID, "xq_env_is_valid_move: null pointer");
    XQ_CUDA(cudaMemcpyAsync(h->d_i32, moves_host, sizeof(int32_t) * 4 * h->n, cudaMemcpyHostToDevice, h->stream));
    is_valid_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, reinterpret_cast<const int4*>(h->d_i32), h->d_u8[0]);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaMemcpyAsync(valid_host, h->d_u8[0], (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_step(xq_env_t h, const xq_action* actions_host, int32_t* reward_host, uint8_t* done_host, uint8_t* winner_host,
                uint8_t* captured_host, uint8_t* valid_host, int auto_reset) {
    XQ_ENV_ENTER(h);
    if (!actions_host) return fail(XQ_ERR_INVALID, "xq_env_step: null actions");
    XQ_CUDA(cudaMemcpyAsync(h->d_actions, actions_host, sizeof(uint16_t) * h->n, cudaMemcpyHostToDevice, h->stream));
    step_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, h->d_actions, h->d_i32, h->d_u8[0], h->d_u8[1],
                                                                      h->d_u8[2], h->d_u8[3], auto_reset);
    XQ_LAUNCH_CHECK();
    if (reward_host) XQ_CUDA(cudaMemcpyAsync(reward_host, h->d_i32, sizeof(int32_t) * h->n, cudaMemcpyDeviceToHost, h->stream));
    uint8_t* outs[4] = {done_host, winner_host, captured_host, valid_host};
    for (int i = 0; i < 4; ++i)
        if (outs[i]) XQ_CUDA(cudaMemcpyAsync(outs[i], h->d_u8[i], (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_legal_moves_device(xq_env_t h, void** counts_dev, void** actions_dev) {
    XQ_ENV_ENTER(h);
    if (int rc = launch_legal_moves(h)) return rc;
    if (counts_dev) *counts_dev = h->d_u8[0];
    if (actions_dev) *actions_dev = h->d_lists;
    return XQ_OK;
}

int xq_env_pick_random_device(xq_env_t h, void** actions_dev) {
    XQ_ENV_ENTER(h);
    if (!h->d_lists) return fail(XQ_ERR_STATE, "xq_env_pick_random_device: call xq_env_legal_moves_device first");
    XQ_CUDA(launch_pick_random(h->d_envs, h->n, h->env_id0, h->seed, h->d_u8[0], reinterpret_cast<const uint16_t*>(h->d_lists), h->d_actions, h->stream));
    if (actions_dev) *actions_dev = h->d_actions;
    return XQ_OK;
}

int xq_env_step_device(xq_env_t h, const void* actions_dev, int auto_reset, void** reward_dev, void** done_dev, void** winner_dev, void** captured_dev,
                       void** valid_dev) {
    XQ_ENV_ENTER(h);
    const uint16_t* a = actions_dev ? static_cast<const uint16_t*>(actions_dev) : h->d_actions;
    h->async_dirty = true;
    step_kernel<<<grid_of(h->n, kThreads), kThreads, 0, h->stream>>>(h->d_envs, h->n, a, h->d_i32, h->d_u8[1], h->d_u8[2], h->d_u8[3], h->d_u8[4], auto_reset);
    XQ_LAUNCH_CHECK();
    if (reward_dev) *reward_dev = h->d_i32;
    if (done_dev) *done_dev = h->d_u8[1];
    if (winner_dev) *winner_dev = h->d_u8[2];
    if (captured_dev) *captured_dev = h->d_u8[3];
    if (valid_dev) *valid_dev = h->d_u8[4];
    return XQ_OK;
}

int xq_env_rollout_random_async(xq_env_t h, int n_plies) {
    XQ_ENV_ENTER(h);
    if (n_plies < 0) return fail(XQ_ERR_INVALID, "xq_env_rollout_random_async: n_plies < 0");
    if (int rc = launch_rollout(h, n_plies, nullptr)) return rc;
    return XQ_OK;
}

static int reserve_trace(xq_env_s* h, int64_t need) {
    if (need > h->trace_cap) {
        cudaFree(h->d_trace); h->d_trace = nullptr; h->trace_cap = 0;
        XQ_CUDA(cudaMalloc(&h->d_trace, sizeof(xq_trace_rec) * need));
        h->trace_cap = need;
    }
    return XQ_OK;
}

int xq_env_rollout_random_traced_async(xq_env_t h, int n_plies, void** trace_dev) {
    XQ_ENV_ENTER(h);
    if (n_plies < 0) return fail(XQ_ERR_INVALID, "xq_env_rollout_random_traced_async: n_plies < 0");
    if (int rc = reserve_trace(h, (int64_t)n_plies * h->n)) return rc;
    if (int rc = launch_rollout(h, n_plies, h->d_trace)) return rc;
    if (trace_dev) *trace_dev = h->d_trace;
    return XQ_OK;
}

int xq_env_get_stats(xq_env_t h, xq_env_stats* stats_host, int reset) {
    XQ_ENV_ENTER(h);
    if (stats_host) XQ_CUDA(cudaMemcpyAsync(stats_host, h->d_stats, sizeof(xq_env_stats), cudaMemcpyDeviceToHost, h->stream));
    if (reset) XQ_CUDA(cudaMemsetAsync(h->d_stats, 0, sizeof(xq_env_stats), h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_env_enable_game_events(xq_env_t h, int64_t capacity) {
    XQ_ENV_ENTER(h);
    if (capacity <= 0) return fail(XQ_ERR_INVALID, "xq_env_enable_game_events: capacity must be > 0");
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    if (capacity != h->event_cap) {
        cudaFree(h->d_events); cudaFree(h->d_event_count); cudaFreeHost(h->h_events); cudaFreeHost(h->h_event_count);
        h->d_events = nullptr; h->d_event_count = nullptr; h->h_events = nullptr; h->h_event_count = nullptr; h->event_cap = 0;
        XQ_CUDA(cudaMalloc(&h->d_events, sizeof(xq_game_event) * capacity));
        XQ_CUDA(cudaMalloc(&h->d_event_count, sizeof(unsigned long long)));
        XQ_CUDA(cudaHostAlloc(&h->h_events, sizeof(xq_game_event) * capacity, cudaHostAllocDefault));
        XQ_CUDA(cudaHostAlloc(&h->h_event_count, sizeof(unsigned long long), cudaHostAllocDefault));
    }
    XQ_CUDA(cudaMemset(h->d_event_count, 0, sizeof(unsigned long long)));
    h->event_cap = capacity; h->event_ply = 0; h->last_events = 0;
    return XQ_OK;
}

int xq_env_drain_game_events(xq_env_t h, xq_game_event* out_host, int64_t max_events, int64_t* n_out, int64_t* n_dropped) {
    XQ_ENV_ENTER(h);
    if (!h->d_events) return fail(XQ_ERR_STATE, "xq_env_drain_game_events: call xq_env_enable_game_events first");
    if (!out_host || !n_out || max_events < h->event_cap) return fail(XQ_ERR_INVALID, "xq_env_drain_game_events: the output must hold the ring's capacity");
    // one synchronisation in the common case: the counter and a prefix of the ring sized from the previous drain travel together into
    // pinned staging memory; only a drain that turns out to be larger than the guess needs a second copy
    const int64_t guess = std::min<int64_t>(h->event_cap, std::max<int64_t>(1024, 2 * h->last_events));
    XQ_CUDA(cudaMemcpyAsync(h->h_event_count, h->d_event_count, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaMemcpyAsync(h->h_events, h->d_events, sizeof(xq_game_event) * guess, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaMemsetAsync(h->d_event_count, 0, sizeof(unsigned long long), h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    const unsigned long long count = *h->h_event_count;
    const int64_t n = (int64_t)count < h->event_cap ? (int64_t)count : h->event_cap;
    if (n > guess) {      // the ring keeps its contents until the next collector ply writes into it
        XQ_CUDA(cudaMemcpyAsync(h->h_events + guess, h->d_events + guess, sizeof(xq_game_event) * (n - guess), cudaMemcpyDeviceToHost, h->stream));
        XQ_CUDA(cudaStreamSynchronize(h->stream));
    }
    memcpy(out_host, h->h_events, sizeof(xq_game_event) * n);
    h->last_events = n;
    // slots were claimed with an atomic counter: restore the order of the batched loop, (ply, env)
    std::sort(out_host, out_host + n, [](const xq_game_event& a, const xq_game_event& b) { return a.ply != b.ply ? a.ply < b.ply : a.env < b.env; });
    *n_out = n;
    if (n_dropped) *n_dropped = (int64_t)count - n;
    return XQ_OK;
}

// side_streams: the copies run on the handle's own copy streams, ordered against the rollout by events -- with two handles alternating on one
// compute stream the boards of the next step arrive and the results of the previous step leave while the other handle's kernel runs.
// Otherwise (the one-call form) pinned buffers are read / written by the rollout kernel itself through mapped memory: no copy launches at all.
static int rollout_io_enqueue(xq_env_s* h, const xq_env_rec* boards_in_host, int n_plies, xq_env_rec* boards_out_host, xq_trace_rec* trace_host,
                              xq_env_stats* stats_host, bool side_streams) {
    if (n_plies < 0) return fail(XQ_ERR_INVALID, "xq_env_rollout_random: n_plies < 0");
    if (h->io_pending) return fail(XQ_ERR_STATE, "xq_env_rollout_random_io_submit: the previous submission of this handle has not been waited for");
    if (!h->ev_io) XQ_CUDA(cudaEventCreateWithFlags(&h->ev_io, cudaEventDisableTiming));
    const int64_t need = (int64_t)n_plies * h->n;
    if (trace_host) if (int rc = reserve_trace(h, need)) return rc;
    if (side_streams) {
        if (!h->io_in) {
            XQ_CUDA(cudaStreamCreateWithFlags(&h->io_in, cudaStreamNonBlocking)); XQ_CUDA(cudaStreamCreateWithFlags(&h->io_out, cudaStreamNonBlocking));
            XQ_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming)); XQ_CUDA(cudaEventCreateWithFlags(&h->ev_run, cudaEventDisableTiming));
            XQ_CUDA(cudaEventCreateWithFlags(&h->ev_prev, cudaEventDisableTiming));
        }
        if (boards_in_host) {
            if (h->async_dirty) {      // asynchronous device-resident calls on this handle since its last synchronisation may still use the boards
                XQ_CUDA(cudaEventRecord(h->ev_prev, h->stream));
                XQ_CUDA(cudaStreamWaitEvent(h->io_in, h->ev_prev, 0));
            }
            XQ_CUDA(cudaMemcpyAsync(h->d_envs, boards_in_host, sizeof(xq_env_rec) * h->n, cudaMemcpyHostToDevice, h->io_in));
            XQ_CUDA(cudaEventRecord(h->ev_in, h->io_in));
            XQ_CUDA(cudaStreamWaitEvent(h->stream, h->ev_in, 0));
            h->maybe_nonstd = true;
        }
        XQ_CUDA(cudaMemsetAsync(h->d_stats, 0, sizeof(xq_env_stats), h->stream));
        if (int rc = launch_rollout(h, n_plies, trace_host ? h->d_trace : nullptr)) return rc;
        XQ_CUDA(cudaEventRecord(h->ev_run, h->stream));
        XQ_CUDA(cudaStreamWaitEvent(h->io_out, h->ev_run, 0));
        if (boards_out_host) XQ_CUDA(cudaMemcpyAsync(boards_out_host, h->d_envs, sizeof(xq_env_rec) * h->n, cudaMemcpyDeviceToHost, h->io_out));
        if (trace_host) XQ_CUDA(cudaMemcpyAsync(trace_host, h->d_trace, sizeof(xq_trace_rec) * need, cudaMemcpyDeviceToHost, h->io_out));
        if (stats_host) XQ_CUDA(cudaMemcpyAsync(stats_host, h->d_stats, sizeof(xq_env_stats), cudaMemcpyDeviceToHost, h->io_out));
        XQ_CUDA(cudaEventRecord(h->ev_io, h->io_out));
        h->io_pending = true;      // nothing else may be called on the handle until _wait: the copies out are not ordered against the compute stream
        return XQ_OK;
    }
    // pinned (mapped) host buffers are read / written by the rollout kernel itself: two copy launches less on the stream
    const xq_env_rec* src = static_cast<const xq_env_rec*>(mapped_alias(boards_in_host));
    xq_env_rec* mirror = static_cast<xq_env_rec*>(mapped_alias(boards_out_host));
    if (boards_in_host) {
        if (!src) XQ_CUDA(cudaMemcpyAsync(h->d_envs, boards_in_host, sizeof(xq_env_rec) * h->n, cudaMemcpyHostToDevice, h->stream));
        h->maybe_nonstd = true;
    }
    XQ_CUDA(cudaMemsetAsync(h->d_stats, 0, sizeof(xq_env_stats), h->stream));
    if (int rc = launch_rollout(h, n_plies, trace_host ? h->d_trace : nullptr, src, mirror)) return rc;
    if (boards_out_host && !mirror) XQ_CUDA(cudaMemcpyAsync(boards_out_host, h->d_envs, sizeof(xq_env_rec) * h->n, cudaMemcpyDeviceToHost, h->stream));
    if (trace_host) XQ_CUDA(cudaMemcpyAsync(trace_host, h->d_trace, sizeof(xq_trace_rec) * need, cudaMemcpyDeviceToHost, h->stream));
    if (stats_host) XQ_CUDA(cudaMemcpyAsync(stats_host, h->d_stats, sizeof(xq_env_stats), cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaEventRecord(h->ev_io, h->stream));
    h->io_pending = true;
    return XQ_OK;
}
int xq_env_rollout_random_io_submit(xq_env_t h, const xq_env_rec* boards_in_host, int n_plies, xq_env_rec* boards_out_host,
                                    xq_trace_rec* trace_host, xq_env_stats* stats_host) {
    XQ_ENV_ENTER(h);
    return rollout_io_enqueue(h, boards_in_host, n_plies, boards_out_host, trace_host, stats_host, true);
}
int xq_env_rollout_random_io_wait(xq_env_t h) {
    XQ_ENV_ENTER_IO(h);
    if (!h->io_pending) return fail(XQ_ERR_STATE, "xq_env_rollout_random_io_wait: nothing was submitted on this handle");
    h->io_pending = false;
    XQ_CUDA(cudaEventSynchronize(h->ev_io));
    h->async_dirty = false;
    return XQ_OK;
}
int xq_env_rollout_random_io(xq_env_t h, const xq_env_rec* boards_in_host, int n_plies, xq_env_rec* boards_out_host,
                             xq_trace_rec* trace_host, xq_env_stats* stats_host) {
    XQ_ENV_ENTER(h);
    if (int rc = rollout_io_enqueue(h, boards_in_host, n_plies, boards_out_host, trace_host, stats_host, false)) return rc;
    return xq_env_rollout_random_io_wait(h);
}
int xq_env_rollout_random(xq_env_t h, int n_plies, xq_trace_rec* trace_host, xq_env_stats* stats_host) {
    return xq_env_rollout_random_io(h, nullptr, n_plies, nullptr, trace_host, stats_host);
}

int xq_env_state_onehot(xq_env_t h, double* out_host) {
    XQ_ENV_ENTER(h);
    if (!out_host) return fail(XQ_ERR_INVALID, "xq_env_state_onehot: null output");
    if (!h->d_state) XQ_CUDA(cudaMalloc(&h->d_state, sizeof(double) * XQ_STATE_SIZE * h->n));
    state_onehot_kernel<<<grid_of(32 * h->n, 256), 256, 0, h->stream>>>(h->d_envs, h->n, h->d_state);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaMemcpyAsync(out_host, h->d_state, sizeof(double) * XQ_STATE_SIZE * h->n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

}  // extern "C"
