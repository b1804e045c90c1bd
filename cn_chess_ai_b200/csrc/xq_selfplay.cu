// xq_selfplay.cu -- GPU-resident replay buffer, batched epsilon-greedy action selection and the
// self-play collection loop (BASELINE configs 3 and 4).
//
// Reference semantics per transition = the body of ChessAI::train (src/chessai.cpp:96-131):
//   validActions = getAllValidActions(player)           (:98,  :347-368)
//   a = dqn->selectAction(state, 0.1, validActions)      (:106, src/dqn.cpp:24-56)
//   movePiece; reward = evaluateBoard(mover, moveCount)  (:113-116)
//   done = checkGameOver() || moveCount+1 >= 200         (:119)
// The reference then trains on that single transition at once; here it is appended to a replay ring in
// HBM and consumed in batches by the tensor-core TD update (xq_dqn_fast.cu).
// Q(s)[to] only needs outputs 0..89 of layer 1 (src/dqn.cpp:47 indexes by action.to), so acting costs the
// layer-0 sums -- carried from ply to ply in fixed point (xq_act_l0.cuh), 2-3 row updates per ply instead of a
// <=32-row gather -- plus a [n x 128] x [128 x 96] split-precision tensor-core contraction (dqn_q90_device in
// xq_dqn_fast.cu), then a team of 4 threads per board picks and applies the action (xq_act_team.cu).
#include <stdlib.h>

#include <algorithm>

#include "xq_act_l0.cuh"
#include "xq_dqn_internal.cuh"
#include "xq_env_dev.cuh"

namespace xq {

constexpr int kQPad = 96;      // Q(s)[0..95] per env, row-major (dqn_q90_device)

struct Transition {
    uint32_t s[12], s2[12];
    uint16_t action; uint8_t mover, done;
    int32_t reward;
    uint32_t pad[6];
};
static_assert(sizeof(Transition) == sizeof(xq_transition), "transition layout");

cudaError_t launch_act_team(bool apply, xq_env_rec* envs, int64_t n, uint64_t env_id0, uint64_t seed, const float* q90, uint32_t eps_thr, int train_done,
                            uint16_t* actions_out, void* ring, int64_t ring_cap, int64_t ring_pos, xq_env_stats* stats, xq_game_event* events,
                            unsigned long long* event_count, int64_t event_cap, uint32_t event_ply, uint8_t* nonstd, const ActCarry* carry, uint32_t event_env0, cudaStream_t stream);

// Action selection (+ optional application), generic thread-per-board version (ordered list staged in shared memory): the fallback
// of act_team_kernel (xq_act_team.cu) for boards with non-standard piece sets.
template <bool APPLY>
__global__ void __launch_bounds__(kThreads) act_kernel(xq_env_rec* __restrict__ envs, int64_t n, uint64_t env_id0, uint64_t seed,
                                                      const float* __restrict__ q90, uint32_t eps_thr, int train_done,
                                                      uint16_t* __restrict__ actions_out, Transition* __restrict__ ring, int64_t ring_cap,
                                                      int64_t ring_pos, xq_env_stats* __restrict__ stats, xq_game_event* __restrict__ events,
                                                      unsigned long long* __restrict__ event_count, int64_t event_cap, uint32_t event_ply,
                                                      const uint8_t* __restrict__ only) {
    __shared__ uint32_t s_board[12 * kThreads];
    __shared__ uint32_t s_list[64 * kThreads];
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * kThreads + tid;
    unsigned long long a_steps = 0, a_games = 0, a_red = 0, a_black = 0, a_capg = 0, a_caps = 0, a_legal = 0;
    long long a_reward = 0;
    if (env < n && (only == nullptr || only[env] != 0)) {   // `only`: boards the team kernel could not map
        SmemBoard b{s_board + tid, kThreads};
        b.load(envs + env);
        Meta m; m.load(envs + env);
        Summary s = summarize(b);
        if (APPLY && (m.move_count >= XQ_MAX_MOVES || !(s.red_alive && s.black_alive))) { reset_board(b); m.reset(); s = summarize(b); }
        uint16_t* list = reinterpret_cast<uint16_t*>(s_list);
        int cnt = 0;
        all_actions(b, m.player, [&](int from, int to) {
            if (cnt < XQ_MAX_ACTIONS) { list[(cnt >> 1) * 2 * kThreads + 2 * tid + (cnt & 1)] = XQ_ACTION(from, to); ++cnt; }
        });
        int a = XQ_ACTION_NONE;
        if (cnt > 0) {
            const uint64_t x = rng(seed, env_id0 + (uint64_t)env, m.ctr);
            const uint32_t coin31 = (uint32_t)(x & 0x7FFFFFFFu), idx31 = (uint32_t)(x >> 33);
            int k = 0;
            if (coin31 < eps_thr) {                                     // rand()/RAND_MAX < epsilon (src/dqn.cpp:30-34)
                k = (int)(idx31 % (uint32_t)cnt);
            } else {                                                    // first valid action maximising Q[action.to] (:39-52)
                const float* q = q90 + env * kQPad;
                float best = -INFINITY;
                for (int i = 0; i < cnt; ++i) {
                    const float v = q[XQ_ACTION_TO(list[(i >> 1) * 2 * kThreads + 2 * tid + (i & 1)])];
                    if (v > best) { best = v; k = i; }
                }
            }
            a = list[(k >> 1) * 2 * kThreads + 2 * tid + (k & 1)];
        }
        if (actions_out) actions_out[env] = (uint16_t)a;
        if (APPLY) {
            Transition t;
#pragma unroll
            for (int i = 0; i < 12; ++i) t.s[i] = b.base[i * kThreads];
            t.mover = (uint8_t)m.player;
            if (cnt == 0) {   // no action: the episode loop ends (chessai.cpp:100-103); recorded as a terminal null transition
                t.action = 0; t.done = 1; t.reward = 0;
#pragma unroll
                for (int i = 0; i < 12; ++i) t.s2[i] = t.s[i];
                if (events) {   // the episode loop breaks without a move (chessai.cpp:100-103); gameCompleted still fires (:161)
                    const unsigned long long slot = atomicAdd(event_count, 1ull);
                    if ((int64_t)slot < event_cap)
                        events[slot] = xq_game_event{event_ply, (uint32_t)env, m.red_score, m.black_score, (uint16_t)m.move_count, (uint8_t)s.winner, 2, 0u};
                }
                reset_board(b); m.reset(); m.ctr++; a_games++;
            } else {
                const int mover = m.player;
                const int cap = apply_move(b, m, XQ_ACTION_FROM(a), XQ_ACTION_TO(a));
                m.ctr++;
                int mat_red = s.mat_red, mat_black = s.mat_black;
                if (cap != 0) { const int sc = piece_score(type_of(cap)); if (cap >= 8) mat_black -= sc; else mat_red -= sc; a_caps++; }
                const int reward = reward_from_material(mover == RED ? mat_red - mat_black : mat_black - mat_red, m.move_count);
                bool over = m.move_count >= XQ_MAX_MOVES;
                int win = NOCOLOR;
                if (over || type_of(cap) == GENERAL) { const Summary e2 = summarize(b); over = over || !(e2.red_alive && e2.black_alive); win = e2.winner; }
#pragma unroll
                for (int i = 0; i < 12; ++i) t.s2[i] = b.base[i * kThreads];
                t.action = (uint16_t)a; t.reward = reward;
                t.done = (uint8_t)((over || (train_done && m.move_count + 1 >= XQ_MAX_MOVES)) ? 1 : 0);     // chessai.cpp:119 / :227
                a_steps++; a_legal += cnt; a_reward += reward;
                if (over) {
                    a_games++;
                    if (win == RED) a_red++; else if (win == BLACK) a_black++;
                    if (m.move_count < XQ_MAX_MOVES) a_capg++;
                    if (events) {   // gameCompleted(game, board->getRedScore(), board->getBlackScore()), chessai.cpp:161
                        const unsigned long long slot = atomicAdd(event_count, 1ull);
                        if ((int64_t)slot < event_cap)
                            events[slot] = xq_game_event{event_ply, (uint32_t)env, m.red_score, m.black_score, (uint16_t)m.move_count, (uint8_t)win,
                                                         (uint8_t)(type_of(cap) == GENERAL ? 0 : 1), 0u};
                    }
                    reset_board(b); m.reset();
                }
            }
            if (ring) {
#pragma unroll
                for (int i = 0; i < 6; ++i) t.pad[i] = 0;
                uint4* dst = reinterpret_cast<uint4*>(ring + (ring_pos + env) % ring_cap);
                const uint4* src = reinterpret_cast<const uint4*>(&t);
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = src[i];
            }
            b.store(envs + env);
            m.store(envs + env);
        }
    }
    if (APPLY && stats) {
        unsigned long long v[8] = {a_steps, a_games, a_red, a_black, a_capg, a_caps, (unsigned long long)a_reward, a_legal};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            unsigned long long r = v[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
            if ((tid & 31) == 0 && r != 0) atomicAdd(reinterpret_cast<unsigned long long*>(stats) + i, r);
        }
    }
}

// uniform sampling with replacement: warp per sample copies one 128-byte record
__global__ void __launch_bounds__(256) sample_kernel(const Transition* __restrict__ ring, int64_t size, int64_t batch, uint64_t seed,
                                                    uint32_t counter, Transition* __restrict__ out, int64_t* __restrict__ index_out) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= batch) return;
    const int64_t idx = (int64_t)((rng(seed, (uint64_t)i, counter) >> 1) % (uint64_t)size);
    if (lane < 8) reinterpret_cast<uint4*>(out + i)[lane] = reinterpret_cast<const uint4*>(ring + idx)[lane];
    if (lane == 0 && index_out) index_out[i] = idx;
}

}  // namespace xq

using namespace xq;

struct xq_replay_s {
    int64_t capacity = 0, total = 0;      // total transitions ever inserted; head = total % capacity
    int device = 0;
    Transition* d_ring = nullptr;
    Transition* d_batch = nullptr; int64_t batch_cap = 0;
    int64_t* d_index = nullptr;
    cudaStream_t stream = nullptr;        // for the host-pointer entry points
    cudaEvent_t ev = nullptr;
};

// Scratch of the collector / xq_dqn_act, OWNED BY THE ENV HANDLE (two env handles on one device -- on different streams, or driven by two
// host threads -- never share Q(s) rows, action buffers, the auxiliary stream or fork / join events), released with it.
struct SelfplayScratch {
    float* q90 = nullptr; int64_t cap = 0; uint16_t* actions = nullptr;
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_order = nullptr;
};
static void free_scratch(void* p) {
    SelfplayScratch* s = static_cast<SelfplayScratch*>(p);
    cudaFree(s->q90); cudaFree(s->actions);
    if (s->aux) cudaStreamDestroy(s->aux);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_order) cudaEventDestroy(s->ev_order);
    delete s;
}

static inline unsigned blocks(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }
static int reserve_scratch(xq_env_t env, int64_t n, SelfplayScratch** out) {
    void** slot = env_scratch_slot(env, free_scratch);
    if (!*slot) {
        *slot = new (std::nothrow) SelfplayScratch();
        if (!*slot) return fail(XQ_ERR_NOMEM, "out of host memory");
    }
    SelfplayScratch& s = *static_cast<SelfplayScratch*>(*slot);
    if (n > s.cap) {        // only ever grows on the env's own stream, after the work that used the old buffers
        cudaFree(s.q90); cudaFree(s.actions); s.q90 = nullptr; s.actions = nullptr; s.cap = 0;
        XQ_CUDA(cudaMalloc(&s.q90, sizeof(float) * kQPad * n));
        XQ_CUDA(cudaMalloc(&s.actions, sizeof(uint16_t) * n));
        s.cap = n;
    }
    *out = &s;
    return XQ_OK;
}
// make `waiter` see everything already enqueued on `producer`
static int order_after(cudaStream_t waiter, cudaStream_t producer, cudaEvent_t* ev) {
    if (waiter == producer) return XQ_OK;
    if (!*ev) XQ_CUDA(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
    XQ_CUDA(cudaEventRecord(*ev, producer));
    XQ_CUDA(cudaStreamWaitEvent(waiter, *ev, 0));
    return XQ_OK;
}

// One ply of selection (+ application) for every env: the team kernel (xq_act_team.cu) for boards with a standard piece set, then
// the generic thread-per-board kernel for the boards it flagged (only possible after xq_env_set_boards injected exotic positions).
// (A board-per-thread act kernel measured 74.7 us per ply against 60.5 at 65,536 envs: DESIGN.md section 4.)
static int launch_act(bool apply, const EnvInfo& ei, const float* q90, uint32_t thr, int train_done, uint16_t* actions, Transition* ring, int64_t ring_cap,
                      int64_t ring_pos, xq_env_stats* stats, uint32_t event_ply, const ActCarry* carry = nullptr, uint32_t event_env0 = 0) {
    XQ_CUDA(launch_act_team(apply, ei.d_envs, ei.n, ei.env_id0, ei.seed, q90, thr, train_done, actions, ring, ring_cap, ring_pos, stats,
                            ei.d_events, ei.d_event_count, ei.event_cap, event_ply, ei.d_nonstd, carry, event_env0, ei.stream));
    if (ei.maybe_nonstd) {
        if (apply)
            act_kernel<true><<<blocks(ei.n, kThreads), kThreads, 0, ei.stream>>>(ei.d_envs, ei.n, ei.env_id0, ei.seed, q90, thr, train_done, actions, ring, ring_cap,
                                                                                ring_pos, stats, ei.d_events, ei.d_event_count, ei.event_cap, event_ply, ei.d_nonstd);
        else
            act_kernel<false><<<blocks(ei.n, kThreads), kThreads, 0, ei.stream>>>(ei.d_envs, ei.n, ei.env_id0, ei.seed, q90, thr, train_done, actions, ring, ring_cap,
                                                                                 ring_pos, stats, ei.d_events, ei.d_event_count, ei.event_cap, event_ply, ei.d_nonstd);
        XQ_LAUNCH_CHECK();
    }
    return XQ_OK;
}

extern "C" {

int xq_replay_destroy(xq_replay_t r) {
    if (!r) return XQ_OK;
    cudaSetDevice(r->device);
    cudaFree(r->d_ring); cudaFree(r->d_batch); cudaFree(r->d_index);
    if (r->stream) cudaStreamDestroy(r->stream);
    if (r->ev) cudaEventDestroy(r->ev);
    delete r;
    return XQ_OK;
}

int xq_replay_create(int64_t capacity, int device, xq_replay_t* out) {
    if (!out || capacity <= 0) return fail(XQ_ERR_INVALID, "xq_replay_create: capacity must be > 0");
    int ndev = 0;
    XQ_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(XQ_ERR_INVALID, "xq_replay_create: device %d out of range", device);
    XQ_CUDA(cudaSetDevice(device));
    xq_replay_s* r = new (std::nothrow) xq_replay_s();
    if (!r) return fail(XQ_ERR_NOMEM, "xq_replay_create: out of host memory");
    r->capacity = capacity; r->device = device;
    cudaError_t e = cudaMalloc(&r->d_ring, sizeof(Transition) * capacity);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMemsetAsync(r->d_ring, 0, sizeof(Transition) * capacity, r->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(r->stream);
    if (e != cudaSuccess) { xq_replay_destroy(r); return fail(e == cudaErrorMemoryAllocation ? XQ_ERR_NOMEM : XQ_ERR_CUDA, "xq_replay_create: %s", cudaGetErrorString(e)); }
    *out = r;
    return XQ_OK;
}

int xq_replay_info(xq_replay_t r, int64_t* size, int64_t* capacity, int64_t* total) {
    if (!r) return fail(XQ_ERR_INVALID, "xq_replay_info: null handle");
    if (size) *size = r->total < r->capacity ? r->total : r->capacity;
    if (capacity) *capacity = r->capacity;
    if (total) *total = r->total;
    return XQ_OK;
}

int xq_replay_insert(xq_replay_t r, const xq_transition* batch, int64_t n) {
    if (!r || !batch || n < 0) return fail(XQ_ERR_INVALID, "xq_replay_insert: bad arguments");
    XQ_CUDA(cudaSetDevice(r->device));
    XQ_CUDA(cudaDeviceSynchronize());     // host-pointer convenience path: order against any stream that touched the ring
    int64_t done = 0;
    while (done < n) {
        const int64_t head = (r->total + done) % r->capacity;
        const int64_t m = std::min(n - done, r->capacity - head);
        XQ_CUDA(cudaMemcpyAsync(r->d_ring + head, batch + done, sizeof(Transition) * m, cudaMemcpyHostToDevice, r->stream));
        done += m;
    }
    XQ_CUDA(cudaStreamSynchronize(r->stream));
    r->total += n;
    return XQ_OK;
}

int xq_replay_get(xq_replay_t r, int64_t first, int64_t n, xq_transition* out) {
    if (!r || !out || first < 0 || n < 0 || first + n > r->capacity) return fail(XQ_ERR_INVALID, "xq_replay_get: bad range");
    XQ_CUDA(cudaSetDevice(r->device));
    XQ_CUDA(cudaDeviceSynchronize());
    XQ_CUDA(cudaMemcpy(out, r->d_ring + first, sizeof(Transition) * n, cudaMemcpyDeviceToHost));
    return XQ_OK;
}

static int replay_sample_dev(xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter, cudaStream_t stream, bool want_index) {
    const int64_t size = r->total < r->capacity ? r->total : r->capacity;
    if (size <= 0) return fail(XQ_ERR_STATE, "xq_replay_sample: the buffer is empty");
    if (batch > r->batch_cap) {
        cudaFree(r->d_batch); cudaFree(r->d_index); r->d_batch = nullptr; r->d_index = nullptr; r->batch_cap = 0;
        XQ_CUDA(cudaMalloc(&r->d_batch, sizeof(Transition) * batch));
        XQ_CUDA(cudaMalloc(&r->d_index, sizeof(int64_t) * batch));
        r->batch_cap = batch;
    }
    sample_kernel<<<blocks(batch * 32, 256), 256, 0, stream>>>(r->d_ring, size, batch, seed, counter, r->d_batch, want_index ? r->d_index : nullptr);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_replay_sample(xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter, xq_transition* out, int64_t* index) {
    if (!r || batch <= 0) return fail(XQ_ERR_INVALID, "xq_replay_sample: bad arguments");
    XQ_CUDA(cudaSetDevice(r->device));
    XQ_CUDA(cudaDeviceSynchronize());
    if (int rc = replay_sample_dev(r, batch, seed, counter, r->stream, true)) return rc;
    if (out) XQ_CUDA(cudaMemcpyAsync(out, r->d_batch, sizeof(Transition) * batch, cudaMemcpyDeviceToHost, r->stream));
    if (index) XQ_CUDA(cudaMemcpyAsync(index, r->d_index, sizeof(int64_t) * batch, cudaMemcpyDeviceToHost, r->stream));
    XQ_CUDA(cudaStreamSynchronize(r->stream));
    return XQ_OK;
}

int xq_dqn_act(xq_dqn_t h, xq_env_t env, double eps, xq_action* actions_host, float* q_host) {
    if (!h || !env || !actions_host) return fail(XQ_ERR_INVALID, "xq_dqn_act: null argument");
    EnvInfo ei;
    if (int rc = env_info(env, &ei)) return rc;
    if (ei.device != h->device) return fail(XQ_ERR_INVALID, "xq_dqn_act: env and network live on different devices");
    XQ_CUDA(cudaSetDevice(h->device));
    { FastWeights fw; if (int rc = dqn_fast_weights(h, &fw)) return rc; }      // refresh the FP32 / BF16 copies on h->stream before ordering after it
    SelfplayScratch* sc;
    if (int rc = reserve_scratch(env, ei.n, &sc)) return rc;
    if (int rc = order_after(ei.stream, h->stream, &sc->ev_order)) return rc;
    if (int rc = dqn_act_enter(h, ei.stream)) return rc;
    if (int rc = dqn_q90_device(h, ei.d_envs, ei.n, sc->q90, ei.stream)) return rc;
    if (int rc = launch_act(false, ei, sc->q90, xq_eps_threshold(eps), 0, sc->actions, nullptr, 1, 0, nullptr, 0u)) return rc;
    if (int rc = dqn_act_leave(h, ei.stream)) return rc;
    XQ_CUDA(cudaMemcpyAsync(actions_host, sc->actions, sizeof(uint16_t) * ei.n, cudaMemcpyDeviceToHost, ei.stream));
    if (q_host) XQ_CUDA(cudaMemcpyAsync(q_host, sc->q90, sizeof(float) * kQPad * ei.n, cudaMemcpyDeviceToHost, ei.stream));
    XQ_CUDA(cudaStreamSynchronize(ei.stream));
    return XQ_OK;
}

int xq_selfplay_collect(xq_dqn_t h, xq_env_t env, xq_replay_t r, int n_plies, double eps, int train_done) {
    if (!h || !env || n_plies < 0) return fail(XQ_ERR_INVALID, "xq_selfplay_collect: bad arguments");
    EnvInfo ei;
    if (int rc = env_info(env, &ei)) return rc;
    if (ei.device != h->device || (r && r->device != h->device)) return fail(XQ_ERR_INVALID, "xq_selfplay_collect: handles live on different devices");
    XQ_CUDA(cudaSetDevice(h->device));
    { FastWeights fw; if (int rc = dqn_fast_weights(h, &fw)) return rc; }      // refresh the FP32 / BF16 copies on h->stream before ordering after it
    SelfplayScratch* sc;
    if (int rc = reserve_scratch(env, ei.n, &sc)) return rc;
    if (int rc = order_after(ei.stream, h->stream, &sc->ev_order)) return rc;    // see the latest weights
    if (int rc = dqn_act_enter(h, ei.stream)) return rc;                           // ... and the previous user of the network's acting state
    xq_env_stats* d_stats = ei.d_stats;
    const uint32_t thr = xq_eps_threshold(eps);
    // the team kernel carries the layer-0 sums and h(s) of its envs into the next ply (tail of act_team_kernel): from the second ply of
    // this call on, the layer-0 kernel is not launched.  Not when boards with non-standard piece sets may go through the generic kernel.
    const bool can_carry = !ei.maybe_nonstd;
    // Two-stream plies from 8192 envs on: once the sums are carried, the env range is cut in two halves that run their
    // [contraction -> act] chains on streams of equal priority, out of step by themselves: the contraction of one half (tensor / HBM) and
    // the tail of an act kernel (HBM) fill the SMs the other half's act kernel (instruction issue) leaves idle between its waves
    const bool multi = can_carry && ei.n >= 8192;
    if (multi && !sc->ev_fork) {
        XQ_CUDA(cudaStreamCreateWithFlags(&sc->aux, cudaStreamNonBlocking));
        XQ_CUDA(cudaEventCreateWithFlags(&sc->ev_join, cudaEventDisableTiming));
        XQ_CUDA(cudaEventCreateWithFlags(&sc->ev_fork, cudaEventDisableTiming));
    }
    bool carried = false, forked = false;
    for (int p = 0; p < n_plies; ++p) {
        const int64_t ring_pos = r ? r->total % r->capacity : 0;
        if (multi && carried) {
            if (!forked) {
                XQ_CUDA(cudaEventRecord(sc->ev_fork, ei.stream));
                XQ_CUDA(cudaStreamWaitEvent(sc->aux, sc->ev_fork, 0));
                forked = true;
            }
            for (int half = 1; half >= 0; --half) {
                EnvInfo eh = ei;
                eh.stream = half ? sc->aux : ei.stream;
                ActCarry cy;
                int64_t o = 0, m = 0;
                if (int rc = dqn_q90_half(h, ei.n, half, sc->q90, eh.stream, &cy, &o, &m)) return rc;
                eh.d_envs = ei.d_envs + o; eh.n = m; eh.env_id0 = ei.env_id0 + (uint64_t)o; eh.d_nonstd = ei.d_nonstd ? ei.d_nonstd + o : nullptr;
                if (int rc = launch_act(true, eh, sc->q90 + o * kQPad, thr, train_done, nullptr, r ? r->d_ring : nullptr, r ? r->capacity : 1,
                                        r ? (ring_pos + o) % r->capacity : 0, d_stats, ei.event_ply + (uint32_t)p, &cy, (uint32_t)o)) return rc;
            }
        } else {
            ActCarry cy;
            if (int rc = dqn_q90_device(h, ei.d_envs, ei.n, sc->q90, ei.stream, carried, &cy)) return rc;
            if (int rc = launch_act(true, ei, sc->q90, thr, train_done, nullptr, r ? r->d_ring : nullptr, r ? r->capacity : 1, ring_pos,
                                    d_stats, ei.event_ply + (uint32_t)p, can_carry ? &cy : nullptr)) return rc;
            carried = can_carry;
        }
        if (r) r->total += ei.n;
    }
    if (forked) { XQ_CUDA(cudaEventRecord(sc->ev_join, sc->aux)); XQ_CUDA(cudaStreamWaitEvent(ei.stream, sc->ev_join, 0)); }
    env_advance_event_ply(env, (uint32_t)n_plies);
    if (int rc = dqn_act_leave(h, ei.stream)) return rc;
    if (int rc = order_after(h->stream, ei.stream, &sc->ev_order)) return rc;    // later TD updates see the new transitions
    return XQ_OK;
}

int xq_dqn_td_update_replay(xq_dqn_t h, xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter, int use_target_net, double lr, int apply) {
    if (!h || !r || batch <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_td_update_replay: bad arguments");
    if (r->device != h->device) return fail(XQ_ERR_INVALID, "xq_dqn_td_update_replay: handles live on different devices");
    XQ_CUDA(cudaSetDevice(h->device));
    const int64_t size = r->total < r->capacity ? r->total : r->capacity;
    if (size <= 0) return fail(XQ_ERR_STATE, "xq_dqn_td_update_replay: the buffer is empty");
    return dqn_td_update_sampled(h, r->d_ring, size, seed, counter, batch, use_target_net, lr, apply);
}

int xq_dqn_td_update_replay_n(xq_dqn_t h, xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter0, int n_updates, int use_target_net,
                              double lr) {
    if (!h || !r || batch <= 0 || n_updates < 0) return fail(XQ_ERR_INVALID, "xq_dqn_td_update_replay_n: bad arguments");
    if (r->device != h->device) return fail(XQ_ERR_INVALID, "xq_dqn_td_update_replay_n: handles live on different devices");
    XQ_CUDA(cudaSetDevice(h->device));
    const int64_t size = r->total < r->capacity ? r->total : r->capacity;
    if (size <= 0) return fail(XQ_ERR_STATE, "xq_dqn_td_update_replay_n: the buffer is empty");
    if (n_updates == 0) return XQ_OK;
    if (use_target_net && n_updates > 1) return dqn_td_update_pipelined(h, r->d_ring, size, seed, counter0, batch, n_updates, lr);
    for (int i = 0; i < n_updates; ++i)      // the online-net bootstrap depends on the previous update: nothing to pipeline
        if (int rc = dqn_td_update_sampled(h, r->d_ring, size, seed, counter0 + (uint32_t)i, batch, use_target_net, lr, 1)) return rc;
    return XQ_OK;
}

}  // extern "C"
