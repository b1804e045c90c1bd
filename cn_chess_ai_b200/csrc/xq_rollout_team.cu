// xq_rollout_team.cu -- fused random-policy rollout with a TEAM of 4 threads per board, 4 piece slots per thread.
//
// Mapping: one CTA = 32 boards x 4 warps; warp = role (0..3), lane = board; every warp runs the same code, the piece type of a
// position being a warp-uniform run-time value (xq_rollout_team.cuh), so there is no divergence on type and the replicated part
// of a ply (selection + apply, 235 of the 407 warp-instructions per ply of the 16-thread kernel) is paid 4 times per board
// instead of 16 times.  The ply itself lives in xq_rollout_team.cuh (host-compilable, diffed against the oracle by
// tests/hostsim); this file is the load / store conversion, the barriers and the launch.
//
// Replaces the loop body of ChessAI::train without the network (src/chessai.cpp:96-119).
#include "xq_common.cuh"
#include "xq_rollout_team.cuh"

namespace xq {

constexpr int kTB = 32;   // boards per CTA

struct TeamIo {           // conversion buffers, [item][board]
    uint8_t slot[32 * kTB];
    uint32_t bb[9 * kTB];
    uint32_t meta[4 * kTB];
    uint32_t words[12 * kTB];
    uint8_t active[kTB];
};

// MEM (teams of 4): the generators read the bitboards through the thread's slice of shared memory (MemView, xq_bitboard.cuh) instead of
// selecting among registers -- fewer integer-ALU instructions, one shared-memory round trip more on the dependent chain: measured
// 3.85e9 against 3.94e9 env steps/s at 4096 envs (latency-bound), 8.6e9 against 8.0e9 at 16,384 (issue-bound)
template <int T, bool MEM>
__global__ void __launch_bounds__(kTB * T) rollout_team_kernel(xq_env_rec* __restrict__ envs, int64_t n, uint64_t env_id0, uint64_t seed, int n_plies,
                                                                  xq_trace_rec* __restrict__ trace, xq_env_stats* __restrict__ stats,
                                                                  uint8_t* __restrict__ nonstd, const xq_env_rec* __restrict__ src,
                                                                  xq_env_rec* __restrict__ mirror) {
    __shared__ TeamShared<kTB> sh;
    __shared__ TeamIo io;
    __shared__ TeamViewMem<MEM ? kTB : 1> vmem;
    uint32_t* const view = MEM ? vmem.w : nullptr;
    const int tid = threadIdx.x, lane = tid & 31;
    const TeamRole R = team_role<T>(tid >> 5);
    const int64_t env = (int64_t)blockIdx.x * kTB + lane;
    team_tables_init(sh, tid, kTB * T);
    if (tid < kTB) sh.move[tid] = 0;

    // ---- load: warp 0 converts 32 records to slots + bitboards ----------------------------------
    if (R.role == 0) {
        bool ok = env < n;
        if (ok) {
            const uint4* rec = reinterpret_cast<const uint4*>((src ? src : envs) + env);      // src: mapped host boards (xq_env_rollout_random_io)
            uint32_t w[12];
#pragma unroll
            for (int i = 0; i < 3; ++i) { const uint4 v = rec[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
            const uint4 m = rec[3];
            if (src) {      // the device array follows the host boards (a board left to the generic kernel is read from there)
                uint4* d = reinterpret_cast<uint4*>(envs + env);
#pragma unroll
                for (int i = 0; i < 3; ++i) d[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
                d[3] = m;
            }
            for (int i = 0; i < 32; ++i) io.slot[i * kTB + lane] = kDeadSq;
            Bits90 red, black, occT;
            ok = team_unpack_record(w, red, black, occT, [&](int s, int q) { io.slot[s * kTB + lane] = (uint8_t)q; });
            io.bb[0 * kTB + lane] = red.w0; io.bb[1 * kTB + lane] = red.w1; io.bb[2 * kTB + lane] = red.w2;
            io.bb[3 * kTB + lane] = black.w0; io.bb[4 * kTB + lane] = black.w1; io.bb[5 * kTB + lane] = black.w2;
            io.bb[6 * kTB + lane] = occT.w0; io.bb[7 * kTB + lane] = occT.w1; io.bb[8 * kTB + lane] = occT.w2;
            io.meta[0 * kTB + lane] = m.x; io.meta[1 * kTB + lane] = m.y; io.meta[2 * kTB + lane] = m.z; io.meta[3 * kTB + lane] = m.w;
            if (nonstd) nonstd[env] = ok ? 0 : 1;
        }
        io.active[lane] = ok ? 1 : 0;
    }
    __syncthreads();

    const bool active = io.active[lane] != 0;
    TeamState st;
    TeamBook bk{0, 0, 1480, 1480, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    team_reset(R, st);
    st.ctr = 0;
    uint64_t rng_base = 0;
    if (active) {
        uint32_t wr = 0, wb = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int s = (int)((R.slots >> (8 * i)) & 0xFFu);
            wr |= (uint32_t)(i < 16 / T ? io.slot[s * kTB + lane] : kDeadSq) << (8 * i);
            wb |= (uint32_t)(i < 16 / T ? io.slot[(16 + s) * kTB + lane] : kDeadSq) << (8 * i);
        }
        const Bits90 red{io.bb[0 * kTB + lane], io.bb[1 * kTB + lane], io.bb[2 * kTB + lane]};
        const Bits90 black{io.bb[3 * kTB + lane], io.bb[4 * kTB + lane], io.bb[5 * kTB + lane]};
        st.occT = Bits90{io.bb[6 * kTB + lane], io.bb[7 * kTB + lane], io.bb[8 * kTB + lane]};
        const int gen_red = io.slot[8 * kTB + lane], gen_black = io.slot[24 * kTB + lane];
        const uint32_t m0 = io.meta[0 * kTB + lane];
        st.move_count = (int)(m0 & 0xFFFFu); st.player = (int)((m0 >> 16) & 0xFFu);
        st.ctr = io.meta[3 * kTB + lane];
        if (R.role == 0) {
            bk.red = (int)io.meta[1 * kTB + lane]; bk.black = (int)io.meta[2 * kTB + lane];
            int mr = 0, mb = 0;      // material per side from the slots (ChessAI::evaluateBoard :313-341)
            for (int i = 0; i < 16; ++i) {
                const int sc = piece_score(slot_type(i));
                if (io.slot[i * kTB + lane] != kDeadSq) mr += sc;
                if (io.slot[(16 + i) * kTB + lane] != kDeadSq) mb += sc;
            }
            bk.mat_red = mr; bk.mat_black = mb;
        }
        if (st.move_count >= XQ_MAX_MOVES || gen_red == kDeadSq || gen_black == kDeadSq) {
            // a finished board is never stepped (chessai.cpp:90,96): restart it
            const uint32_t c = st.ctr; team_reset(R, st); st.ctr = c;
            bk.red = bk.black = 0; bk.mat_red = bk.mat_black = 1480;
        } else if (st.player == RED) {
            st.sq_own = wr; st.sq_opp = wb; st.own = red; st.opp = black; st.gen_own = gen_red; st.gen_opp = gen_black;
        } else {
            st.sq_own = wb; st.sq_opp = wr; st.own = black; st.opp = red; st.gen_own = gen_black; st.gen_opp = gen_red;
        }
        rng_base = seed + (env_id0 + (uint64_t)env) * 0x9E3779B97F4A7C15ull;
    }
    // lanes without a board (tail of the last CTA, non-standard piece sets) play a private game from the opening: the ply loop has no
    // `active` test; they get no trace, no statistics and no store
    xq_trace_rec* const my_trace = active ? trace : nullptr;
    const uint32_t ctr0 = st.ctr;
    team_rng_chunk<T, kTB>(R, sh, lane, 0, rng_base, ctr0);
    if (view) team_view_put<kTB>(R, st, view, lane);      // this thread's bitboards for run-time word indices (MemView)
    __syncthreads();
    TeamPly pl;
#pragma unroll 1
    for (int p = 0; p < n_plies; ++p) {
        if ((p & 15) == 0) team_rng_chunk<T, kTB>(R, sh, lane, (p >> 4) + 1, rng_base, ctr0);   // read from ply p + 16 on
        team_phase_a<T, kTB>(R, st, pl, sh, lane, p, view);
        __syncthreads();
        if (R.role == 0) team_finalize<kTB>(bk, sh, lane, my_trace, n, env);
        team_phase_b<T, kTB>(R, st, pl, sh, lane, p);
        __syncthreads();
        team_phase_c<kTB>(R, st, pl, sh, bk, lane, p, view);
    }
    if (active) {
        const uint32_t wr = st.player == RED ? st.sq_own : st.sq_opp, wb = st.player == RED ? st.sq_opp : st.sq_own;
#pragma unroll
        for (int i = 0; i < 16 / T; ++i) {
            const int s = (int)((R.slots >> (8 * i)) & 0xFFu);
            io.slot[s * kTB + lane] = (uint8_t)(wr >> (8 * i));
            io.slot[(16 + s) * kTB + lane] = (uint8_t)(wb >> (8 * i));
        }
    }
    __syncthreads();

    // ---- store: slots -> nibble board ---------------------------------------------------------------
    if (R.role == 0) {
        if (active) {
            team_finalize<kTB>(bk, sh, lane, my_trace, n, env);      // the last ply
            for (int i = 0; i < 12; ++i) io.words[i * kTB + lane] = 0;
            for (int i = 0; i < 32; ++i) {
                const int q = io.slot[i * kTB + lane];
                if (q != kDeadSq) io.words[(q >> 3) * kTB + lane] |= (uint32_t)(slot_type(i & 15) + (i >= 16 ? 7 : 0)) << (4 * (q & 7));
            }
            uint4* rec = reinterpret_cast<uint4*>(envs + env);
#pragma unroll
            for (int i = 0; i < 3; ++i)
                rec[i] = make_uint4(io.words[(4 * i) * kTB + lane], io.words[(4 * i + 1) * kTB + lane], io.words[(4 * i + 2) * kTB + lane],
                                    io.words[(4 * i + 3) * kTB + lane]);
            const uint32_t flags = io.meta[0 * kTB + lane] & 0xFF000000u;
            rec[3] = make_uint4((uint32_t)(st.move_count & 0xFFFF) | ((uint32_t)st.player << 16) | flags, (uint32_t)bk.red, (uint32_t)bk.black, st.ctr);
            if (mirror) {   // the same record into the caller's mapped host buffer
                uint4* mr = reinterpret_cast<uint4*>(mirror + env);
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    mr[i] = make_uint4(io.words[(4 * i) * kTB + lane], io.words[(4 * i + 1) * kTB + lane], io.words[(4 * i + 2) * kTB + lane],
                                       io.words[(4 * i + 3) * kTB + lane]);
                mr[3] = make_uint4((uint32_t)(st.move_count & 0xFFFF) | ((uint32_t)st.player << 16) | flags, (uint32_t)bk.red, (uint32_t)bk.black, st.ctr);
            }
        } else {
            bk = TeamBook{0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        }
        if (stats) {
            unsigned long long v[8] = {bk.a_steps, bk.a_games, bk.a_red, bk.a_black, bk.a_capg, bk.a_caps, (unsigned long long)bk.a_reward, bk.a_legal};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                unsigned long long r = v[i];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
                if (lane == 0 && r != 0) atomicAdd(reinterpret_cast<unsigned long long*>(stats) + i, r);
            }
        }
    }
}

cudaError_t launch_rollout_team(xq_env_rec* envs, int64_t n, uint64_t env_id0, uint64_t seed, int n_plies, xq_trace_rec* trace,
                                xq_env_stats* stats, uint8_t* nonstd, cudaStream_t stream, const xq_env_rec* src, xq_env_rec* mirror) {
    const unsigned grid = (unsigned)((n + kTB - 1) / kTB);
    const char* ve = getenv("XQ_TEAM_VIEW");      // A/B and tests (read per call): 0 registers, 1 shared-memory view
    const int view_env = ve ? atoi(ve) : -1;
    const bool mem = view_env >= 0 ? view_env != 0 : n > 148 * kTB;      // more than one CTA per SM: issue-bound enough for the view to pay (4.84e9 against 4.66e9 at 6144 envs)
    if (mem) rollout_team_kernel<4, true><<<grid, kTB * 4, 0, stream>>>(envs, n, env_id0, seed, n_plies, trace, stats, nonstd, src, mirror);
    else rollout_team_kernel<4, false><<<grid, kTB * 4, 0, stream>>>(envs, n, env_id0, seed, n_plies, trace, stats, nonstd, src, mirror);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace xq
