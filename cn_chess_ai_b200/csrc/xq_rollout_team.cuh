// xq_rollout_team.cuh -- one ply of the fused random-policy rollout for a TEAM of 4 threads per board, each thread owning 4 piece
// slots of either side.  The three phases of a ply are host-compilable functions (tests/hostsim runs the 4 threads of a board one
// after the other, phase by phase, and diffs the whole trace against the oracle before any GPU time); the kernel in
// xq_rollout_team.cu is these phases with two __syncthreads per ply between them.
//
// Why teams: in a 16-threads-per-board kernel (one thread per piece slot; DESIGN.md section 4) every thread keeps a replica of the board and repeats the
// selection and the apply step -- ncu attributes 136 of its 407 warp-instructions per ply to move generation and 235 to the
// replicated part.  With 4 slots per thread the replicated part is paid 4 times per board instead of 16 times, and warps stay
// piece-type uniform: role = warp, lane = board, and position i of every lane of a warp holds the same piece type.
//
// State is kept RELATIVE to the side to move (own / opp) and swapped after every ply, so neither the generator nor the apply
// step selects on the mover's colour.  The 4 squares of a side are packed one per byte (127 = captured); capture detection, the
// move of the own piece and the reference-order prefix (sum of the move counts of the pieces on lower squares,
// ChessAI::getAllValidActions scans squares row-major: src/chessai.cpp:347-368) are byte-SIMD on those words.
#pragma once
#include <stdint.h>

#include "../../include/xq.h"
#include "xq_bitboard.cuh"

namespace xq {

#if defined(__CUDA_ARCH__)
XQ_HD uint32_t dp4a_u(uint32_t a, uint32_t b, uint32_t c) { return __dp4a(a, b, c); }
XQ_HD uint32_t umulhi_u(uint32_t a, uint32_t b) { return __umulhi(a, b); }
#else
XQ_HD uint32_t dp4a_u(uint32_t a, uint32_t b, uint32_t c) {
    for (int i = 0; i < 4; ++i) c += ((a >> (8 * i)) & 0xFFu) * ((b >> (8 * i)) & 0xFFu);
    return c;
}
XQ_HD uint32_t umulhi_u(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
#endif
XQ_HD Bits90 bit_mask(int i) { return Bits90::bit(i); }

// ---- the team: T threads per board, S = 16/T piece slots per thread, ONE code path for all roles ---------------------------------
// T = 4 (the throughput shape)                                                    T = 8 (small env counts: twice the warps per board)
// position:   0 (slider)        1                 2                  3            position:  0                 1
// role 0:     Chariot  slot 0   Horse    slot 2   Soldier  slot 11   Soldier 12   role 0,1:  Chariot 0,1       Soldier 11,12
// role 1:     Chariot  slot 1   Horse    slot 3   Soldier  slot 13   Soldier 14   role 2,3:  Cannon  9,10      Soldier 13,14
// role 2:     Cannon   slot 9   Advisor  slot 6   Elephant slot 4    General 8    role 4,5:  Horse   2,3       Advisor 6,7
// role 3:     Cannon   slot 10  Advisor  slot 7   Elephant slot 5    Soldier 15   role 6,7:  Elephant 4,5      General 8 / Soldier 15
// The piece type of a position is a warp-uniform RUN-TIME value (role = warp): a select for the sliders, a short branch for the
// leapers.  Every warp therefore runs the same ~14 KB loop body -- a first version with one template instantiation per role
// (4 x 30 KB of straight-line code) spent most of its cycles in `no_instruction` stalls (ncu), the instruction cache being 32 KB.
struct TeamRole {
    int role;
    uint32_t slots;                // slot of position i in byte i (unused positions: 0xFF)
    uint32_t types;                // PieceType of position i in byte i (unused: 0)
    uint32_t score5;               // piece value / 5
    uint32_t open_red, open_black; // opening squares of my slots (ChessBoard::initializeBoard, src/chessboard.cpp:13-28); unused bytes 127
    // destination offsets of a leaper at position i, one signed byte per direction in the order of generate*Moves
    // (src/chessboard.cpp:150,163,180,249,267-281); a Horse has eight (tab_hi); a Soldier's table is Red's and sold[i] = 0xFE
    // flips its 9 into -9 for Black
    uint32_t tab_lo[4], tab_hi, sold[4];
};
constexpr int open_sq_c(int s) {   // opening square of slot s (0..15 Red, 16..31 Black)
    constexpr uint8_t t[32] = {0, 8, 1, 7, 2, 6, 3, 5, 4, 19, 25, 27, 29, 31, 33, 35, 81, 89, 82, 88, 83, 87, 84, 86, 85, 64, 70, 54, 56, 58, 60, 62};
    return t[s];
}
constexpr int slot_type_c(int s) {
    return s < 2 ? CHARIOT : (s < 4 ? HORSE : (s < 6 ? ELEPHANT : (s < 8 ? ADVISOR : (s == 8 ? GENERAL : (s < 11 ? CANNON : SOLDIER)))));
}
constexpr int piece_score_c(int type) { return type == GENERAL ? 1000 : (type == ADVISOR || type == ELEPHANT ? 20 : (type == HORSE ? 40 : (type == CHARIOT ? 90 : (type == CANNON ? 45 : 10)))); }
constexpr int team_slot_c(int T, int role, int pos) {      // -1: unused position
    constexpr int8_t t4[4][4] = {{0, 2, 11, 12}, {1, 3, 13, 14}, {9, 6, 4, 8}, {10, 7, 5, 15}};
    constexpr int8_t t8[8][2] = {{0, 11}, {1, 12}, {9, 13}, {10, 14}, {2, 6}, {3, 7}, {4, 8}, {5, 15}};
    return T == 4 ? t4[role][pos] : (pos < 2 ? t8[role][pos] : -1);
}
constexpr TeamRole team_role_c(int T, int role) {
    TeamRole r{};
    r.role = role;
    for (int i = 0; i < 4; ++i) {
        const int slot = team_slot_c(T, role, i);
        const int type = slot < 0 ? 0 : slot_type_c(slot);
        r.slots |= (uint32_t)(slot < 0 ? 0xFF : slot) << (8 * i);
        r.types |= (uint32_t)type << (8 * i);
        r.score5 |= (uint32_t)(slot < 0 ? 0 : piece_score_c(type) / 5) << (8 * i);
        r.open_red |= (uint32_t)(slot < 0 ? 127 : open_sq_c(slot)) << (8 * i);
        r.open_black |= (uint32_t)(slot < 0 ? 127 : open_sq_c(16 + slot)) << (8 * i);
        r.tab_lo[i] = type == HORSE ? 0xF5F9070Bu          // 11,7,-7,-11 (| 19,17,-17,-19 in tab_hi)
                    : (type == ADVISOR ? 0xF6F8080Au       // 10,8,-8,-10
                    : (type == ELEPHANT ? 0xECF01014u      // 20,16,-16,-20
                    : (type == GENERAL ? 0xFF01F709u       // 9,-9,1,-1
                    : (type == SOLDIER ? 0x0001FF09u : 0u))));   // Red: 9,-1,1
        if (type == HORSE) r.tab_hi = 0xEDEF1113u;
        r.sold[i] = type == SOLDIER ? 0xFEu : 0u;
    }
    return r;
}
template <int T>
XQ_HD TeamRole team_role(int role) {      // once per thread
    constexpr TeamRole r0 = team_role_c(T, 0), r1 = team_role_c(T, 1), r2 = team_role_c(T, 2), r3 = team_role_c(T, 3);
    constexpr TeamRole r4 = team_role_c(T, T == 8 ? 4 : 0), r5 = team_role_c(T, T == 8 ? 5 : 0), r6 = team_role_c(T, T == 8 ? 6 : 0), r7 = team_role_c(T, T == 8 ? 7 : 0);
    switch (role) {
        case 0: return r0;
        case 1: return r1;
        case 2: return r2;
        case 3: return r3;
        case 4: return r4;
        case 5: return r5;
        case 6: return r6;
        default: return r7;
    }
}
XQ_HD Bits90 team_open_red() { return Bits90{0xAA0801FFu, 0x0000000Au, 0x00000000u}; }
XQ_HD Bits90 team_open_black() { return Bits90{0x00000000u, 0x55400000u, 0x03FE0041u}; }
XQ_HD Bits90 team_open_occT() { return Bits90{0x649A1649u, 0x98064980u, 0x0249A164u}; }

// shared memory of a CTA of KB boards, every array [item][board]: lane == bank
template <int KB>
struct TeamShared {
    uint32_t q[4 * KB];            // [role][board]: squares of the mover's 16 slots, one byte each
    uint32_t c[4 * KB];            // their move counts
    uint32_t move[KB];             // from | to << 8
    uint32_t cap[2 * KB];          // value | code << 16 of the captured piece, double-buffered by ply parity
    uint32_t rng[2 * 16 * KB];     // idx31 draws of 16 plies, double-buffered by chunk parity
    uint32_t magic[XQ_MAX_ACTIONS + 1];
    uint32_t geo[kGeoWords];       // geometry table of the leapers (xq_bitboard.cuh: geo_entry), [colour][128]
};
// teams of 4, kernels that run many plies per launch: every thread's bitboards [word][role * KB + board] for run-time word indices (MemView)
template <int KB>
struct TeamViewMem { uint32_t w[kViewWords * 4 * KB]; };
// the two tables of a CTA: magic[d] = team_mod_magic(d), geo[colour * 128 + sq] = geo_entry(colour, sq); a barrier must follow
template <class SH>
XQ_HD void team_tables_init(SH& sh, int tid, int n_threads) {
    for (int d = tid + 1; d <= XQ_MAX_ACTIONS; d += n_threads) sh.magic[d] = (0xFFFFFFFFu / (uint32_t)d) + 1u;
    for (int i = tid; i < kGeoWords; i += n_threads) sh.geo[i] = geo_word(i);
}

struct TeamState {
    uint32_t sq_own, sq_opp;       // packed squares of my 4 slots: side to move / the other side
    Bits90 own, opp, occT;
    int gen_own, gen_opp;
    int move_count, player;
    uint32_t ctr;
};
// a thread's slice of the view memory (teams of 4): written after every change of st.own / st.opp / st.occT, read by its own phase A
template <int KB>
XQ_HD void team_view_store(const TeamRole& R, const TeamState& st, uint32_t* view, int lane) {
    view_store(view + R.role * KB + lane, 4 * KB, st.own, st.opp, st.occT);
}
template <int KB>
XQ_HD void team_view_put(const TeamRole& R, const TeamState& st, uint32_t* view, int lane) {      // padding words + the bitboards
    view_init(view + R.role * KB + lane, 4 * KB);
    team_view_store<KB>(R, st, view, lane);
}
struct TeamPly {                   // scratch of one ply, phase A -> B -> C
    uint32_t desc[4];
    uint32_t cntw;
    uint32_t total;
};
// scores / material / reward / statistics / trace: role 0 alone, one barrier late
struct TeamBook {
    int red, black, mat_red, mat_black;
    uint32_t pend, pend_tr0;
    int pend_p;
    uint32_t a_steps, a_games, a_red, a_black, a_capg, a_caps, a_legal;
    long long a_reward;
};

XQ_HD void team_reset(const TeamRole& R, TeamState& st) {
    st.sq_own = R.open_red; st.sq_opp = R.open_black;
    st.own = team_open_red(); st.opp = team_open_black(); st.occT = team_open_occT();
    st.gen_own = 4; st.gen_opp = 85; st.move_count = 0; st.player = RED;
}

XQ_HD uint32_t team_draw(uint64_t rng_base, uint32_t ctr) {       // idx31 of xq_rng (include/xq.h)
    uint64_t z = rng_base + (uint64_t)ctr * 0xD1B54A32D192ED03ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (uint32_t)(z >> 33);
}
// the draws of plies [16*chunk, 16*chunk+16): thread (role, lane) computes 4 of them.  The RNG counter of ply p is ctr0 + p
// whatever happens in between (a move and a no-action restart both advance it by one).
template <int T, int KB>
XQ_HD void team_rng_chunk(const TeamRole& R, TeamShared<KB>& sh, int lane, int chunk, uint64_t rng_base, uint32_t ctr0) {
#pragma unroll 1
    for (int i = 0; i < 16 / T; ++i) {
        const int j = R.role * (16 / T) + i;
        sh.rng[((chunk & 1) * 16 + j) * KB + lane] = team_draw(rng_base, ctr0 + (uint32_t)(chunk * 16 + j));
    }
}

XQ_HD uint32_t team_mod_magic(uint32_t d) { return (0xFFFFFFFFu / d) + 1u; }
// n % d for n < 2^31, 1 <= d <= 128 without a hardware divide: q = umulhi(n, ceil(2^32/d)) is floor(n/d) or one above
// (error < n*d/2^32 < 1), so one conditional fix-up makes the remainder exact
XQ_HD uint32_t team_mod(uint32_t n, uint32_t d, uint32_t magic) {
    const uint32_t q = umulhi_u(n, magic);
    const int32_t r = (int32_t)(n - q * d);
    return d == 1 ? 0u : (uint32_t)(r < 0 ? r + (int32_t)d : r);
}

// sliders with the piece type at run time: the capture square is the second blocker for a Cannon, the first for a Chariot
XQ_HD int slider_desc_rt(const Pos& P, int sq, bool cannon, uint32_t* desc) {
    const int r = row_of(sq), c = sq - 9 * r;
    const uint32_t rank = P.occ.field(9 * r, 9), file = P.occT.field(10 * c, 10);
    int total = 0;
    uint32_t d = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const bool horiz = k < 2;
        const int p = horiz ? c : r;
        const Ray ray = (k & 1) ? ray_down(horiz ? rank : file, p, horiz ? 9 : 10) : ray_up(horiz ? rank : file, p, horiz ? 9 : 10);
        const int tgt = cannon ? ray.second : ray.first;
        const int s = horiz ? 9 * r + tgt : 9 * tgt + c;                      // tgt == -1 reads some bit: discarded
        const bool cap = (tgt >= 0) & !P.own.test(s);
        const int capdist = cap ? ((k & 1) ? p - tgt : tgt - p) : 0;
        d |= ((uint32_t)ray.empties | ((uint32_t)capdist << 4)) << (8 * k);
        total += ray.empties + (cap ? 1 : 0);
    }
    *desc = d;
    return total;
}
// index of the j-th (0-based) set bit of an 8-bit mask with at least j+1 bits set: three halving steps
XQ_HD int nth_set_bit8(uint32_t m, int j) {
    int c = popc32(m & 0xFu);
    const bool h4 = j >= c;
    j -= h4 ? c : 0; m = h4 ? m >> 4 : m;
    c = popc32(m & 0x3u);
    const bool h2 = j >= c;
    j -= h2 ? c : 0; m = h2 ? m >> 2 : m;
    return (h4 ? 4 : 0) + (h2 ? 2 : 0) + ((j >= (int)(m & 1u)) ? 1 : 0);
}
// ---- phase A: every thread counts the moves of its S pieces of the side to move and publishes (squares, counts) -------------
// view (teams of 4, optional): TeamViewMem<KB>::w holding the bitboards of st (team_view_store) -- the generators then take run-time word
// indices from shared memory (MemView) instead of selecting among registers (RegView); same results
template <int T, int KB>
XQ_HD void team_phase_a(const TeamRole& R, const TeamState& st, TeamPly& pl, TeamShared<KB>& sh, int lane, int p, const uint32_t* view = nullptr) {
    Pos P;
    P.own = st.own;
    P.occ = Bits90{st.own.w0 | st.opp.w0, st.own.w1 | st.opp.w1, st.own.w2 | st.opp.w2};
    P.occT = st.occT;
    const int color = st.player;
    const int q0 = (int)(st.sq_own & 0xFFu), q1 = (int)((st.sq_own >> 8) & 0xFFu);
    // a captured piece (square 127) reads garbage bits: a slider's count is discarded, a leaper's table word is 0
    if (T == 4) {
        const bool hi = R.role >= 2;
        const int q2 = (int)((st.sq_own >> 16) & 0xFFu), q3 = (int)(st.sq_own >> 24);
        const uint32_t* gq = sh.geo + color * 128;
        const uint32_t g1 = gq[q1], g2 = gq[q2], g3 = gq[q3];
        int c0;
        uint32_t m1, m2, m3;
        auto gen = [&](const auto& V) {
            c0 = slider_desc_v(V, q0, hi, &pl.desc[0]);
            if (!hi) { m1 = horse_mask_g(V, q1, g1); m2 = soldier_mask_g(V, q2, color, g2); m3 = soldier_mask_g(V, q3, color, g3); }
            else {
                m1 = advisor_mask_g(V, q1, g1); m2 = elephant_mask_g(V, q2, g2);
                m3 = R.role == 2 ? general_mask_g(V, q3, g3) : soldier_mask_g(V, q3, color, g3);
            }
        };
        if (view) gen(MemView{view + R.role * KB + lane, 4 * KB});      // == (st.own, st.own | st.opp, st.occT): team_view_store
        else gen(RegView{P.own, P.occ, P.occT});
        pl.desc[1] = m1; pl.desc[2] = m2; pl.desc[3] = m3;
        c0 = q0 == kDeadSq ? 0 : c0;
        const int c1 = popc32(m1), c2 = popc32(m2), c3 = popc32(m3);
        pl.cntw = (uint32_t)c0 | ((uint32_t)c1 << 8) | ((uint32_t)c2 << 16) | ((uint32_t)c3 << 24);
        sh.q[R.role * KB + lane] = st.sq_own;
        sh.c[R.role * KB + lane] = pl.cntw;
    } else {
        int c0;
        uint32_t d0, m1;
        if (R.role < 4) c0 = slider_desc_rt(P, q0, R.role >= 2, &d0);
        else { d0 = R.role < 6 ? horse_mask(P, q0) : elephant_mask(P, q0, color); c0 = popc32(d0); }
        if (R.role < 4 || R.role == 7) m1 = soldier_mask(P, q1, color);
        else m1 = R.role < 6 ? advisor_mask(P, q1, color) : general_mask(P, q1);
        pl.desc[0] = d0; pl.desc[1] = m1;
        c0 = q0 == kDeadSq ? 0 : c0;
        const int c1 = q1 == kDeadSq ? 0 : popc32(m1);
        pl.cntw = (uint32_t)c0 | ((uint32_t)c1 << 8);
        reinterpret_cast<uint16_t*>(sh.q)[((R.role >> 1) * KB + lane) * 2 + (R.role & 1)] = (uint16_t)st.sq_own;      // half a word per role
        reinterpret_cast<uint16_t*>(sh.c)[((R.role >> 1) * KB + lane) * 2 + (R.role & 1)] = (uint16_t)pl.cntw;
    }
    if (R.role == 0) sh.cap[(p & 1) * KB + lane] = 0;
}

// ---- bookkeeping of the previous ply (role 0): the captured value published in its phase C is visible now ---------------------
template <int KB>
XQ_HD void team_finalize(TeamBook& bk, const TeamShared<KB>& sh, int lane, xq_trace_rec* trace, int64_t n, int64_t env) {
    if (bk.pend == 0) return;
    const int mover = (bk.pend >> 2) & 1, win = (bk.pend >> 4) & 3, mc = (bk.pend >> 8) & 0xFF, total = (int)(bk.pend >> 16);
    const bool over = (bk.pend >> 3) & 1;
    uint32_t capcode = 0;
    int reward = 0;
    if ((bk.pend & 3) == 1) {
        const uint32_t capw = sh.cap[(bk.pend_p & 1) * KB + lane];
        const int capscore = (int)(capw & 0xFFFFu);
        capcode = capw >> 16;
        if (capscore) {      // ChessBoard::movePiece, src/chessboard.cpp:51-58
            if (mover == RED) { bk.red += capscore; bk.mat_black -= capscore; } else { bk.black += capscore; bk.mat_red -= capscore; }
        }
        reward = reward_from_material(mover == RED ? bk.mat_red - bk.mat_black : bk.mat_black - bk.mat_red, mc);
        bk.a_steps++; bk.a_legal += (uint32_t)total; bk.a_reward += reward; if (capscore) bk.a_caps++;
        if (over) { bk.a_games++; if (win == RED) bk.a_red++; else bk.a_black++; if (mc < XQ_MAX_MOVES) bk.a_capg++; }
    } else {
        bk.a_games++;
    }
    if (trace) {   // one 8-byte record: action | n_legal << 16 | flags << 24 (bits 4-7 of flags = captured piece code), reward
        uint32_t* t = reinterpret_cast<uint32_t*>(trace) + 2 * ((int64_t)bk.pend_p * n + env);
        t[0] = bk.pend_tr0 | (capcode << 28);
        t[1] = (uint32_t)reward;
    }
    if ((bk.pend & 3) == 2 || over) { bk.red = bk.black = 0; bk.mat_red = bk.mat_black = 1480; }     // ChessBoard::reset
    bk.pend = 0;
}

// ---- phase B: list size, draw, reference-order prefix of my pieces; the owner of the k-th action decodes it ------------------
template <int T, int KB>
XQ_HD void team_phase_b(const TeamRole& R, const TeamState& st, TeamPly& pl, TeamShared<KB>& sh, int lane, int p) {
    uint32_t qw[4], cw[4], tot = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) { qw[w] = sh.q[w * KB + lane]; cw[w] = sh.c[w * KB + lane]; tot = dp4a_u(cw[w], 0x01010101u, tot); }
    pl.total = tot;
    if (tot > 0) {
        const uint32_t draw = sh.rng[(((p >> 4) & 1) * 16 + (p & 15)) * KB + lane];
        const uint32_t k = team_mod(draw, tot, sh.magic[tot]);
        // which of my pieces (if any) owns the k-th action of the reference-ordered list: selects only, then ONE decode
        uint32_t hsq = 0, hdesc = 0, hwant = 0, hlo = 0, hhi = 0;
        bool hit = false, hslider = false;
        const uint32_t flip = st.player ? 0xFFFFFFFFu : 0u;          // a Black Soldier moves towards row 0
#pragma unroll
        for (int i = 0; i < 16 / T; ++i) {
            const uint32_t sq = (st.sq_own >> (8 * i)) & 0xFFu;
            // byte j of (base - qw) has bit 7 set iff square_j < sq (bytes <= 127, so no borrow crosses a byte); dp4a sums 128 * count_j over them
            const uint32_t base = sq * 0x01010101u + 0x7F7F7F7Fu;
            uint32_t acc = 0;
#pragma unroll
            for (int w = 0; w < 4; ++w) acc = dp4a_u(cw[w], (base - qw[w]) & 0x80808080u, acc);
            const uint32_t want = k - (acc >> 7), cnt = (pl.cntw >> (8 * i)) & 0xFFu;
            const bool h = want < cnt;
            hit |= h;
            hsq = h ? sq : hsq; hdesc = h ? pl.desc[i] : hdesc; hwant = h ? want : hwant;
            hlo = h ? (R.tab_lo[i] ^ (R.sold[i] & flip)) : hlo;
            if (i == 0) hslider = h & (T == 4 || R.role < 4);
            if (i == (T == 4 ? 1 : 0)) hhi = h ? R.tab_hi : 0u;      // the only position that can hold a Horse
        }
        if (hit) {
            const int to_s = slider_decode(hdesc, (int)hsq, (int)hwant);
            const int dk = nth_set_bit8(hdesc & 0xFFu, (int)hwant & 7);
            const int to_l = (int)hsq + (int)(int8_t)(uint8_t)((((uint64_t)hhi << 32) | hlo) >> (8 * dk));
            sh.move[lane] = hsq | ((uint32_t)(hslider ? to_s : to_l) << 8);
        }
    }
}

// ---- phase C: every thread applies the move to its replica; the thread owning the captured slot publishes value | code -------
// ChessBoard::movePiece (src/chessboard.cpp:38-64), checkGameOver / getWinner (:286-320), reset (:95-102)
template <int KB>
XQ_HD void team_phase_c(const TeamRole& R, TeamState& st, const TeamPly& pl, TeamShared<KB>& sh, TeamBook& bk, int lane, int p, uint32_t* view = nullptr) {
    // straight-line for the common case; with no legal action (pl.total == 0, below) the stale move read here is discarded
    const uint32_t mv = sh.move[lane];
    const int from = (int)(mv & 0xFFu), to = (int)((mv >> 8) & 0xFFu);
    const int mover = st.player;
    // is one of my pieces of the side NOT moving on `to`?  x has a zero byte there; bytes <= 127, so 0x80 - byte never borrows
    uint32_t z = (0x80808080u - (st.sq_opp ^ ((uint32_t)to * 0x01010101u))) & 0x80808080u;
    if (z) {
        const int sh8 = ffs32(z) - 8;                                   // 8 * position
        const uint32_t type = (R.types >> sh8) & 0xFFu, sc5 = (R.score5 >> sh8) & 0xFFu;
        sh.cap[(p & 1) * KB + lane] = (sc5 * 5u) | ((type + (mover ? 0u : 7u)) << 16);
    }
    const uint32_t sq_opp = st.sq_opp | (z >> 7) * 0x7Fu;                 // captured: square 127
    z = (0x80808080u - (st.sq_own ^ ((uint32_t)from * 0x01010101u))) & 0x80808080u;
    const uint32_t m8 = (z >> 7) * 0xFFu;
    const uint32_t sq_own = (st.sq_own & ~m8) | (((uint32_t)to * 0x01010101u) & m8);
    const int fr = row_of(from), tr = row_of(to);
    const Bits90 fm = bit_mask(from), tm = bit_mask(to);
    const Bits90 cf = bit_mask(cm_index(fr, from - 9 * fr)), ct = bit_mask(cm_index(tr, to - 9 * tr));
    const Bits90 own{(st.own.w0 & ~fm.w0) | tm.w0, (st.own.w1 & ~fm.w1) | tm.w1, (st.own.w2 & ~fm.w2) | tm.w2};
    const Bits90 opp{st.opp.w0 & ~tm.w0, st.opp.w1 & ~tm.w1, st.opp.w2 & ~tm.w2};
    const Bits90 occT{(st.occT.w0 & ~cf.w0) | ct.w0, (st.occT.w1 & ~cf.w1) | ct.w1, (st.occT.w2 & ~cf.w2) | ct.w2};
    const bool took_general = to == st.gen_opp;
    const int gen_own = from == st.gen_own ? to : st.gen_own;
    const int mc = st.move_count + 1;
    st.ctr++;
    const bool over = took_general | (mc >= XQ_MAX_MOVES);
    if (R.role == 0) {
        // getWinner: colour of the first General in square order (SURVEY F4)
        const int gen_red = mover ? st.gen_opp : gen_own, gen_black = mover ? gen_own : st.gen_opp;
        const int win = took_general ? mover : (gen_red < gen_black ? RED : BLACK);
        bk.pend = 1u | ((uint32_t)mover << 2) | ((uint32_t)over << 3) | ((uint32_t)win << 4) | ((uint32_t)mc << 8) | (pl.total << 16);
        bk.pend_p = p;
        bk.pend_tr0 = (uint32_t)XQ_ACTION(from, to) | (pl.total << 16) | ((uint32_t)((over ? 1 : 0) | ((over ? win : NOCOLOR) << 1)) << 24);
    }
    // the other side is to move -- or, after the last move of a game, Red from the opening (ChessBoard::reset): selects, no branch
    const Bits90 o_red = team_open_red(), o_black = team_open_black(), o_occT = team_open_occT();
    st.sq_own = over ? R.open_red : sq_opp; st.sq_opp = over ? R.open_black : sq_own;
    st.own = Bits90{over ? o_red.w0 : opp.w0, over ? o_red.w1 : opp.w1, over ? o_red.w2 : opp.w2};
    st.opp = Bits90{over ? o_black.w0 : own.w0, over ? o_black.w1 : own.w1, over ? o_black.w2 : own.w2};
    st.occT = Bits90{over ? o_occT.w0 : occT.w0, over ? o_occT.w1 : occT.w1, over ? o_occT.w2 : occT.w2};
    st.gen_own = over ? 4 : st.gen_opp; st.gen_opp = over ? 85 : gen_own;
    st.move_count = over ? 0 : mc; st.player = over ? RED : (mover ^ 1);
    if (pl.total == 0) {   // no legal action: the episode loop ends (chessai.cpp:100-103); the slot restarts (the counter advanced above)
        const uint32_t c = st.ctr; team_reset(R, st); st.ctr = c;
        if (R.role == 0) { bk.pend = 2; bk.pend_p = p; bk.pend_tr0 = (uint32_t)XQ_ACTION_NONE | ((uint32_t)(1 | (NOCOLOR << 1)) << 24); }
    }
    if (view) team_view_store<KB>(R, st, view, lane);
}

// ---- record <-> slots (once per launch) ---------------------------------------------------------------------------------------
// The three bitboards of a record come out of the 12 nibble words WITHOUT a per-piece loop (the loop below runs at the densest board of a
// warp: it used to spend ~35 of its ~70 instructions per piece on single-bit masks):
//   row-major: a flag per nibble (occupied / Black), 8 flags of a word compressed into a byte (three shift-or-mask steps), four bytes = a word;
//   column-major: the 9 bits of a rank spread to stride 10 (three multiplications that place bit c at 10 c, cross terms masked away) and
//   shifted up by the row.
XQ_HD uint32_t compress_nibble_flags(uint32_t x) {      // flags in bits 0, 4, ..., 28 -> bits 0..7
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    return (x | (x >> 12)) & 0xFFu;
}
// which (0: every piece, 1: Red, 2: Black) of the 12 words as a row-major bitboard
XQ_HD Bits90 record_bitboard(const uint32_t (&w)[12], int which) {
    uint32_t b[3] = {0, 0, 0};
#pragma unroll
    for (int i = 0; i < 12; ++i) {
        const uint32_t nz = (w[i] | (w[i] >> 1) | (w[i] >> 2) | (w[i] >> 3)) & 0x11111111u, hi = (w[i] >> 3) & 0x11111111u;
        uint32_t f = which == 0 ? nz : (which == 1 ? (nz & ~hi) : hi);
        if (i == 11) f &= 0x00000011u;                 // squares 88, 89; the rest of the last word is padding
        b[i >> 2] |= compress_nibble_flags(f) << (8 * (i & 3));
    }
    return Bits90{b[0], b[1], b[2]};
}
// row-major (bit 9 r + c) -> column-major (bit 10 c + r)
XQ_HD Bits90 transpose_bitboard(const Bits90& o) {
    uint32_t t0 = 0, t1 = 0, t2 = 0;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const int pos = 9 * r;
        const uint32_t lo = pos < 32 ? o.w0 : (pos < 64 ? o.w1 : o.w2), hi = pos < 32 ? o.w1 : o.w2;
        const uint32_t x = ((pos & 31) + 9 <= 32 ? lo >> (pos & 31) : funnel_r(lo, hi, pos & 31)) & 0x1FFu;
        const uint32_t s0 = ((x & 0xFu) * 0x08040201u) & 0x40100401u;             // columns 0..3 -> bits 0, 10, 20, 30
        const uint32_t s1 = (((x >> 4) & 7u) * 0x04020100u) & 0x10040100u;        // columns 4..6 -> bits 40, 50, 60
        const uint32_t s2 = ((x >> 7) * 0x00008040u) & 0x00010040u;               // columns 7, 8 -> bits 70, 80
        if (r == 0) { t0 |= s0; t1 |= s1; t2 |= s2; }
        else { t0 |= s0 << r; t1 |= funnel_r(s0, s1, 32 - r); t2 |= funnel_r(s1, s2, 32 - r); }
    }
    return Bits90{t0, t1, t2};
}

// put(slot 0..31, square); returns false for a board whose piece counts exceed a standard set (left to the generic kernel)
template <class PUT>
XQ_HD bool team_unpack_record(const uint32_t (&w)[12], Bits90& red, Bits90& black, Bits90& occT, PUT&& put) {
    bool ok = true;
    uint64_t cnt = 0;   // 4-bit counter per piece code
#pragma unroll
    for (int wi = 0; wi < 12; ++wi) {
        // one iteration per OCCUPIED square of the word (a board holds <= 32 pieces on 90 squares), lowest square first
        uint32_t nz = (w[wi] | (w[wi] >> 1) | (w[wi] >> 2) | (w[wi] >> 3)) & 0x11111111u;
        if (wi == 11) nz &= 0x00000011u;            // squares 88, 89; the rest of the last word is padding
        while (nz) {
            const int sh = ffs32(nz) - 1;           // 4 * (square within the word)
            nz &= nz - 1;
            const int s = wi * 8 + (sh >> 2);
            const int code = (int)((w[wi] >> sh) & 15u);
            const int t = type_of(code);
            const int ord = (int)((cnt >> (4 * code)) & 15);
            if (code == 15 || ord >= slot_cap(t)) { ok = false; }
            else {
                put((code >= 8 ? 16 : 0) + slot_base(t) + ord, s);
                cnt += 1ull << (4 * code);
            }
        }
    }
    // (a board that is not ok is discarded by the caller: its bitboards may hold pieces the loop did not place)
    red = record_bitboard(w, 1);
    black = record_bitboard(w, 2);
    occT = transpose_bitboard(Bits90{red.w0 | black.w0, red.w1 | black.w1, red.w2 | black.w2});
    return ok;
}

// The same with ONE loop over the pieces of the board, lowest square first, instead of one loop per record word: a warp then runs as many
// iterations as its densest board has pieces (<= 32 for a standard set) -- the per-word loops add up the densest word of each of the 12
// word positions over the warp's 32 boards (~50).  The piece code of a square needs the record at a run-time word index: m / stride is a
// scratch slice of >= 12 words laid out [word][thread] (the view memory of the board-per-thread kernels, free at that point).
template <class PUT>
XQ_HD bool team_unpack_record_m(const uint32_t (&w)[12], uint32_t* m, int stride, Bits90& red, Bits90& black, Bits90& occT, PUT&& put) {
#pragma unroll
    for (int i = 0; i < 12; ++i) m[i * stride] = w[i];
    red = record_bitboard(w, 1);
    black = record_bitboard(w, 2);
    uint32_t o0 = red.w0 | black.w0, o1 = red.w1 | black.w1, o2 = red.w2 | black.w2;
    occT = transpose_bitboard(Bits90{o0, o1, o2});
    bool ok = true;
    uint64_t cnt = 0;   // 4-bit counter per piece code
    while ((o0 | o1 | o2) != 0u) {
        const bool z0 = o0 == 0u, z1 = o1 == 0u;
        const uint32_t word = z0 ? (z1 ? o2 : o1) : o0;
        const int s = (z0 ? (z1 ? 64 : 32) : 0) + ffs32(word) - 1;
        const uint32_t rest = word & (word - 1u);
        o0 = z0 ? o0 : rest; o1 = (z0 && !z1) ? rest : o1; o2 = (z0 && z1) ? rest : o2;
        const int code = (int)((m[(s >> 3) * stride] >> (4 * (s & 7))) & 15u);
        const int t = type_of(code);
        const int ord = (int)((cnt >> (4 * code)) & 15);
        if (code == 15 || ord >= slot_cap(t)) { ok = false; }
        else {
            put((code >= 8 ? 16 : 0) + slot_base(t) + ord, s);
            cnt += 1ull << (4 * code);
        }
    }
    return ok;
}

// one colour only (side 0 Red, 1 Black): its 16 slots put(slot 0..15, square), its bitboard and its part of the column-major
// occupancy -- the two colours of a board can be unpacked by two warps at once (act_team_kernel)
template <class PUT>
XQ_HD bool team_unpack_side(const uint32_t (&w)[12], int side, Bits90& bb, Bits90& occT, PUT&& put) {
    bool ok = true;
    uint32_t cnt = 0;   // 4-bit counter per piece type
#pragma unroll
    for (int wi = 0; wi < 12; ++wi) {
        const uint32_t hi = (w[wi] >> 3) & 0x11111111u;                                      // nibble >= 8: Black (or the invalid code 15)
        uint32_t nz = (w[wi] | (w[wi] >> 1) | (w[wi] >> 2)) & 0x11111111u;                   // nibble & 7 != 0
        nz = side ? hi : (nz & ~hi);
        if (wi == 11) nz &= 0x00000011u;
        while (nz) {
            const int sh = ffs32(nz) - 1;
            nz &= nz - 1;
            const int s = wi * 8 + (sh >> 2);
            const int code = (int)((w[wi] >> sh) & 15u);
            const int t = code - (side ? 7 : 0);                                             // 1..7, or 8 for code 15, or 1 for code 8 = Black General
            const int ord = (int)((cnt >> (4 * (t & 7))) & 15u);
            if (t > 7 || ord >= slot_cap(t)) { ok = false; }
            else {
                put(slot_base(t) + ord, s);
                cnt += 1u << (4 * t);
            }
        }
    }
    bb = record_bitboard(w, side ? 2 : 1);
    occT = transpose_bitboard(bb);
    return ok;
}

}  // namespace xq
