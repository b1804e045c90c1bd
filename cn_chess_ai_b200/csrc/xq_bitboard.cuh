// xq_bitboard.cuh -- per-piece move COUNT (+ a 32-bit descriptor) and k-th-move DECODE (from the descriptor) on 90-bit occupancy bitboards.
//
// Used by the team kernels (xq_rollout_team.cuh): the pieces a thread owns are piece-type uniform
// across a warp, so every function here runs without divergence across a warp.  Sliders are
// O(1): the rank / file occupancy is pulled out of the row-major / column-major bitboards with a
// funnel shift and the first and second blocker on each ray come from ffs/clz -- no per-square
// loops.  Emission order is the reference's (SURVEY Appendix A.3): direction order as written in
// generate*Moves (src/chessboard.cpp:149-283), distance ascending along a ray.
//
// Host-compilable (tests/hostsim) so the CPU suite can diff count+decode against the oracle.
#pragma once
#include <stdint.h>

#include "xq_rules.cuh"

namespace xq {

#if defined(__CUDA_ARCH__)
XQ_HD int ffs32(uint32_t x) { return __ffs((int)x); }          // 1-based, 0 if x == 0
XQ_HD int clz32(uint32_t x) { return __clz((int)x); }
XQ_HD int popc32(uint32_t x) { return __popc(x); }
XQ_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, int sh) { return __funnelshift_r(lo, hi, sh); }
// PTX shl.b32 clamps the shift amount (n > 31 gives 0): the three words of a single-bit mask without selects
XQ_HD uint32_t shl_clamp(uint32_t x, uint32_t n) { uint32_t r; asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n)); return r; }
#else
XQ_HD int ffs32(uint32_t x) { return __builtin_ffs((int)x); }
XQ_HD int clz32(uint32_t x) { return x ? __builtin_clz(x) : 32; }
XQ_HD int popc32(uint32_t x) { return __builtin_popcount(x); }
XQ_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, int sh) { return (uint32_t)((((uint64_t)hi << 32) | lo) >> (sh & 31)); }
XQ_HD uint32_t shl_clamp(uint32_t x, uint32_t n) { return n > 31u ? 0u : x << n; }
#endif

// Branch-free word multiplexer: m = all ones picks b, m = 0 picks a (one LOP3).  Nested ternaries on a run-time word index were
// compiled into branch regions with predicated moves (21 BSSY regions per ply in the generator); masks taken from the index bits
// with two shifts are plain arithmetic.
XQ_HD uint32_t mux(uint32_t a, uint32_t b, uint32_t m) { return a ^ ((a ^ b) & m); }
XQ_HD uint32_t bit_to_mask(int x, int bit) { return (uint32_t)((int32_t)((uint32_t)x << (31 - bit)) >> 31); }   // all ones iff bit `bit` of x is set

// 90-bit set in three words.  Row-major index = row*9+col; column-major index = col*10+row.
struct Bits90 {
    uint32_t w0, w1, w2;
    // word (i >> 5) for a bit index i in [0, 96); indices outside read w0..w2 of some word (callers discard the result)
    XQ_HD uint32_t word_of_bit(int i) const { return mux(mux(w0, w1, bit_to_mask(i, 5)), w2, bit_to_mask(i, 6)); }
    XQ_HD uint32_t word(int i) const { return mux(mux(w0, w1, bit_to_mask(i, 0)), w2, bit_to_mask(i, 1)); }
    XQ_HD bool test(int i) const { return (word_of_bit(i) >> (i & 31)) & 1u; }
    XQ_HD void set(int i) { const uint32_t b = 1u << (i & 31); const int w = i >> 5; w0 |= w == 0 ? b : 0u; w1 |= w == 1 ? b : 0u; w2 |= w == 2 ? b : 0u; }
    XQ_HD void clear(int i) { const uint32_t b = ~(1u << (i & 31)); const int w = i >> 5; w0 &= w == 0 ? b : ~0u; w1 &= w == 1 ? b : ~0u; w2 &= w == 2 ? b : ~0u; }
    // single-bit mask of index i spread over the three words (computed once, applied with plain logic ops)
    static XQ_HD Bits90 bit(int i) { return Bits90{shl_clamp(1u, (uint32_t)i), shl_clamp(1u, (uint32_t)(i - 32)), shl_clamp(1u, (uint32_t)(i - 64))}; }
    XQ_HD void or_with(const Bits90& m) { w0 |= m.w0; w1 |= m.w1; w2 |= m.w2; }
    XQ_HD void andnot(const Bits90& m) { w0 &= ~m.w0; w1 &= ~m.w1; w2 &= ~m.w2; }
    // nbits (<= 10) starting at bit pos (0 <= pos < 96)
    XQ_HD uint32_t field(int pos, int nbits) const {
        const uint32_t m1 = bit_to_mask(pos, 5), m2 = bit_to_mask(pos, 6);
        const uint32_t lo = mux(mux(w0, w1, m1), w2, m2), hi = mux(w1, w2, m1) & ~m2;
        return funnel_r(lo, hi, pos & 31) & ((1u << nbits) - 1u);
    }
};
XQ_HD int rm_index(int r, int c) { return r * 9 + c; }
XQ_HD int cm_index(int r, int c) { return c * 10 + r; }
XQ_HD int row_of(int sq) { return (sq * 57) >> 9; }      // sq/9 for 0 <= sq < 128

// Position seen by the side to move: `own`/`occ` row-major, `occT` column-major (all pieces).
struct Pos {
    Bits90 own, occ, occT;
};

// One slider ray on a line occupancy L (nb bits) from index p: number of empty squares before the
// first blocker, index of the first blocker (-1: none) and of the second blocker (-1: none).
struct Ray { int empties, first, second; };
// (written with selects only: a ray is ~12 straight-line instructions, no branch for the "no blocker" case)
XQ_HD Ray ray_up(uint32_t L, int p, int nb) {      // towards higher index
    const uint32_t m = L >> (p + 1);
    const int d = ffs32(m);                          // 0: no blocker
    const uint32_t m2 = m & (m - 1);
    Ray r;
    r.empties = m ? d - 1 : nb - 1 - p;
    r.first = m ? p + d : -1;
    r.second = m2 ? p + ffs32(m2) : -1;
    return r;
}
XQ_HD Ray ray_down(uint32_t L, int p, int) {       // towards lower index
    const uint32_t m = L & ((1u << p) - 1u);
    const int top = 31 - clz32(m);                   // -1: no blocker
    const uint32_t m2 = m & ~(1u << (top & 31));
    Ray r;
    r.empties = p - top - 1;
    r.first = top;
    r.second = m2 ? 31 - clz32(m2) : -1;             // m == 0 gives m2 == 0
    return r;
}

// Sliders.  IS_CANNON: capture target is the SECOND blocker (src/chessboard.cpp:220-246, :399-421),
// else the first (:198-218, :382-397).  Ray order E, W, S(row+1), N = (0,1),(0,-1),(1,0),(-1,0).
// The generator runs ONCE per ply: it returns the count and a 32-bit DESCRIPTOR -- per ray k a byte
// (number of empty squares before the first blocker) | (distance of the capture square, 0 = none) << 4 --
// from which the k-th destination (reference order) is decoded without touching the board again.
template <bool IS_CANNON>
XQ_HD int slider_desc(const Pos& P, int sq, uint32_t* desc) {
    const int r = row_of(sq), c = sq - 9 * r;
    const uint32_t rank = P.occ.field(9 * r, 9), file = P.occT.field(10 * c, 10);
    int total = 0;
    uint32_t d = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const bool horiz = k < 2;
        const int p = horiz ? c : r;
        const Ray ray = (k & 1) ? ray_down(horiz ? rank : file, p, horiz ? 9 : 10)
                                : ray_up(horiz ? rank : file, p, horiz ? 9 : 10);
        const int tgt = IS_CANNON ? ray.second : ray.first;
        const int s = horiz ? 9 * r + tgt : 9 * tgt + c;                      // tgt == -1 reads some bit: discarded
        const bool cap = (tgt >= 0) & !P.own.test(s);
        const int capdist = cap ? ((k & 1) ? p - tgt : tgt - p) : 0;
        d |= ((uint32_t)ray.empties | ((uint32_t)capdist << 4)) << (8 * k);
        total += ray.empties + (cap ? 1 : 0);
    }
    *desc = d;
    return total;
}
XQ_HD int slider_decode(uint32_t desc, int sq, int want) {
    int to = sq;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int e = (desc >> (8 * k)) & 15, capdist = (desc >> (8 * k + 4)) & 15;
        const int cnt = e + (capdist ? 1 : 0);
        const int step = k == 0 ? 1 : (k == 1 ? -1 : (k == 2 ? 9 : -9));
        if (want >= 0 && want < cnt) to = sq + step * (want < e ? want + 1 : capdist);
        want -= cnt;                      // once negative it stays negative: exactly one ray matches
    }
    return to;
}

// Leapers: bit k of the returned mask = direction k (reference order) is playable; the destinations are recomputed by
// *_dir().  color: RED/BLACK of the piece.
// Every square a leaper looks at lies within +-20 of its own square, so instead of a dynamic 3-word bit test per
// square (two selects + shift + and, 16 of them for a horse) the 41 bits around the piece are pulled out of a
// bitboard ONCE with two funnel shifts; after that every test is a compile-time bit position.  Squares beyond the
// board read as empty -- the row / column bounds are tested separately, as the reference does (isInsideBoard).
struct Win41 {
    uint32_t lo, hi;                     // bit (off + 20) = board bit (sq + off), off in [-20, 20]
    XQ_HD uint32_t at(int off) const { const int p = off + 20; return (p < 32 ? lo >> p : hi >> (p - 32)) & 1u; }
};
XQ_HD Win41 window(const Bits90& b, int sq) {
    const int q = sq + 12;               // (sq - 20) + 32: bit index into the padded word array A = {0, w0, w1, w2, 0, 0}
    const uint32_t m1 = bit_to_mask(q, 5), m2 = bit_to_mask(q, 6);      // word index q >> 5 in 0..3; wanted: A[wi], A[wi+1], A[wi+2]
    const uint32_t b0 = b.w1 & m2, b1 = mux(b.w0, b.w2, m2), b2 = b.w1 & ~m2, b3 = b.w2 & ~m2;      // A[wi & 2 ...]
    const uint32_t x0 = mux(b0, b1, m1), x1 = mux(b1, b2, m1), x2 = mux(b2, b3, m1);
    return Win41{funnel_r(x0, x1, q & 31), funnel_r(x1, x2, q & 31)};
}
XQ_HD int general_dir(int k) { return k == 0 ? 9 : (k == 1 ? -9 : (k == 2 ? 1 : -1)); }           // :150
XQ_HD uint32_t general_mask(const Pos& P, int sq) {                                               // :149-160, :328-343
    const int r = row_of(sq), c = sq - 9 * r;
    const Win41 own = window(P.own, sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int nr = r + (k == 0 ? 1 : (k == 1 ? -1 : 0)), nc = c + (k == 2 ? 1 : (k == 3 ? -1 : 0));
        m |= ((in_any_palace(nr, nc) ? 1u : 0u) & ~own.at(k == 0 ? 9 : (k == 1 ? -9 : (k == 2 ? 1 : -1)))) << k;
    }
    return in_any_palace(r, c) ? m : 0u;
}
XQ_HD int advisor_dir(int k) { return k == 0 ? 10 : (k == 1 ? 8 : (k == 2 ? -8 : -10)); }         // :163
XQ_HD uint32_t advisor_mask(const Pos& P, int sq, int color) {                                    // :162-177
    const int r = row_of(sq), c = sq - 9 * r;
    const Win41 own = window(P.own, sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int nr = r + (k < 2 ? 1 : -1), nc = c + ((k & 1) ? -1 : 1);
        m |= ((in_palace_of(color, nr, nc) ? 1u : 0u) & ~own.at(k == 0 ? 10 : (k == 1 ? 8 : (k == 2 ? -8 : -10)))) << k;
    }
    return m;
}
XQ_HD int elephant_dir(int k) { return k == 0 ? 20 : (k == 1 ? 16 : (k == 2 ? -16 : -20)); }      // :180
XQ_HD uint32_t elephant_mask(const Pos& P, int sq, int color) {                                   // :179-196, :355-367
    const int r = row_of(sq), c = sq - 9 * r;
    const Win41 own = window(P.own, sq), occ = window(P.occ, sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int dr = k < 2 ? 2 : -2, dc = (k & 1) ? -2 : 2;
        const int nr = r + dr, nc = c + dc;
        const bool side_ok = color == RED ? (nr <= 4 && r < 5) : (nr >= 5 && r >= 5);
        const int d = k == 0 ? 20 : (k == 1 ? 16 : (k == 2 ? -16 : -20));
        m |= (((inside(nr, nc) & side_ok) ? 1u : 0u) & ~occ.at(d / 2) & ~own.at(d)) << k;
    }
    return m;
}
XQ_HD int horse_dir(int k) {                                                                       // :249
    const int a = (k & 2) ? -1 : 1, b = (k & 1) ? -1 : 1;
    return k < 4 ? 9 * a + 2 * b : 18 * a + b;
}
XQ_HD uint32_t horse_mask(const Pos& P, int sq) {                                                 // :248-263, :369-380
    const int r = row_of(sq), c = sq - 9 * r;
    const Win41 own = window(P.own, sq), occ = window(P.occ, sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int a = (k & 2) ? -1 : 1, b = (k & 1) ? -1 : 1;
        const int nr = r + (k < 4 ? a : 2 * a), nc = c + (k < 4 ? 2 * b : b);
        const int leg = k < 4 ? b : 9 * a, dest = k < 4 ? 9 * a + 2 * b : 18 * a + b;       // offsets from sq: compile-time after unrolling
        m |= ((inside(nr, nc) ? 1u : 0u) & ~occ.at(leg) & ~own.at(dest)) << k;
    }
    return m;
}
XQ_HD int soldier_dir(int k, int color) { return k == 0 ? (color == RED ? 9 : -9) : (k == 1 ? -1 : 1); }   // :267-281
XQ_HD uint32_t soldier_mask(const Pos& P, int sq, int color) {                                    // :265-283
    const int r = row_of(sq), c = sq - 9 * r;
    const Win41 own = window(P.own, sq);
    uint32_t m = 0;
    const int nr = r + (color == RED ? 1 : -1);
    m |= ((unsigned)nr < 10u ? 1u : 0u) & ~(color == RED ? own.at(9) : own.at(-9));
    const uint32_t crossed = (color == RED ? r > 4 : r < 5) ? 1u : 0u;
    m |= (crossed & (c > 0 ? 1u : 0u) & ~own.at(-1)) << 1;
    m |= (crossed & (c < 8 ? 1u : 0u) & ~own.at(1)) << 2;
    return m;
}
// ---- geometry table (shared-memory piece table) ---------------------------------------------------------------------------------
// Everything a leaper's mask needs that depends on the SQUARE and the colour only -- board bounds, palaces, the river -- is one table
// word per (colour, square): the kernels keep the 2 x 128 words in shared memory and the *_mask_g functions AND it onto the bits taken
// from the bitboards.  In the rollout kernels (bound by the integer ALU pipe) this moves ~10 % of a ply's instructions -- the row /
// column arithmetic and 3-7 compares per direction -- to one shared-memory load per piece.  Entries 90..127 are 0: a captured piece
// (square 127) gets an empty mask without a select.
//   bits 0-7 Horse | 8-11 Elephant | 12-15 Advisor | 16-19 General | 20-22 Soldier   (direction order of generate*Moves)
constexpr int kGeoWords = 256;                     // [colour][128]
XQ_HD constexpr uint32_t geo_entry(int color, int sq) {
    if (sq >= 90) return 0u;
    const int r = sq / 9, c = sq - 9 * r;
    uint32_t g = 0;
    for (int k = 0; k < 8; ++k) {                  // :248-263
        const int a = (k & 2) ? -1 : 1, b = (k & 1) ? -1 : 1;
        const int nr = r + (k < 4 ? a : 2 * a), nc = c + (k < 4 ? 2 * b : b);
        g |= (inside(nr, nc) ? 1u : 0u) << k;
    }
    for (int k = 0; k < 4; ++k) {
        {                                          // Elephant :179-196, :355-367
            const int nr = r + (k < 2 ? 2 : -2), nc = c + ((k & 1) ? -2 : 2);
            const bool side_ok = color == RED ? (nr <= 4 && r < 5) : (nr >= 5 && r >= 5);
            g |= ((inside(nr, nc) & side_ok) ? 1u : 0u) << (8 + k);
        }
        {                                          // Advisor :162-177
            const int nr = r + (k < 2 ? 1 : -1), nc = c + ((k & 1) ? -1 : 1);
            g |= (in_palace_of(color, nr, nc) ? 1u : 0u) << (12 + k);
        }
        {                                          // General :149-160, :328-343
            const int nr = r + (k == 0 ? 1 : (k == 1 ? -1 : 0)), nc = c + (k == 2 ? 1 : (k == 3 ? -1 : 0));
            g |= ((in_any_palace(nr, nc) & in_any_palace(r, c)) ? 1u : 0u) << (16 + k);
        }
    }
    {                                              // Soldier :265-283
        const int nr = r + (color == RED ? 1 : -1);
        const bool crossed = color == RED ? r > 4 : r < 5;
        g |= ((unsigned)nr < 10u ? 1u : 0u) << 20;
        g |= ((crossed && c > 0) ? 1u : 0u) << 21;
        g |= ((crossed && c < 8) ? 1u : 0u) << 22;
    }
    return g;
}
struct GeoTable { uint32_t v[kGeoWords]; };
constexpr GeoTable make_geo_table() {
    GeoTable t{};
    for (int i = 0; i < kGeoWords; ++i) t.v[i] = geo_entry(i >> 7, i & 127);
    return t;
}
#if defined(__CUDACC__)
static __device__ const GeoTable d_geo = make_geo_table();       // built by the compiler; the kernels copy it into shared memory
#endif
XQ_HD uint32_t geo_word(int i) {
#if defined(__CUDA_ARCH__)
    return d_geo.v[i];
#else
    return geo_entry(i >> 7, i & 127);
#endif
}
// ---- board views: where the generators read the three bitboards from -------------------------------------------------------------
// RegView: the bitboards live in registers (three words each); a run-time word index costs arithmetic -- two mask builds and two to four
// LOP3 per selected word (mux above), ~12 integer-ALU instructions per 41-bit window, ~10 per rank / file, ~8 per bit test.
struct RegView {
    Bits90 own, occ, occT;
    XQ_HD Win41 win_own(int sq) const { return window(own, sq); }
    XQ_HD Win41 win_occ(int sq) const { return window(occ, sq); }
    XQ_HD uint32_t rank(int r) const { return occ.field(9 * r, 9); }
    XQ_HD uint32_t file(int c) const { return occT.field(10 * c, 10); }
    XQ_HD bool own_test(int s) const { return own.test(s); }
};
// MemView: a copy of the same bitboards in (shared) memory, one private slice per thread laid out [word][thread]: the bank of an access is
// the thread's lane whatever the word index, so a RUN-TIME word index is conflict-free and costs one address computation -- the word
// selection moves from the integer ALU (the pipe that bounds the rollout kernels) to the load / store unit.  Three arrays of 8 words,
// own | occ (= own | opp) | occT, each stored padded as {0, w0, w1, w2, 0, 0, 0, 0}: a window or a field that hangs over either end of
// the board (and every access of a captured piece, square 127) reads zeros.  The registers stay the master copy; view_store writes the
// arrays after every change of the board.
constexpr int kViewWords = 24;
struct MemView {
    const uint32_t* m;       // this thread's slice: word i of array a at m[(8 a + i) * stride]
    int stride;
    XQ_HD uint32_t w(int a, int i) const { return m[(8 * a + i) * stride]; }
    XQ_HD Win41 win(int a, int sq) const {
        const int q = sq + 12, wi = q >> 5;             // bit (sq - 20) + 32 of the padded array; wi = 0..4
        const uint32_t x0 = w(a, wi), x1 = w(a, wi + 1), x2 = w(a, wi + 2);
        return Win41{funnel_r(x0, x1, q & 31), funnel_r(x1, x2, q & 31)};
    }
    XQ_HD Win41 win_own(int sq) const { return win(0, sq); }
    XQ_HD Win41 win_occ(int sq) const { return win(1, sq); }
    XQ_HD uint32_t fld(int a, int pos, int nbits) const {
        const int wi = pos >> 5;                         // 0..3
        return funnel_r(w(a, 1 + wi), w(a, 2 + wi), pos & 31) & ((1u << nbits) - 1u);
    }
    XQ_HD uint32_t rank(int r) const { return fld(1, 9 * r, 9); }
    XQ_HD uint32_t file(int c) const { return fld(2, 10 * c, 10); }
    XQ_HD bool own_test(int s) const { return (w(0, 1 + ((s >> 5) & 3)) >> (s & 31)) & 1u; }      // an index off the board reads some bit: callers discard it
};
XQ_HD void view_init(uint32_t* m, int stride) {          // the padding words, once
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        m[(8 * a) * stride] = 0u;
#pragma unroll
        for (int i = 4; i < 8; ++i) m[(8 * a + i) * stride] = 0u;
    }
}
XQ_HD void view_store(uint32_t* m, int stride, const Bits90& own, const Bits90& opp, const Bits90& occT) {
    m[1 * stride] = own.w0; m[2 * stride] = own.w1; m[3 * stride] = own.w2;
    m[9 * stride] = own.w0 | opp.w0; m[10 * stride] = own.w1 | opp.w1; m[11 * stride] = own.w2 | opp.w2;
    m[17 * stride] = occT.w0; m[18 * stride] = occT.w1; m[19 * stride] = occT.w2;
}

// the masks of the leapers on a view, with the geometry from the table word g = geo[colour * 128 + sq]
template <class V>
XQ_HD uint32_t horse_mask_g(const V& v, int sq, uint32_t g) {
    const Win41 own = v.win_own(sq), occ = v.win_occ(sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int a = (k & 2) ? -1 : 1, b = (k & 1) ? -1 : 1;
        const int leg = k < 4 ? b : 9 * a, dest = k < 4 ? 9 * a + 2 * b : 18 * a + b;
        m |= (occ.at(leg) | own.at(dest)) << k;
    }
    return ~m & g & 0xFFu;
}
template <class V>
XQ_HD uint32_t elephant_mask_g(const V& v, int sq, uint32_t g) {
    const Win41 own = v.win_own(sq), occ = v.win_occ(sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int d = k == 0 ? 20 : (k == 1 ? 16 : (k == 2 ? -16 : -20));
        m |= (occ.at(d / 2) | own.at(d)) << k;
    }
    return ~m & (g >> 8) & 0xFu;
}
template <class V>
XQ_HD uint32_t advisor_mask_g(const V& v, int sq, uint32_t g) {
    const Win41 own = v.win_own(sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) m |= own.at(k == 0 ? 10 : (k == 1 ? 8 : (k == 2 ? -8 : -10))) << k;
    return ~m & (g >> 12) & 0xFu;
}
template <class V>
XQ_HD uint32_t general_mask_g(const V& v, int sq, uint32_t g) {
    const Win41 own = v.win_own(sq);
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) m |= own.at(k == 0 ? 9 : (k == 1 ? -9 : (k == 2 ? 1 : -1))) << k;
    return ~m & (g >> 16) & 0xFu;
}
template <class V>
XQ_HD uint32_t soldier_mask_g(const V& v, int sq, int color, uint32_t g) {
    const Win41 own = v.win_own(sq);
    const uint32_t m = (color == RED ? own.at(9) : own.at(-9)) | (own.at(-1) << 1) | (own.at(1) << 2);
    return ~m & (g >> 20) & 0x7u;
}
// slider_desc (above) on a view; `cannon`: the capture square is the second blocker
template <class V>
XQ_HD int slider_desc_v(const V& v, int sq, bool cannon, uint32_t* desc) {
    const int r = row_of(sq), c = sq - 9 * r;
    const uint32_t rank = v.rank(r), file = v.file(c);
    int total = 0;
    uint32_t d = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const bool horiz = k < 2;
        const int p = horiz ? c : r;
        const Ray ray = (k & 1) ? ray_down(horiz ? rank : file, p, horiz ? 9 : 10) : ray_up(horiz ? rank : file, p, horiz ? 9 : 10);
        const int tgt = cannon ? ray.second : ray.first;
        const int s = horiz ? 9 * r + tgt : 9 * tgt + c;                      // tgt == -1 reads some bit: discarded
        const bool cap = (tgt >= 0) & !v.own_test(s);
        const int capdist = cap ? ((k & 1) ? p - tgt : tgt - p) : 0;
        d |= ((uint32_t)ray.empties | ((uint32_t)capdist << 4)) << (8 * k);
        total += ray.empties + (cap ? 1 : 0);
    }
    *desc = d;
    return total;
}

// index of the j-th (0-based) set bit of an 8-bit mask
XQ_HD int nth_set_bit(uint32_t m, int j) {
#pragma unroll
    for (int i = 0; i < 7; ++i) { if (j > 0) { m &= m - 1; --j; } }
    return ffs32(m) - 1;
}

// Uniform entry points.  piece_count<TYPE>: number of moves of the piece of `type` / `color` on `sq` plus the descriptor
// (sliders: see slider_desc; leapers: the direction mask).  piece_decode<TYPE>: the want-th destination in reference
// order from the descriptor alone.
template <int TYPE>
XQ_HD int piece_count(const Pos& P, int sq, int color, uint32_t* desc) {
    if (TYPE == CHARIOT) return slider_desc<false>(P, sq, desc);
    if (TYPE == CANNON) return slider_desc<true>(P, sq, desc);
    uint32_t m;
    if (TYPE == GENERAL) m = general_mask(P, sq);
    else if (TYPE == ADVISOR) m = advisor_mask(P, sq, color);
    else if (TYPE == ELEPHANT) m = elephant_mask(P, sq, color);
    else if (TYPE == HORSE) m = horse_mask(P, sq);
    else m = soldier_mask(P, sq, color);
    *desc = m;
    return popc32(m);
}
template <int TYPE>
XQ_HD int piece_decode(uint32_t desc, int sq, int color, int want) {
    if (TYPE == CHARIOT || TYPE == CANNON) return slider_decode(desc, sq, want);
    const int k = nth_set_bit(desc, want);
    int d;
    if (TYPE == GENERAL) d = general_dir(k);
    else if (TYPE == ADVISOR) d = advisor_dir(k);
    else if (TYPE == ELEPHANT) d = elephant_dir(k);
    else if (TYPE == HORSE) d = horse_dir(k);
    else d = soldier_dir(k, color);
    return sq + d;
}

XQ_HD int piece_count_dyn(int type, const Pos& P, int sq, int color, uint32_t* desc) {
    switch (type) {
        case GENERAL: return piece_count<GENERAL>(P, sq, color, desc);
        case ADVISOR: return piece_count<ADVISOR>(P, sq, color, desc);
        case ELEPHANT: return piece_count<ELEPHANT>(P, sq, color, desc);
        case HORSE: return piece_count<HORSE>(P, sq, color, desc);
        case CHARIOT: return piece_count<CHARIOT>(P, sq, color, desc);
        case CANNON: return piece_count<CANNON>(P, sq, color, desc);
        case SOLDIER: return piece_count<SOLDIER>(P, sq, color, desc);
        default: *desc = 0; return 0;
    }
}
XQ_HD int piece_decode_dyn(int type, uint32_t desc, int sq, int color, int want) {
    switch (type) {
        case GENERAL: return piece_decode<GENERAL>(desc, sq, color, want);
        case ADVISOR: return piece_decode<ADVISOR>(desc, sq, color, want);
        case ELEPHANT: return piece_decode<ELEPHANT>(desc, sq, color, want);
        case HORSE: return piece_decode<HORSE>(desc, sq, color, want);
        case CHARIOT: case CANNON: return slider_decode(desc, sq, want);
        case SOLDIER: return piece_decode<SOLDIER>(desc, sq, color, want);
        default: return sq;
    }
}
// count, and (want >= 0) the want-th destination: the two steps above in one call (host differential tests)
XQ_HD int piece_moves_dyn(int type, const Pos& P, int sq, int color, int want, int* to) {
    uint32_t desc;
    const int n = piece_count_dyn(type, P, sq, color, &desc);
    if (want >= 0) *to = piece_decode_dyn(type, desc, sq, color, want);
    return n;
}

// Board summary straight from the 12 nibble words of a record, without a per-square loop (step_kernel): material per colour
// (ChessAI::evaluateBoard, src/chessai.cpp:311-342) and the lowest square holding each General (ChessBoard::checkGameOver :286-309,
// getWinner :312-320), 127 = none.  Bit-plane SIMD: plane j of the words 4g .. 4g+3 is packed into ONE word (bit 4i + k = bit j of
// nibble i of word 4g + k), a piece code is then a 4-input boolean function of the planes and its count a popcount.
struct WordSummary { int mat_red, mat_black, gen_red, gen_black; };
XQ_HD WordSummary summarize_words(const uint32_t (&w)[12]) {
    uint32_t P[3][4];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t acc = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t x = w[4 * g + k];
                acc |= (k >= j ? x << (k - j) : x >> (j - k)) & (0x11111111u << k);
            }
            P[g][j] = acc;
        }
    int n[15];      // pieces per code 1..14
#pragma unroll
    for (int code = 1; code <= 14; ++code) {
        int c = 0;
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            uint32_t m = 0xFFFFFFFFu;
#pragma unroll
            for (int j = 0; j < 4; ++j) m &= ((code >> j) & 1) ? P[g][j] : ~P[g][j];
            c += popc32(m);
        }
        n[code] = c;
    }
    WordSummary s;      // piece_score / 5: 200, 4, 4, 8, 18, 9, 2
    s.mat_red = 5 * (200 * n[1] + 4 * (n[2] + n[3]) + 8 * n[4] + 18 * n[5] + 9 * n[6] + 2 * n[7]);
    s.mat_black = 5 * (200 * n[8] + 4 * (n[9] + n[10]) + 8 * n[11] + 18 * n[12] + 9 * n[13] + 2 * n[14]);
    int gen[2] = {127, 127};
#pragma unroll
    for (int side = 0; side < 2; ++side) {
        const uint32_t pat = side ? 0x88888888u : 0x11111111u;      // nibble == 1 (Red General) / == 8 (Black General)
#pragma unroll
        for (int i = 11; i >= 0; --i) {                              // descending: the lowest word with a match is written last
            const uint32_t x = w[i] ^ pat;
            const uint32_t nz = (x | (x >> 1) | (x >> 2) | (x >> 3)) & 0x11111111u;      // 1 per NON-matching nibble
            const uint32_t hit = nz ^ 0x11111111u;
            gen[side] = hit ? 8 * i + ((ffs32(hit) - 1) >> 2) : gen[side];
        }
    }
    s.gen_red = gen[0]; s.gen_black = gen[1];
    return s;
}

// Piece slots: every side has 16 fixed slots (no promotion in Xiangqi); slot -> type is static,
// which is what makes warps type-uniform.  0,1 Chariot | 2,3 Horse | 4,5 Elephant | 6,7 Advisor |
// 8 General | 9,10 Cannon | 11..15 Soldier.
XQ_HD int slot_type(int s) {
    return s < 2 ? CHARIOT : (s < 4 ? HORSE : (s < 6 ? ELEPHANT : (s < 8 ? ADVISOR : (s == 8 ? GENERAL : (s < 11 ? CANNON : SOLDIER)))));
}
XQ_HD int slot_base(int type) { return (int)((0xB9024680u >> (4 * type)) & 15u); }   // first slot of a type
XQ_HD int slot_cap(int type) { return (int)((0x52222210u >> (4 * type)) & 15u); }    // pieces of a type per side
constexpr int kDeadSq = 127;

}  // namespace xq
