// xq_dqn_fast.cu -- batched tensor-core path of the {1260,128,8100} self-play Q-network.
//
// What the reference does per ply (src/chessai.cpp:106-131): up to 3 forwards + 1 backward of a dense
// FP64 MLP at batch 1.  Here a TD update runs on a batch of B transitions (s, a, r, s', done):
//   layer 0   h = tanh(W0 x + b0): x is one-hot with <= 32 ones (src/chessai.cpp:268-289), so the
//             pre-activation is a gather-sum of <= 32 rows of W0^T read straight from the packed board
//             (FP32, exact; the 1260-wide one-hot vector is never materialised)            [l0_forward_kernel]
//   layer 1   z = W1 h + b1 over ALL 8100 outputs is the one dense contraction:
//             [B x 128] x [128 x 8100] on tcgen05 tensor cores, BF16 operands staged by TMA (128-B swizzle),
//             FP32 accumulators in TMEM, W1 tile stationary in shared memory, epilogue warps reduce the
//             row max straight out of TMEM (max_a tanh(z_a) = tanh(max_a z_a): no Q matrix, no 33M tanh)   [l1_gemm_kernel]
//   TD error  the live loop's target equals Q(s) except at index `to` (src/chessai.cpp:122-128), so delta1 is
//             one-hot per sample: q(s)[to] is a 128-long dot product, dW1 touches row `to` only, delta0 is one
//             row of W1 (as written: src/dqn.cu:406-423, SURVEY F7; or corrected)            [td_delta_kernel]
//   dW0       X^T . delta0 on tcgen05: the transposed one-hot operand tile is built in shared memory from the packed
//             boards, delta0^T (BF16 hi+lo) arrives by TMA; db0 rides along as a constant-one feature    [dw_gemm_kernel]
//   SGD       W -= lr * sum of per-sample gradients (B = 1 reproduces one reference step)     [apply_kernel]
// FP32 master weights; BF16 only as MMA operands.  Tolerance vs the FP64 oracle: |dQ| <= 2e-3.
#include <cuda.h>

#include <algorithm>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "xq_act_l0.cuh"
#include "xq_act_quant.cuh"
#include "xq_dqn_internal.cuh"
#include "xq_tc.cuh"

namespace xq {

// -DXQ_TIMELINE: per-CTA clock64 timestamps of the pipeline events of the two tcgen05 kernels (profiling builds only;
// scripts/tl_dump.py reads them back through xq_debug_timeline)
#ifdef XQ_TIMELINE
__device__ long long g_tl[2 * 160 * 64];
#define XQ_TL(kern, slot) (g_tl[((kern) * 160 + blockIdx.y * gridDim.x + blockIdx.x) * 64 + (slot)] = clock64())
#define XQ_TLV(kern, slot, v) (g_tl[((kern) * 160 + blockIdx.y * gridDim.x + blockIdx.x) * 64 + (slot)] = (v))
#else
#define XQ_TL(kern, slot) ((void)0)
#define XQ_TLV(kern, slot, v) ((void)0)
#endif

constexpr int kIn = XQ_STATE_SIZE, kHid = 128, kOut = 8100, kQRows = 90;   // Q is indexed by `to` < 90 (src/dqn.cpp:47)
[[maybe_unused]] constexpr int kGradW0 = 0;
constexpr int kGradB0 = kIn * kHid, kGradW1 = kGradB0 + kHid, kGradB1 = kGradW1 + kQRows * kHid;
constexpr int kGradSize = kGradB1 + kQRows;   // 173,018 floats: the only non-zero gradient entries of a TD step (SURVEY section 5)

// ---- GEMM tile configuration ----------------------------------------------------------------
constexpr int BM = 128;            // rows (samples) per MMA = TMEM lanes
constexpr int BN = 224;            // outputs per CTA tile: 37 tiles x 4 row splits = 148 CTAs = one per SM
constexpr int BK = 64;             // BF16 elements per 128-byte swizzle row
constexpr int kKBlocks = kHid / BK;                 // 2
constexpr int kAStages = 3;
constexpr int kNTiles = (kOut + BN - 1) / BN;       // 37
constexpr uint32_t kABytes = BM * kHid * 2;         // 32 KB: one A tile (both k-blocks)
constexpr uint32_t kBBytes = BN * kHid * 2;         // 56 KB: the stationary W1 tile
constexpr uint32_t kTmemCols = 512;                 // 2 accumulator stages x BN columns (power of two >= 448)
constexpr int kGemmThreads = 384;                   // warp 0 TMA, 1 MMA, 2 TMEM alloc, 2-3 bias-step operands, 4-11 epilogue
constexpr int kEpiWarps = 8;                        // two warps per TMEM lane quarter, each drains half of the BN columns
constexpr int kParts = 2 * kNTiles;                 // row-max partials per sample (74)
constexpr int kPartsPad = 96;                       // zpart is [row][96]: a sample's partials are 3 coalesced 128-byte reads
constexpr uint32_t kBiasBBytes = BN * BK * 2;       // 28 KB: b1 as the B operand of the bias step
constexpr uint32_t kOnesBytes = BM * BK * 2;        // 16 KB: the constant-one A operand of the bias step
constexpr size_t kGemmSmem = 1024 + kBBytes + kBiasBBytes + kOnesBytes + kAStages * kABytes + 256;

struct Fast {
    int64_t cap = 0;                                   // batch capacity of the workspace
    float *W0T = nullptr, *b0 = nullptr, *W1 = nullptr, *b1 = nullptr;          // online, FP32 master
    __nv_bfloat16* W1bf = nullptr;
    float *tW0T = nullptr, *tb0 = nullptr, *tW1 = nullptr, *tb1 = nullptr;      // target network
    __nv_bfloat16* tW1bf = nullptr;
    bool target_current = false;
    float* grad = nullptr;                             // kGradSize
    // batch workspace
    xq_env_rec* boards = nullptr;                      // staging for xq_dqn_forward_boards
    __nv_bfloat16 *Hbf = nullptr, *H2bf = nullptr;     // h(s), h(s') as MMA A operands [cap][128]
    float* Hf = nullptr;                               // h(s) FP32 [cap][128]
    float* zpart = nullptr;                            // [cap][kPartsPad] row-max partials
    float* part = nullptr;                             // [11 row tiles][8 splits][128][128] FP32 partials of the gradient contraction (L2 scratch)
    uint32_t* cb = nullptr;                            // [15][ld] compact batch, word-major: 12 board words of s | action,mover,done | reward | delta1
    float* dbpart = nullptr;                           // [8 splits][128] per-CTA sums of delta1 per action.to
    float* info_slots = nullptr;                       // [16][4] loss statistics accumulated by td_delta_kernel
    __nv_bfloat16 *d0hi = nullptr, *d0lo = nullptr;    // delta0^T [128][ld] BF16 hi / lo (B operand of the dW0 contraction)
    __nv_bfloat16 *ghi = nullptr, *glo = nullptr;      // (delta1 h)^T [128][ld] BF16 hi / lo (B operand of the dW1 contraction)
    float* q = nullptr;                                // [cap][8100] (debug path only, allocated on demand)
    int64_t q_cap = 0;
    float* info = nullptr;                             // 4 floats
    CUtensorMap tmW1, tmTW1, tmH, tmH2, tmD0hi, tmD0lo, tmGhi, tmGlo, tmCb;
    // pipelined multi-update path (td_update_pipelined): the bootstrap branch [h(s') -> row-max GEMM] of update i+1 / i+2 runs on
    // an auxiliary stream while the online branch of update i runs on the handle's stream; two slots of its buffers alternate
    __nv_bfloat16* H2bf_b = nullptr;
    float* zpart_b = nullptr;
    CUtensorMap tmH2_b;
    cudaStream_t aux = nullptr, main_hi = nullptr;
    cudaEvent_t ev_join = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_aux[2] = {nullptr, nullptr}, ev_td[2] = {nullptr, nullptr};
    // multi-GPU gradient exchange over peer memory (xq_dqn_dist_*): when connected, the compact gradient of an update is written
    // into slot `parity` of this rank's exchange buffer, which every peer maps through CUDA IPC
    uint8_t* exch = nullptr;                           // [2][kGradPad] FP32 gradient slots | flags[kMaxRanks] u32 | status u32
    uint8_t* peer[16] = {};                            // exchange buffers of all ranks (peer[rank] == exch)
    int rank = 0, world = 1, parity = 0;
    uint32_t epoch = 0;
    bool connected = false;
    uint32_t *status_host = nullptr, *status_dev = nullptr;   // mapped pinned word: epoch of the first exchange that timed out (sticky; read without a sync)
    long long timeout_ticks = 0;                       // clock64 ticks (XQ_DIST_TIMEOUT_MS, default 20 s)
    uint8_t* hg_stage = nullptr;                       // device staging of xq_dqn_dist_allgather
    uint8_t* hg_pin = nullptr;                         // pinned host staging: [send kHgCap | recv kMaxRanks x kHgCap]
    uint32_t hg_seq = 0;
    // acting (Q(s)[0..89] for every env of a self-play shard): split-precision operands, see q90_gemm_kernel
    __nv_bfloat16* W1lo = nullptr;                     // [96][128] BF16 residual of W1 rows 0..95 (W1 = W1bf + W1lo to ~16 mantissa bits)
    __nv_bfloat16 *actHhi = nullptr, *actHlo = nullptr;   // [act_cap][128] h(s) as BF16 hi + lo
    int64_t act_cap = 0, act_rows = 0;
    // fixed-point layer-0 sums carried from ply to ply (l0_act_kernel)
    int32_t *W0Q = nullptr, *b0Q = nullptr;            // [(1260 + 1)][128], [128]: rint(W0^T * 2^k), rint(b0 * 2^k)
    int32_t* zOpen = nullptr;                          // [128] sum of the opening position
    uint32_t* actMax = nullptr;                        // two slots of max |w| bits (alternating per weight version) | inv_scale (float) at [2]
    int32_t* actZ = nullptr;                           // [act_cap][128] fixed-point z0 of the board in actPrev
    uint32_t* actPrev = nullptr;                       // [act_cap][12] board words actZ belongs to
    uint64_t w_version = 1, actq_version = 0, actz_version = 0;   // online W0 / b0 version; version W0Q / actZ were built from
    int act_slot = 0;
    int64_t act_carried_n = -1;
    CUtensorMap tmActHiS[2], tmActLoS[2];              // the halves of the collector's env range (two-stream plies)
    int64_t act_sub_n = -1;
    CUtensorMap tmActHi, tmActLo, tmW1q, tmW1loq;
    int64_t tm_rows = 0;
};

// A TD batch is either a contiguous array of transitions or `n` uniform draws from a replay ring, resolved in place:
// index_b = (xq_rng(seed, b, counter) >> 1) % size   (include/xq.h: xq_replay_sample).  No gather pass, no copy.
struct BatchRef {
    const uint8_t* base;      // transitions (128 B each)
    int64_t size;             // ring size when sampled
    uint64_t seed;
    uint32_t counter;
    int sampled;
    __device__ __forceinline__ const uint8_t* at(int64_t b) const {
        const int64_t i = sampled ? (int64_t)((rng(seed, (uint64_t)b, counter) >> 1) % (uint64_t)size) : b;
        return base + i * 128;
    }
};

// ---------------------------------------------------------------------------------------------
// layer 0: one warp per board, lane owns 4 hidden units; <= 32 coalesced 512-byte row reads of W0^T
__device__ __forceinline__ float4 l0_gather(uint32_t word, int lane, const float* __restrict__ W0T, const float* __restrict__ b0) {   // word = board word `lane` (lanes 0..11)
    float4 acc = reinterpret_cast<const float4*>(b0)[lane];
    for (int wi = 0; wi < 12; ++wi) {
        uint32_t v = __shfl_sync(0xFFFFFFFFu, word, wi);
        while (v) {                                         // warp-uniform: every lane sees the same board
            const int nib = (__ffs((int)v) - 1) >> 2;
            const int code = (v >> (4 * nib)) & 15;
            v &= ~(15u << (4 * nib));
            const int row = (wi * 8 + nib) * 14 + code - 1;      // getStateRepresentation index, src/chessai.cpp:278-282
            if (code < 15 && row < kIn) {
                const float4 r = reinterpret_cast<const float4*>(W0T + (size_t)row * kHid)[lane];
                acc.x += r.x; acc.y += r.y; acc.z += r.z; acc.w += r.w;
            }
        }
    }
    return make_float4(tanhf(acc.x), tanhf(acc.y), tanhf(acc.z), tanhf(acc.w));
}
__device__ __forceinline__ void store_h_bf16(__nv_bfloat16* __restrict__ Hbf, int64_t s, int lane, const float4& h) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(h.x, h.y), hi = __floats2bfloat162_rn(h.z, h.w);
    uint2 packed;
    packed.x = *reinterpret_cast<uint32_t*>(&lo); packed.y = *reinterpret_cast<uint32_t*>(&hi);
    reinterpret_cast<uint2*>(Hbf + s * kHid)[lane] = packed;
}
__global__ void __launch_bounds__(256) l0_forward_kernel(const uint8_t* __restrict__ boards, int64_t stride_bytes, int64_t n,
                                                        const float* __restrict__ W0T, const float* __restrict__ b0,
                                                        __nv_bfloat16* __restrict__ Hbf, float* __restrict__ Hf) {
    const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (s >= n) return;
    const float4 h = l0_gather(lane < 12 ? reinterpret_cast<const uint32_t*>(boards + s * stride_bytes)[lane] : 0u, lane, W0T, b0);
    if (Hf) reinterpret_cast<float4*>(Hf + s * kHid)[lane] = h;
    store_h_bf16(Hbf, s, lane, h);
}
// Acting: h(s) for every env of a shard (8 lanes per board), written as BF16 hi + lo (h = hi + lo to ~16 mantissa bits) for the
// split-precision layer-1 contraction of q90_gemm_kernel.
//
// The pre-activation z0 = b0 + (sum of the <= 32 rows of W0^T a board selects, src/chessai.cpp:268-289) is kept PER ENV between plies
// and UPDATED from the squares a ply changed (a quiet move: -row(from, piece) +row(to, piece); a capture: one more subtraction), the
// way an efficiently-updatable evaluation network does it: 2-3 rows per ply instead of ~30.  For the update to be exact -- Q(s) must stay
// a pure function of (board, weights), or two runs that reach a position along different paths would break arg-max ties differently --
// the sum is carried in 32-bit FIXED POINT: W0Q = rint(W0 * 2^k), k chosen per weight version from max |W0|, |b0| so that 92 terms
// cannot overflow (act_quant_*_kernel).  Integer addition is associative, so "previous sum - old rows + new rows" IS the fresh sum,
// bit for bit (and wrap-around in an intermediate value is harmless).  With the reference's U(-0.05, 0.05) initialisation k = 28: a
// quantum of 3.7e-9 = the FP32 ulp of the larger weights, so the fixed-point sum is closer to the FP64 oracle than a sequential FP32 sum.
// Per env the kernel keeps the sum (512 B) and the board it belongs to (48 B); a board that differs from the remembered one in more than
// 4 squares (reset, xq_env_set_boards, another env handle) or a new weight version (`fresh_all`) takes the gather path over all rows.
__global__ void __launch_bounds__(256) act_quant_max_kernel(const float* __restrict__ W0T, const float* __restrict__ b0, uint32_t* __restrict__ slot) {
    uint32_t m = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kIn * kHid + kHid; i += gridDim.x * blockDim.x)
        m = max(m, __float_as_uint(i < kIn * kHid ? W0T[i] : b0[i - kIn * kHid]) & 0x7FFFFFFFu);      // |w| as ordered bits (NaN sorts above inf)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(slot, m);
}
__global__ void __launch_bounds__(256) act_quant_kernel(const float* __restrict__ W0T, const float* __restrict__ b0, const uint32_t* __restrict__ slot,
                                                       uint32_t* __restrict__ next_slot, int32_t* __restrict__ W0Q, int32_t* __restrict__ b0Q,
                                                       float* __restrict__ inv_scale) {
    const int k = act_quant_shift(*slot);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < (kIn + 1) * kHid + kHid; i += gridDim.x * blockDim.x) {
        if (i < kIn * kHid) W0Q[i] = act_quantize(W0T[i], k);
        else if (i < (kIn + 1) * kHid) W0Q[i] = 0;                                     // row kIn = zeros: the padding row of the lists
        else b0Q[i - (kIn + 1) * kHid] = act_quantize(b0[i - (kIn + 1) * kHid], k);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { *inv_scale = ldexpf(1.0f, -k); *next_slot = 0u; }     // the other slot serves the next weight version
}
// the sum of the opening position (ChessBoard::reset): what a restarted env carries into its next ply
__global__ void __launch_bounds__(kHid) act_zopen_kernel(const int32_t* __restrict__ W0Q, const int32_t* __restrict__ b0Q, int32_t* __restrict__ zOpen) {
    uint32_t z = (uint32_t)b0Q[threadIdx.x];
    for (int q = 0; q < XQ_SQUARES; ++q) {
        const int code = (int)((kOpening[q >> 3] >> (4 * (q & 7))) & 15u);
        if (code != 0) z += (uint32_t)W0Q[(q * 14 + code - 1) * kHid + threadIdx.x];
    }
    zOpen[threadIdx.x] = (int32_t)z;
}
// Mapping: 8 lanes per env, 4 envs per warp (the bookkeeping that finds the changed squares is warp-uniform work: 8 lanes amortise it
// four times better than 32), lane `sub` owns hidden units (i*8 + sub)*4 .. +3 for i < 4, so one load instruction reads 128
// contiguous bytes of a row per env.  tanh is evaluated as 1 - 2 / (1 + 2^(2 log2(e) |z|)) on the SFU (absolute error ~1e-7, below
// the 2^-17 relative error of the hi + lo operand split that follows).
__device__ __forceinline__ uint32_t act_nibble_flags(uint32_t x) { return (x | (x >> 1) | (x >> 2) | (x >> 3)) & 0x11111111u; }     // bit 4i: nibble i != 0
__global__ void __launch_bounds__(256) l0_act_kernel(const xq_env_rec* __restrict__ envs, int64_t n, const int32_t* __restrict__ W0Q,
                                                    const int32_t* __restrict__ b0Q, const float* __restrict__ inv_scale_p,
                                                    int32_t* __restrict__ Z, uint32_t* __restrict__ Prev, int fresh_all,
                                                    __nv_bfloat16* __restrict__ Hhi, __nv_bfloat16* __restrict__ Hlo) {
    __shared__ __align__(8) uint16_t s_rows[32][100];                 // per env: rows entering (+) / leaving (bit 15) the sum, padded with the zero row kIn
    const int lane = threadIdx.x & 31, sub = lane & 7, slot = threadIdx.x >> 3;
    const int64_t e0 = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 3;
    const bool live = e0 < n;                                         // tail lanes idle along (the shuffles need whole warps)
    const int64_t e = live ? e0 : 0;
    const uint4* W = reinterpret_cast<const uint4*>(W0Q) + sub;       // unsigned: wrap-around is defined
    // board words sub and 8 + sub (sub < 4); word 11 holds squares 88, 89 only
    uint32_t w[2], pv[2];
    w[0] = live ? envs[e].sq[sub] : 0u;
    w[1] = (live && sub < 4) ? envs[e].sq[8 + sub] : 0u;
    pv[0] = (live && !fresh_all) ? Prev[e * 12 + sub] : 0u;
    pv[1] = (live && !fresh_all && sub < 4) ? Prev[e * 12 + 8 + sub] : 0u;
    uint4 a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)      // issued before the board is looked at: one memory round trip less on the carried path
        a[i] = (live && !fresh_all) ? reinterpret_cast<const uint4*>(Z + e * kHid)[i * 8 + sub] : make_uint4(0u, 0u, 0u, 0u);
    w[0] = act_sanitize(w[0]); w[1] = act_sanitize(w[1]) & (sub == 3 ? 0xFFu : 0xFFFFFFFFu);
    const uint32_t x[2] = {act_nibble_flags(w[0] ^ pv[0]), act_nibble_flags(w[1] ^ pv[1])};
    int changed = __popc(x[0]) + __popc(x[1]);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) changed += __shfl_xor_sync(0xFFFFFFFFu, changed, o);
    const bool fresh = live && (fresh_all || changed > 4);            // uniform over the env's 8 lanes
    // rows that leave (old piece on a changed square) and rows that enter (new piece on a changed square; every piece on the gather path)
    uint32_t leave[2], enter[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        leave[r] = fresh ? 0u : x[r] & act_nibble_flags(pv[r]);
        enter[r] = (fresh ? 0x11111111u : x[r]) & act_nibble_flags(w[r]);
    }
    const int mine = __popc(leave[0]) + __popc(leave[1]) + __popc(enter[0]) + __popc(enter[1]);
    int pos = mine;                                                   // inclusive scan over the env's 8 lanes
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, pos, o, 8); if (sub >= o) pos += t; }
    const int total = __shfl_sync(0xFFFFFFFFu, pos, 7, 8);
    pos -= mine;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int sq0 = (r * 8 + sub) * 8;
        for (uint32_t v = leave[r]; v; v &= v - 1u) {
            const int sh = (__ffs((int)v) - 1) & 28;
            s_rows[slot][pos++] = (uint16_t)(0x8000 | ((sq0 + (sh >> 2)) * 14 + (int)((pv[r] >> sh) & 15u) - 1));
        }
        for (uint32_t v = enter[r]; v; v &= v - 1u) {
            const int sh = (__ffs((int)v) - 1) & 28;
            s_rows[slot][pos++] = (uint16_t)((sq0 + (sh >> 2)) * 14 + (int)((w[r] >> sh) & 15u) - 1);      // src/chessai.cpp:278-282
        }
    }
    if (sub < 4) s_rows[slot][total + sub] = (uint16_t)kIn;           // pad the last group of 4
    __syncwarp();
    if (fresh) {
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = reinterpret_cast<const uint4*>(b0Q)[i * 8 + sub];
        for (int k = 0; k < total; k += 4) {                          // the gather over all occupied squares: 4 rows in flight
            const uint2 l = *reinterpret_cast<const uint2*>(&s_rows[slot][k]);
            const uint32_t idx[4] = {l.x & 0xFFFFu, l.x >> 16, l.y & 0xFFFFu, l.y >> 16};
            uint4 v[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i) v[u][i] = W[(size_t)idx[u] * (kHid / 4) + i * 8];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i) { a[i].x += v[u][i].x; a[i].y += v[u][i].y; a[i].z += v[u][i].z; a[i].w += v[u][i].w; }
        }
    } else {
        for (int k = 0; k < total; k += 4) {                          // the carried sum: 2 rows for a quiet move, 3 for a capture
            const uint2 l = *reinterpret_cast<const uint2*>(&s_rows[slot][k]);
            const uint32_t idx[4] = {l.x & 0xFFFFu, l.x >> 16, l.y & 0xFFFFu, l.y >> 16};
            uint4 v[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i) v[u][i] = W[(size_t)(idx[u] & 0x7FFFu) * (kHid / 4) + i * 8];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t sg = 0u - (idx[u] >> 15);              // 0 or ~0: (x ^ sg) - sg negates
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    a[i].x += (v[u][i].x ^ sg) - sg; a[i].y += (v[u][i].y ^ sg) - sg; a[i].z += (v[u][i].z ^ sg) - sg; a[i].w += (v[u][i].w ^ sg) - sg;
                }
            }
        }
    }
    if (!live) return;
    const float is = *inv_scale_p;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        reinterpret_cast<uint4*>(Z + e * kHid)[i * 8 + sub] = a[i];
        act_emit_h(a[i], is, Hhi, Hlo, e, i * 8 + sub);
    }
    Prev[e * 12 + sub] = w[0];
    if (sub < 4) Prev[e * 12 + 8 + sub] = w[1];
}

// Both states of every transition in one launch, ONE WARP PER TRANSITION: the 128-byte replay record is read once
// (one coalesced line); lane l decodes squares l, l+32, l+64 of both boards, ballots compact the occupied squares into
// two row lists in shared memory (padded with the all-zero row kIn), and the two gather-sums -- h(s) with the online
// net, h(s') with the bootstrap net (online: ChessAI::train; target: DQN::train) -- run interleaved, four rows of
// each in flight, ~9 instructions per piece.  The warp also writes the compact batch record (board of s, action,
// reward, done; word-major) that the later kernels of the update read: the replay ring is touched here only.
// Block 0 clears db1 and the loss statistics (td_delta_kernel accumulates into them).
constexpr int kL0Warps = 4;
__global__ void __launch_bounds__(kL0Warps * 32) l0_pair_kernel(BatchRef batch, int64_t n, const float* __restrict__ W0T, const float* __restrict__ b0,
                                                               const float* __restrict__ W0T2, const float* __restrict__ b02,
                                                               float* __restrict__ Hf, __nv_bfloat16* __restrict__ H2bf,
                                                               uint32_t* __restrict__ cb, int64_t ld, float* __restrict__ zero_me, int n_zero,
                                                               int which /* bit 0: h(s) + compact batch, bit 1: h(s') */) {
    __shared__ __align__(8) uint16_t s_rows[kL0Warps][2][96];   // any board: up to 90 occupied squares (a legal one has <= 32)
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * kL0Warps + wib;
    // transition words: 0..11 board of s, 12..23 board of s', 24 = action | mover << 16 | done << 24, 25 = reward
    // (the replay ring is not written by the kernels of an update: it may be read before the PDL wait)
    const uint32_t word = (s < n && lane < 26) ? reinterpret_cast<const uint32_t*>(batch.at(s))[lane] : 0u;
#pragma unroll
    for (int r = 0; r < 3; ++r) { s_rows[wib][0][lane + 32 * r] = (uint16_t)kIn; s_rows[wib][1][lane + 32 * r] = (uint16_t)kIn; }
    __syncwarp();
    int cnt[2] = {0, 0};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int q = lane + 32 * r;                            // square; q < 90 in the last round only for lanes < 26
        const uint32_t wa = __shfl_sync(0xFFFFFFFFu, word, (q >> 3) % 12), wb = __shfl_sync(0xFFFFFFFFu, word, 12 + (q >> 3) % 12);
#pragma unroll
        for (int which = 0; which < 2; ++which) {
            const int code = ((which ? wb : wa) >> (4 * (q & 7))) & 15;
            const bool piece = q < XQ_SQUARES && code >= 1 && code <= 14;
            const unsigned m = __ballot_sync(0xFFFFFFFFu, piece);
            const int rank = cnt[which] + __popc(m & ((1u << lane) - 1u));
            if (piece) s_rows[wib][which][rank] = (uint16_t)(q * 14 + code - 1);      // getStateRepresentation index, src/chessai.cpp:278-282
            cnt[which] += __popc(m);
        }
    }
    __syncwarp();
    tc::pdl_wait();                 // the previous update's SGD step (W0T) and its readers of cb / the statistics slots are complete
    tc::pdl_launch_dependents();
    const bool do_a = which & 1, do_b = which & 2;              // the pipelined multi-update path runs the two halves on two streams
    if (do_a && blockIdx.x == 0) for (int i = threadIdx.x; i < n_zero; i += blockDim.x) zero_me[i] = 0.0f;
    if (s >= n) return;
    if (do_a) {
        if (lane < 12) cb[lane * ld + s] = word;               // word-major: the readers walk consecutive samples
        else if (lane >= 24 && lane < 26) cb[(lane - 12) * ld + s] = word;
    }
    const int steps = max(do_a ? cnt[0] : 0, do_b ? cnt[1] : 0);    // <= 90; the lists are padded to a multiple of 4 with the zero row
    float4 a = reinterpret_cast<const float4*>(b0)[lane], b = reinterpret_cast<const float4*>(b02)[lane];
    const float4* Wa = reinterpret_cast<const float4*>(W0T) + lane;
    const float4* Wb = reinterpret_cast<const float4*>(W0T2) + lane;
    for (int k = 0; k < steps; k += 4) {
        float4 ra[4], rb[4];
        const uint2 la = *reinterpret_cast<const uint2*>(&s_rows[wib][0][k]), lb = *reinterpret_cast<const uint2*>(&s_rows[wib][1][k]);     // 4 rows each
        const uint32_t ia[4] = {la.x & 0xFFFFu, la.x >> 16, la.y & 0xFFFFu, la.y >> 16}, ib[4] = {lb.x & 0xFFFFu, lb.x >> 16, lb.y & 0xFFFFu, lb.y >> 16};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            ra[u] = do_a ? Wa[(size_t)ia[u] * (kHid / 4)] : make_float4(0.f, 0.f, 0.f, 0.f);
            rb[u] = do_b ? Wb[(size_t)ib[u] * (kHid / 4)] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            a.x += ra[u].x; a.y += ra[u].y; a.z += ra[u].z; a.w += ra[u].w;
            b.x += rb[u].x; b.y += rb[u].y; b.z += rb[u].z; b.w += rb[u].w;
        }
    }
    if (do_a) reinterpret_cast<float4*>(Hf + s * kHid)[lane] = make_float4(tanhf(a.x), tanhf(a.y), tanhf(a.z), tanhf(a.w));
    if (do_b) store_h_bf16(H2bf, s, lane, make_float4(tanhf(b.x), tanhf(b.y), tanhf(b.z), tanhf(b.w)));
}

// ---------------------------------------------------------------------------------------------
// layer 1 on tcgen05: Z[M x 8100] = H[M x 128] * W1[8100 x 128]^T + b1, W1 tile stationary.
// CTA (n_tile, split): loads its [BN x 128] BF16 slice of W1 once, then streams the A tiles of its row range
// through a 3-stage TMA ring; one elected thread issues 9 UMMA (M128 x N224 x K16) per tile into one of two
// TMEM accumulator stages: 8 over the hidden units and ONE more whose A operand is a constant tile of ones and
// whose B operand holds b1 split into three BF16 terms (hi + lo + lo2 = 24 mantissa bits) -- the bias comes out
// of the tensor core, so the row-max epilogue is pure FMNMX straight out of TMEM (it was issue-bound on the
// bias adds: 1.5 k cycles per tile against 0.9 k of MMA).  8 epilogue warps (two per TMEM lane quarter) pull
// their 112 columns with four in-flight tcgen05.ld, release the accumulator stage, then reduce.
enum { EPI_ROWMAX = 0, EPI_STORE_TANH = 1 };

__device__ __forceinline__ uint32_t sw128_offset(int row, int col) {   // byte offset of bf16 (row, col) in a [rows x 64] SW128 K-major tile
    return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((((col >> 3) ^ row) & 7) << 4) + (col & 7) * 2);
}

template <int MODE>
__global__ void __launch_bounds__(kGemmThreads, 1) l1_gemm_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmW1,
                                                                 const float* __restrict__ b1, int M, int m_tiles, int n_splits,
                                                                 float* __restrict__ zpart, int64_t zstride, float* __restrict__ Q) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);   // SW128 tiles need 1024-B alignment
    uint8_t* sB = smem;                                    // [kKBlocks][BN][64] bf16
    uint8_t* sBb = sB + kBBytes;                           // [BN][64] bf16: k = 0,1,2 hold b1 as hi, lo, lo2; only k < 16 is ever read
    uint8_t* sAo = sBb + kBiasBBytes;                      // [BM][64] bf16: k = 0,1,2 are 1.0
    uint8_t* sA = sAo + kOnesBytes;                        // [kAStages][kKBlocks][BM][64] bf16
    uint64_t* bars = reinterpret_cast<uint64_t*>(sA + kAStages * kABytes);
    uint64_t* b_full = bars;              // 1
    uint64_t* a_full = bars + 1;          // kAStages
    uint64_t* a_empty = bars + 4;         // kAStages
    uint64_t* acc_full = bars + 7;        // 2
    uint64_t* acc_empty = bars + 9;       // 2
    uint64_t* c_full = bars + 11;         // bias / ones tiles written (warps 2, 3)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tile = blockIdx.x, split = blockIdx.y;
    const int n0 = n_tile * BN;
    // rows of this CTA: m-tiles split, split + n_splits, ... of [0, m_tiles)
    const int my_tiles = (m_tiles - split + n_splits - 1) / n_splits;
    if (threadIdx.x == 0) XQ_TL(0, 0);

    if (threadIdx.x == 0) {
        tc::mbar_init(b_full, 1);
        for (int i = 0; i < kAStages; ++i) { tc::mbar_init(a_full + i, 1); tc::mbar_init(a_empty + i, 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(acc_full + i, 1); tc::mbar_init(acc_empty + i, kEpiWarps); }
        tc::mbar_init(c_full, 2);
        tc::fence_barrier_init();
        // the operand loads do not depend on the rest of the set-up: start them before the CTA-wide barrier
        tc::prefetch_tmap(&tmH); tc::prefetch_tmap(&tmW1);
        tc::mbar_expect_tx(b_full, kBBytes);
        for (int kb = 0; kb < kKBlocks; ++kb) tc::tma_load_2d(sB + kb * (BN * BK * 2), &tmW1, kb * BK, n0, b_full);
        tc::pdl_wait();             // W1 / b1 were final before the producer of H started; H itself is the predecessor's output
        for (int i = 0; i < kAStages && i < my_tiles; ++i) {
            tc::mbar_expect_tx(a_full + i, kABytes);
            const int row0 = (split + i * n_splits) * BM;
            for (int kb = 0; kb < kKBlocks; ++kb) tc::tma_load_2d(sA + i * kABytes + kb * (BM * BK * 2), &tmH, kb * BK, row0, a_full + i);
        }
    }
    if (warp == 2) tc::tmem_alloc<kTmemCols>(tmem_slot);
    if (warp == 2 || warp == 3) {   // constant operand tiles of the bias step: b1 -> (hi, lo, lo2) rows of sBb, ones into sAo
        constexpr int kRowsPerThread = (BN + BM + 63) / 64;
        const int t = threadIdx.x - 64;
        float bv[kRowsPerThread];
#pragma unroll
        for (int u = 0; u < kRowsPerThread; ++u) {           // all loads in flight at once
            const int r = t + 64 * u;
            bv[u] = (r < BN && n0 + r < kOut) ? b1[n0 + r] : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < kRowsPerThread; ++u) {
            const int r = t + 64 * u;
            if (r >= BN + BM) break;
            const bool is_b = r < BN;
            const int row = is_b ? r : r - BN;
            uint8_t* tile = is_b ? sBb : sAo;
            __nv_bfloat16 v0, v1, v2;
            if (is_b) {
                const bool real = n0 + row < kOut;
                const float b = real ? bv[u] : -1e30f;                               // padded outputs never win the max
                v0 = __float2bfloat16_rn(b);
                const float r1 = real ? b - __bfloat162float(v0) : 0.0f;
                v1 = __float2bfloat16_rn(r1);
                v2 = __float2bfloat16_rn(r1 - __bfloat162float(v1));
            } else {
                v0 = v1 = v2 = __float2bfloat16_rn(1.0f);
            }
            const uint32_t w0 = (uint32_t)__bfloat16_as_ushort(v0) | ((uint32_t)__bfloat16_as_ushort(v1) << 16);
            const uint32_t w1 = (uint32_t)__bfloat16_as_ushort(v2);
            *reinterpret_cast<uint4*>(tile + sw128_offset(row, 0)) = make_uint4(w0, w1, 0u, 0u);     // k = 0..7
            *reinterpret_cast<uint4*>(tile + sw128_offset(row, 8)) = make_uint4(0u, 0u, 0u, 0u);     // k = 8..15
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    tc::pdl_wait();
    tc::pdl_launch_dependents();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) XQ_TL(0, 1);

    if (warp == 0) {
        if (lane == 0) {   // ===== TMA producer (stages 0..kAStages-1 were filled above) =====
            for (int i = kAStages; i < my_tiles; ++i) {
                const int st = i % kAStages;
                tc::mbar_wait(a_empty + st, ((i / kAStages) & 1) ^ 1);
                tc::mbar_expect_tx(a_full + st, kABytes);
                const int row0 = (split + i * n_splits) * BM;
                for (int kb = 0; kb < kKBlocks; ++kb) tc::tma_load_2d(sA + st * kABytes + kb * (BM * BK * 2), &tmH, kb * BK, row0, a_full + st);
            }
        }
        __syncwarp();      // the whole warp reaches the closing __syncthreads together (bar.sync is warp-aligned)
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer =====
            constexpr uint32_t idesc = tc::umma_idesc_bf16(BM, BN);
            const uint64_t d_ones = tc::umma_desc_sw128(tc::smem_u32(sAo)), d_bias = tc::umma_desc_sw128(tc::smem_u32(sBb));
            tc::mbar_wait(b_full, 0);
            XQ_TL(0, 2);
            for (int i = 0; i < my_tiles; ++i) {
                const int st = i % kAStages, acc = i & 1;
                tc::mbar_wait(acc_empty + acc, ((i >> 1) & 1) ^ 1);
                if (i < 8) XQ_TL(0, 4 + i);
                tc::mbar_wait(a_full + st, (i / kAStages) & 1);
                if (i < 8) XQ_TL(0, 12 + i);
                tc::tc_fence_after();
#pragma unroll
                for (int kb = 0; kb < kKBlocks; ++kb)
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        const uint64_t da = tc::umma_desc_sw128(tc::smem_u32(sA + st * kABytes + kb * (BM * BK * 2)) + k * 32);
                        const uint64_t db = tc::umma_desc_sw128(tc::smem_u32(sB + kb * (BN * BK * 2)) + k * 32);
                        tc::umma_bf16(tmem_base + acc * BN, da, db, idesc, (kb | k) != 0);
                    }
                tc::umma_commit(a_empty + st);      // A stage free once these MMAs have read it
                if (i == 0) { tc::mbar_wait(c_full, 0); tc::tc_fence_after(); }
                tc::umma_bf16(tmem_base + acc * BN, d_ones, d_bias, idesc, 1);      // + 1 * (b1_hi + b1_lo + b1_lo2)
                tc::umma_commit(acc_full + acc);    // accumulator ready for the epilogue
            }
        }
        __syncwarp();
    } else if (warp < 4) {   // ===== warps 2, 3: the bias-step operand tiles were written before the barrier =====
        tc::fence_proxy_async();            // generic-proxy stores -> visible to the tensor core
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(c_full);
    } else {   // ===== epilogue: warps w and w+4 drain TMEM lanes 32*(w&3).. +31, one half of the columns each =====
        const int quarter = warp & 3, half = (warp - 4) >> 2;
        constexpr int kHalfCols = BN / 2;                                   // 112 = 3 x 32 + 16 columns
        for (int i = 0; i < my_tiles; ++i) {
            const int acc = i & 1;
            const int row = (split + i * n_splits) * BM + quarter * 32 + lane;
            tc::mbar_wait(acc_full + acc, (i >> 1) & 1);
            if (warp == 4 && lane == 0 && i < 8) XQ_TL(0, 20 + i);
            tc::tc_fence_after();
            const uint32_t t0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + half * kHalfCols;
            if (MODE == EPI_ROWMAX) {
                uint32_t r[kHalfCols];
                tc::tmem_ld32_nowait(t0, r); tc::tmem_ld32_nowait(t0 + 32, r + 32); tc::tmem_ld32_nowait(t0 + 64, r + 64);
                tc::tmem_ld16_nowait(t0 + 96, r + 96);
                tc::tmem_wait_ld();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(acc_empty + acc);             // the values are in registers: the stage is free
                if (warp == 4 && lane == 0 && i < 8) XQ_TL(0, 28 + i);
                float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
                for (int j = 0; j < kHalfCols; j += 4) {
                    best[0] = fmaxf(best[0], __uint_as_float(r[j])); best[1] = fmaxf(best[1], __uint_as_float(r[j + 1]));
                    best[2] = fmaxf(best[2], __uint_as_float(r[j + 2])); best[3] = fmaxf(best[3], __uint_as_float(r[j + 3]));
                }
                if (row < M) zpart[(int64_t)row * kPartsPad + n_tile * 2 + half] = fmaxf(fmaxf(best[0], best[1]), fmaxf(best[2], best[3]));
            } else {
#pragma unroll 1
                for (int c = 0; c < kHalfCols / 16; ++c) {
                    uint32_t r[16];
                    tc::tmem_ld16_nowait(t0 + c * 16, r);
                    tc::tmem_wait_ld();
                    if (row < M) {
                        const int col0 = n0 + half * kHalfCols + c * 16;
                        float* out = Q + (size_t)row * kOut + col0;
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (col0 + j < kOut) out[j] = tanhf(__uint_as_float(r[j]));
                    }
                }
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(acc_empty + acc);
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) XQ_TL(0, 3);
    if (threadIdx.x == 128) XQ_TL(0, 36);
    if (threadIdx.x == 32) XQ_TL(0, 37);
    if (warp == 2) { tc::tc_fence_after(); tc::tmem_dealloc<kTmemCols>(tmem_base); }
}

// ---------------------------------------------------------------------------------------------
// Acting: Q(s)[0..95] = tanh(W1[0..95] h + b1) for every env -- DQN::selectAction indexes Q by action.to < 90 only
// (src/dqn.cpp:47), so 96 of the 8100 outputs are enough.  The reference's argmax is over FP64 Q-values; to keep
// near-ties where they are, the contraction runs in SPLIT precision on the tensor cores: h = h_hi + h_lo and
// W = W_hi + W_lo in BF16, z = h_hi W_hi + h_lo W_hi + h_hi W_lo (FP32 accumulate; the dropped lo*lo term is
// < 2^-17 relative) -- 24 UMMA (M128 x N96 x K16) per 128-env tile.  Persistent CTAs stride over the tiles;
// 8 epilogue warps add the FP32 bias, apply tanh (act_tanh: SFU exp2 + rcp, |error| ~1e-7) and write FP32 rows [env][96] through a small per-warp
// shared-memory transpose so that every store instruction covers contiguous 96-byte row pieces.
constexpr int QN = 96;
constexpr int kQStages = 2;
constexpr uint32_t kQBBytes = QN * kHid * 2;             // 24 KB per precision part of W1[0..95]
constexpr uint32_t kQABytes = BM * kHid * 2;             // 32 KB per precision part of an A tile
constexpr uint32_t kQXposeBytes = 8 * 32 * 24 * 4;       // 24 KB: per epilogue warp 32 rows x 24 columns FP32
constexpr size_t kQSmem = 1024 + 2 * kQBBytes + kQStages * 2 * kQABytes + kQXposeBytes + QN * 4 + 256;

__global__ void __launch_bounds__(kGemmThreads, 1) q90_gemm_kernel(const __grid_constant__ CUtensorMap tmHhi, const __grid_constant__ CUtensorMap tmHlo,
                                                                  const __grid_constant__ CUtensorMap tmWhi, const __grid_constant__ CUtensorMap tmWlo,
                                                                  const float* __restrict__ b1, int M, int m_tiles, float* __restrict__ q90) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* sB = smem;                                    // [hi | lo][2 k-blocks][96][64] bf16
    uint8_t* sA = sB + 2 * kQBBytes;                       // [stage][hi | lo][2 k-blocks][128][64] bf16
    float* sX = reinterpret_cast<float*>(sA + kQStages * 2 * kQABytes);     // [8 warps][32][24]
    float* sBias = sX + kQXposeBytes / 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + QN);
    uint64_t* b_full = bars;              // 1
    uint64_t* a_full = bars + 1;          // kQStages
    uint64_t* a_empty = bars + 3;         // kQStages
    uint64_t* acc_full = bars + 5;        // 2
    uint64_t* acc_empty = bars + 7;       // 2
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int my_tiles = (m_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;     // tiles blockIdx.x, + gridDim.x, ...
    auto load_a = [&](int i) {
        const int st = i % kQStages, row0 = ((int)blockIdx.x + i * (int)gridDim.x) * BM;
        tc::mbar_expect_tx(a_full + st, 2 * kQABytes);
        for (int kb = 0; kb < kKBlocks; ++kb) {
            tc::tma_load_2d(sA + st * 2 * kQABytes + kb * (BM * BK * 2), &tmHhi, kb * BK, row0, a_full + st);
            tc::tma_load_2d(sA + st * 2 * kQABytes + kQABytes + kb * (BM * BK * 2), &tmHlo, kb * BK, row0, a_full + st);
        }
    };
    if (threadIdx.x == 0) {
        tc::mbar_init(b_full, 1);
        for (int i = 0; i < kQStages; ++i) { tc::mbar_init(a_full + i, 1); tc::mbar_init(a_empty + i, 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(acc_full + i, 1); tc::mbar_init(acc_empty + i, kEpiWarps); }
        tc::fence_barrier_init();
        tc::prefetch_tmap(&tmHhi); tc::prefetch_tmap(&tmHlo); tc::prefetch_tmap(&tmWhi); tc::prefetch_tmap(&tmWlo);
        tc::mbar_expect_tx(b_full, 2 * kQBBytes);
        for (int kb = 0; kb < kKBlocks; ++kb) {
            tc::tma_load_2d(sB + kb * (QN * BK * 2), &tmWhi, kb * BK, 0, b_full);
            tc::tma_load_2d(sB + kQBBytes + kb * (QN * BK * 2), &tmWlo, kb * BK, 0, b_full);
        }
        tc::pdl_wait();             // h(s) is the predecessor's output
        for (int i = 0; i < kQStages && i < my_tiles; ++i) load_a(i);
    }
    if (warp == 2) tc::tmem_alloc<256>(tmem_slot);
    if (warp == 3) for (int i = lane; i < QN; i += 32) sBias[i] = b1[i];
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    tc::pdl_wait();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0)     // ===== TMA producer =====
            for (int i = kQStages; i < my_tiles; ++i) { tc::mbar_wait(a_empty + i % kQStages, ((i / kQStages) & 1) ^ 1); load_a(i); }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer: (h_hi, W_hi) + (h_lo, W_hi) + (h_hi, W_lo) =====
            constexpr uint32_t idesc = tc::umma_idesc_bf16(BM, QN);
            tc::mbar_wait(b_full, 0);
            for (int i = 0; i < my_tiles; ++i) {
                const int st = i % kQStages, acc = i & 1;
                tc::mbar_wait(acc_empty + acc, ((i >> 1) & 1) ^ 1);
                tc::mbar_wait(a_full + st, (i / kQStages) & 1);
                tc::tc_fence_after();
#pragma unroll
                for (int part = 0; part < 3; ++part) {
                    const uint8_t* a = sA + st * 2 * kQABytes + (part == 1 ? kQABytes : 0);
                    const uint8_t* b = sB + (part == 2 ? kQBBytes : 0);
#pragma unroll
                    for (int kb = 0; kb < kKBlocks; ++kb)
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k)
                            tc::umma_bf16(tmem_base + acc * QN, tc::umma_desc_sw128(tc::smem_u32(a + kb * (BM * BK * 2)) + k * 32),
                                          tc::umma_desc_sw128(tc::smem_u32(b + kb * (QN * BK * 2)) + k * 32), idesc, (part | kb | k) != 0);
                }
                tc::umma_commit(a_empty + st);
                tc::umma_commit(acc_full + acc);
            }
        }
        __syncwarp();
    } else if (warp >= 4) {   // ===== epilogue: warps w and w+4 share TMEM lanes 32*(w&3).. +31, 48 columns each =====
        const int quarter = warp & 3, half = (warp - 4) >> 2;
        float* xw = sX + (warp - 4) * (32 * 24);
        for (int i = 0; i < my_tiles; ++i) {
            const int acc = i & 1;
            const int row0 = ((int)blockIdx.x + i * (int)gridDim.x) * BM + quarter * 32;
            tc::mbar_wait(acc_full + acc, (i >> 1) & 1);
            tc::tc_fence_after();
            uint32_t r[48];
            const uint32_t t0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * QN + half * 48;
            tc::tmem_ld32_nowait(t0, r); tc::tmem_ld16_nowait(t0 + 32, r + 32);
            tc::tmem_wait_ld();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(acc_empty + acc);
#pragma unroll
            for (int c0 = 0; c0 < 48; c0 += 24) {             // two rounds of 24 columns through the warp's transpose buffer
#pragma unroll
                for (int j = 0; j < 24; j += 4) {
                    const float4 b4 = *reinterpret_cast<const float4*>(sBias + half * 48 + c0 + j);
                    *reinterpret_cast<float4*>(xw + lane * 24 + j) = make_float4(act_tanh(__uint_as_float(r[c0 + j]) + b4.x), act_tanh(__uint_as_float(r[c0 + j + 1]) + b4.y),
                                                                                 act_tanh(__uint_as_float(r[c0 + j + 2]) + b4.z), act_tanh(__uint_as_float(r[c0 + j + 3]) + b4.w));
                }
                __syncwarp();
                // lane = (row within a group of 5 rows, 16-byte chunk): 30 lanes move 5 rows x 96 bytes per step
                const int rr = lane / 6, ch = lane % 6;
                if (lane < 30)
                    for (int rb = 0; rb < 32; rb += 5) {
                        const int row = rb + rr;
                        if (row < 32 && row0 + row < M)
                            *reinterpret_cast<float4*>(q90 + (size_t)(row0 + row) * QN + half * 48 + c0 + ch * 4) = *reinterpret_cast<const float4*>(xw + row * 24 + ch * 4);
                    }
                __syncwarp();
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc::tc_fence_after(); tc::tmem_dealloc<256>(tmem_base); }
}

// ---------------------------------------------------------------------------------------------
// Transition record of the replay buffer / TD batch (include/xq.h: xq_transition, 128 B)
struct Transition {
    uint32_t s[12], s2[12];
    uint16_t action; uint8_t mover, done;
    int32_t reward;
    uint32_t pad[6];
};
static_assert(sizeof(Transition) == 128 && sizeof(xq_transition) == 128, "transition record must be 128 bytes");

// TD error, one warp per transition (src/chessai.cpp:121-131 + src/dqn.cu:288-308 specialised to a one-hot delta1).
// Outputs per sample: delta1, its row `to`, delta0 as FP32 and, transposed and split into BF16 hi + lo, as the
// K-major B operand of the dW0 contraction; delta1 itself goes into row 14 of the compact batch (db1 is summed by
// dw_gemm_kernel).  Global atomics: 3 per CTA for the loss statistics, spread over 16 slots (same-address L2
// atomics serialise at ~27 cycles each: 512 CTAs on one address were 14 k cycles, the whole kernel).
constexpr int kInfoSlots = 16;
__global__ void __launch_bounds__(256) td_delta_kernel(uint32_t* __restrict__ cb, int64_t n, const float* __restrict__ Hf,
                                                      const float* __restrict__ W1, const float* __restrict__ b1,
                                                      const float* __restrict__ zpart, int64_t zstride, int n_parts, float gamma, int mode,
                                                      __nv_bfloat16* __restrict__ d0hi, __nv_bfloat16* __restrict__ d0lo,
                                                      __nv_bfloat16* __restrict__ ghi, __nv_bfloat16* __restrict__ glo, int64_t ld,
                                                      float* __restrict__ info_slots) {
    __shared__ float s_info[8][3];
    __shared__ __align__(16) float s_d0[8][kHid];          // delta0 of the CTA's 8 consecutive samples, for the transposed stores
    __shared__ __align__(16) float s_g[8][kHid];           // delta1 * h (the dW1 contraction's B operand)
    const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    tc::pdl_wait();
    tc::pdl_launch_dependents();
    float loss = 0.0f, qv = 0.0f, tv = 0.0f;
    reinterpret_cast<float4*>(s_d0[wib])[lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    reinterpret_cast<float4*>(s_g[wib])[lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s < n) {
        const uint32_t meta = cb[12 * ld + s];
        const int to = XQ_ACTION_TO(meta & 0xFFFFu);           // the Q index of the taken action is action.to (:124,:127)
        const bool done = (meta >> 24) != 0;
        const float reward = (float)(int32_t)cb[13 * ld + s];
        const float4 h = reinterpret_cast<const float4*>(Hf + s * kHid)[lane];
        const float4 w = reinterpret_cast<const float4*>(W1 + (size_t)to * kHid)[lane];
        float z = h.x * w.x + h.y * w.y + h.z * w.z + h.w * w.w;
        float zmax = -INFINITY;
        if (!done) for (int i = lane; i < n_parts; i += 32) zmax = fmaxf(zmax, zpart[s * kPartsPad + i]);
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) { z += __shfl_xor_sync(0xFFFFFFFFu, z, k); zmax = fmaxf(zmax, __shfl_xor_sync(0xFFFFFFFFu, zmax, k)); }
        const float q = tanhf(z + b1[to]);
        const float target = done ? reward : reward + gamma * tanhf(zmax);
        const float d1 = (q - target) * (1.0f - q * q);        // outputLayerDeltaKernel, src/dqn.cu:288-295
        // hidden delta: as written W1flat[i*1260 + j] with i = to (only i < 128 is summed and delta1 is one-hot), or W1[to][j]
        const float* wrow = mode == XQ_DQN_AS_WRITTEN ? W1 + (size_t)to * kIn : W1 + (size_t)to * kHid;
        const float4 wd = reinterpret_cast<const float4*>(wrow)[lane];
        const float d0[4] = {wd.x * d1 * (1.0f - h.x * h.x), wd.y * d1 * (1.0f - h.y * h.y), wd.z * d1 * (1.0f - h.z * h.z),
                             wd.w * d1 * (1.0f - h.w * h.w)};
        reinterpret_cast<float4*>(s_d0[wib])[lane] = make_float4(d0[0], d0[1], d0[2], d0[3]);
        reinterpret_cast<float4*>(s_g[wib])[lane] = make_float4(d1 * h.x, d1 * h.y, d1 * h.z, d1 * h.w);
        if (lane == 0) cb[14 * ld + s] = __float_as_uint(d1);
        loss = 0.5f * (q - target) * (q - target); qv = q; tv = target;
    }
    if (lane == 0) { s_info[wib][0] = loss; s_info[wib][1] = qv; s_info[wib][2] = tv; }
    __syncthreads();
    {   // delta0^T[j][s0..s0+7] and (delta1 h)^T[j][s0..s0+7] as BF16 hi (threads 0..127) / lo (128..255): 16-byte stores
        const int j = threadIdx.x & (kHid - 1);
        const bool want_lo = threadIdx.x >= kHid;
        const int64_t s0 = (int64_t)blockIdx.x * 8;
#pragma unroll
        for (int which = 0; which < 2; ++which) {
            uint32_t packed[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const float v0 = which ? s_g[2 * p][j] : s_d0[2 * p][j], v1 = which ? s_g[2 * p + 1][j] : s_d0[2 * p + 1][j];
                const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
                __nv_bfloat162 o;
                if (want_lo) { o.x = __float2bfloat16_rn(v0 - __bfloat162float(h0)); o.y = __float2bfloat16_rn(v1 - __bfloat162float(h1)); }
                else { o.x = h0; o.y = h1; }
                packed[p] = *reinterpret_cast<uint32_t*>(&o);
            }
            __nv_bfloat16* dst = which ? (want_lo ? glo : ghi) : (want_lo ? d0lo : d0hi);
            if (s0 < ld) *reinterpret_cast<uint4*>(dst + (int64_t)j * ld + s0) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
        }
    }
    if (threadIdx.x < 3) {
        float a = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k) a += s_info[k][threadIdx.x];
        atomicAdd(info_slots + (blockIdx.x % kInfoSlots) * 4 + threadIdx.x, a);
    }
}

// ---- multi-GPU exchange buffer (one per rank, IPC-mapped by every peer; see grad_exchange_apply_kernel) ----
// [2 parities][kMaxRanks source ranks][kGradPad] FP32: slot (parity, r) of rank q's buffer is WRITTEN BY RANK r (its gradient contraction pushes
// the finished rows over NVLink) and read by rank q only | flags[kMaxRanks] u32: epoch of the last complete gradient of each source rank |
// status u32 | completion counter of the local contraction u32
constexpr int kMaxRanks = 16;
constexpr int kGradPad = (kGradSize + 3) / 4 * 4;
constexpr size_t kExchFlagsOff = sizeof(float) * 2 * (size_t)kMaxRanks * kGradPad;                 // 16-byte aligned
constexpr size_t kExchFlagsEnd = kExchFlagsOff + sizeof(uint32_t) * (kMaxRanks + 4);                   // flags, status word, completion counter, 2 spare
// The fused exchange: reduce-scatter + all-gather of the 16-row blocks with the flag carried INSIDE the data
// (the idea of the "LL" / "LL128" protocols of collective libraries): a 16-byte line holds three FP32 values x, y, z and the word
// epoch ^ x ^ y ^ z, written by one 16-byte vector store and read by one 16-byte vector load -- the receiver polls the data itself, no
// fence, no separate flag.  A line is accepted when x ^ y ^ z ^ w equals the epoch it waits for, so a line caught half-written (old and
// new words mixed) is simply polled again: no assumption about the atomicity of vector accesses beyond single words, 75 % of the bytes
// on the wire are payload (LL: 50 %).  tests/test_dist_gpu.py compares every exchanged bit with NCCL's sum over many updates.
//   inbox 1 (reduce-scatter): [2 parities][kMaxRanks source ranks][kLLBlocks][kLLLinesPerBlock] lines, written by the source rank, read by the block's owner
//   inbox 2 (all-gather):     [2 parities][kLLBlocks][kLLLinesPerBlock] lines, written by the block's owner, read by everybody else
// A block = the 16 x 128 FP32 rows one CTA of the contraction reduces: 8 values per reducing thread + 1 (db1) = 3 lines per thread.
constexpr int kLLBlocks = 88;                                                                        // 11 row tiles x 8 splits
constexpr int kLLLinesPerThread = 3;
constexpr int kLLLinesPerBlock = kLLLinesPerThread * 256;
constexpr size_t kLLBlockBytes = (size_t)kLLLinesPerBlock * 16;                                      // 12 KB for 8.4 KB of payload
constexpr size_t kExchLL1Off = (kExchFlagsEnd + 255) / 256 * 256;
constexpr size_t kExchLL1Bytes = 2 * (size_t)kMaxRanks * kLLBlocks * kLLBlockBytes;                  // 33 MB
constexpr size_t kExchLL2Off = kExchLL1Off + kExchLL1Bytes;
constexpr size_t kExchLL2Bytes = 2 * (size_t)kLLBlocks * kLLBlockBytes;                              // 2 MB
// host-level all-gather of small messages between the ranks' processes (the multi-GPU episode driver: finished-game events, round totals)
constexpr size_t kHgCap = 64 << 10;                                                                  // bytes per rank per call
constexpr size_t kExchHgOff = kExchLL2Off + kExchLL2Bytes;                                           // [2 parities][kMaxRanks][kHgCap] | flags[kMaxRanks] u32
constexpr size_t kExchHgFlagsOff = kExchHgOff + 2 * (size_t)kMaxRanks * kHgCap;
constexpr size_t kExchBytes = kExchHgFlagsOff + 256;
__host__ __device__ constexpr size_t exch_slot_floats(int parity, int src_rank) { return ((size_t)parity * kMaxRanks + (size_t)src_rank) * kGradPad; }
__host__ __device__ constexpr size_t exch_ll1_off(int parity, int src_rank, int blk) {
    return kExchLL1Off + (((size_t)parity * kMaxRanks + (size_t)src_rank) * kLLBlocks + (size_t)blk) * kLLBlockBytes;
}
__host__ __device__ constexpr size_t exch_ll2_off(int parity, int blk) { return kExchLL2Off + ((size_t)parity * kLLBlocks + (size_t)blk) * kLLBlockBytes; }
struct PeerPtrs { uint8_t* p[kMaxRanks]; };
__device__ __forceinline__ void ll_store(uint8_t* line, float a, float b, float c, uint32_t flag) {
    const uint32_t x = __float_as_uint(a), y = __float_as_uint(b), z = __float_as_uint(c);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(line), "r"(x), "r"(y), "r"(z), "r"(flag ^ x ^ y ^ z) : "memory");
}
__device__ __forceinline__ bool ll_valid(const uint4& l, uint32_t flag) { return (l.x ^ l.y ^ l.z ^ l.w) == flag; }
__device__ __forceinline__ uint4 ll_load(const uint8_t* line) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(line) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_peer_f4(const float* p) {
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
struct DwPush {               // world == 0: the gradient stays local (grad)
    PeerPtrs peers;
    int rank = 0, world = 0, parity = 0;
    uint32_t epoch = 0;
    bool fused = false;       // the contraction itself exchanges its row blocks (reduce-scatter + all-gather of the blocks, flag-in-data lines),
                              // sums them and applies the SGD step (no exchange kernel)
    long long timeout = 0;    // clock64 ticks a wait for a peer may last; then the update is NOT applied and *status is raised (sticky)
    uint32_t* status = nullptr;   // host-mapped word: epoch of the first exchange that timed out (0 = none)
};

// ---------------------------------------------------------------------------------------------
// dW0^T = X^T . delta0 on tcgen05: C[feature 0..1279][hidden 0..127] = sum_b onehot_b[feature] * delta0_b[hidden].
// (updateWeightsBiasesKernel for layer 0, src/dqn.cu:310-319, summed over the batch.)  Feature 1260 is a constant
// one, so row 1260 of C is db0; an 11th row tile contracts one-hot(action.to) with delta1*h = dW1 rows 0..89.
// A operand: the transposed one-hot tile [128 features x 64 samples] is BUILT in shared memory (128-byte-swizzled
// K-major layout) by 8 warps straight from the compact batch -- the 1260-wide one-hot matrix never exists in HBM.
// B operand: delta0^T as BF16 hi + lo (two MMAs, ~16 mantissa bits) by TMA.
// Grid (11 row tiles, 8 sample splits); the 8 CTAs of a row tile form a thread-block CLUSTER: each accumulates its
// sample range in TMEM and writes its FP32 partial to an L2-resident scratch (distributed shared memory moves only
// ~20 B/clk per SM, far too slow for 64 KB per CTA); after ONE cluster barrier (release / acquire at cluster scope)
// each CTA sums the 8 partials of its 16 rows (fixed order: deterministic) and applies the SGD step (or writes the
// compact gradient for the all-reduce).  No second kernel.
constexpr int kFeatPad = 1280, kBiasFeat = kIn;
constexpr int kDwMTiles = kFeatPad / BM + 1;             // 10 feature tiles of dW0^T (+ db0) and one tile for dW1 (rows = action.to)
constexpr int kDwSplits = 8;                             // sample splits = cluster size (portable maximum)
constexpr int kDwStages = 4;
constexpr uint32_t kDwABytes = BM * BK * 2;              // 16 KB
constexpr uint32_t kDwBBytes = 2 * kHid * BK * 2;        // 32 KB: rows 0..127 = hi, rows 128..255 = lo -> ONE N = 256 operand
constexpr int kDwThreads = 384;                          // warp 0 TMA, 1 MMA, 2 TMEM alloc, 4-11 one-hot builders (4-7 also epilogue)
constexpr int kCbRows = 15;                              // compact batch rows: 12 board words | action,mover,done | reward | delta1 (FP32 bits)
constexpr uint32_t kDwCBytes = kCbRows * BK * 4;         // 3.75 KB: the compact-batch words of the k-block's 64 samples, [word][sample]
constexpr uint32_t kDwCStride = 4096;
constexpr size_t kDwSmem = 1024 + kDwStages * (kDwABytes + kDwBBytes + kDwCStride) + 256;
static_assert(kDwStages * (kDwABytes + kDwBBytes) >= BM * kHid * 4, "the epilogue stages the FP32 tile in the operand buffers");
constexpr int kRowsPerCta = BM / kDwSplits;              // 16 rows of the tile are reduced and applied by each CTA of the cluster

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__global__ void __launch_bounds__(kDwThreads, 1) dw_gemm_kernel(const __grid_constant__ CUtensorMap tmD0Hi, const __grid_constant__ CUtensorMap tmD0Lo,
                                                               const __grid_constant__ CUtensorMap tmGHi, const __grid_constant__ CUtensorMap tmGLo,
                                                               const __grid_constant__ CUtensorMap tmCb, int n, float* __restrict__ part,
                                                               float* __restrict__ dbpart, float* __restrict__ info_slots, float* __restrict__ info,
                                                               float* __restrict__ grad,
                                                               float* __restrict__ W0T, float* __restrict__ b0, float* __restrict__ W1,
                                                               float* __restrict__ b1, __nv_bfloat16* __restrict__ W1bf,
                                                               __nv_bfloat16* __restrict__ W1lo, float lr, int apply, const DwPush push) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* sA = smem;                                        // [stage][128 features][64 samples]
    uint8_t* sB = smem + kDwStages * kDwABytes;                // [stage][hi rows | lo rows][64 samples]
    uint8_t* sC = sB + kDwStages * kDwBBytes;                  // [stage][14 words][64 samples] compact-batch words
    uint64_t* bars = reinterpret_cast<uint64_t*>(sC + kDwStages * kDwCStride);
    uint64_t* full = bars;                 // kDwStages: 1 TMA arrive(+tx) + 8 builder warps
    uint64_t* empty = bars + kDwStages;    // kDwStages: MMA commit
    uint64_t* cfull = bars + 2 * kDwStages;   // kDwStages: board words landed
    uint64_t* acc_full = bars + 3 * kDwStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kDwStages + 1);
    __shared__ float s_db1[2 * BM];        // the dW1 tile's CTAs: sum of delta1 per action.to over this CTA's samples, one row per builder warp of samples

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mt = blockIdx.x, ks = (int)cluster_rank();     // cluster = the kDwSplits CTAs (blockIdx.y) of one row tile
    const int total_kb = (n + BK - 1) / BK;
    const int my_kb = ks < total_kb ? (total_kb - ks + kDwSplits - 1) / kDwSplits : 0;     // k-blocks ks, ks + kDwSplits, ...
    const int f0 = mt * BM;
    const bool w1_tile = mt == kDwMTiles - 1;            // the dW1 tile: A = one-hot of action.to, B = (delta1 h)^T
    const CUtensorMap& tmHi = w1_tile ? tmGHi : tmD0Hi;
    const CUtensorMap& tmLo = w1_tile ? tmGLo : tmD0Lo;
    if (threadIdx.x == 0) XQ_TL(1, 0);

    auto issue_stage = [&](int i) {        // operands of k-block i -> stage i % kDwStages
        const int st = i % kDwStages, kb = ks + i * kDwSplits;
        tc::mbar_expect_tx(cfull + st, kDwCBytes);
        tc::tma_load_2d(sC + st * kDwCStride, &tmCb, kb * BK, 0, cfull + st);
        tc::mbar_expect_tx(full + st, kDwBBytes);
        tc::tma_load_2d(sB + st * kDwBBytes, &tmHi, kb * BK, 0, full + st);
        tc::tma_load_2d(sB + st * kDwBBytes + kDwBBytes / 2, &tmLo, kb * BK, 0, full + st);
    };
    if (threadIdx.x == 0) {
        for (int i = 0; i < kDwStages; ++i) { tc::mbar_init(full + i, 9); tc::mbar_init(empty + i, 1); tc::mbar_init(cfull + i, 1); }
        tc::mbar_init(acc_full, 1);
        tc::fence_barrier_init();
        tc::prefetch_tmap(&tmCb); tc::prefetch_tmap(&tmHi); tc::prefetch_tmap(&tmLo);
        tc::pdl_wait();             // delta0 / delta1 h / the compact batch are the predecessor's outputs
        for (int i = 0; i < kDwStages && i < my_kb; ++i) issue_stage(i);      // the first stages need no `empty` wait: start them before the CTA barrier
    }
    if (warp == 2) tc::tmem_alloc<256>(tmem_slot);

    // the reducing threads (0..255, two 16-byte chunks each of the 16 rows this CTA owns) fetch the old weights now:
    // they do not depend on anything this kernel computes
    static_assert(kRowsPerCta * (kHid / 4) == 2 * 256, "two chunks per reducing thread");
    int e[2];                                                   // element of the compact gradient, -1 = padding row
    const float* src[2];
    float4 wold[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int item = (int)threadIdx.x + 256 * u;
        const int row = ks * kRowsPerCta + ((item >> 5) % kRowsPerCta), chunk = item & 31;
        src[u] = part + ((size_t)(mt * kDwSplits) * BM + row) * kHid + chunk * 4;
        const int f = f0 + row;
        e[u] = -1;
        if (threadIdx.x < 256) {
            if (w1_tile) { if (row < kQRows) e[u] = kGradW1 + row * kHid + chunk * 4; }
            else if (f < kIn) e[u] = f * kHid + chunk * 4;
            else if (f == kBiasFeat) e[u] = kGradB0 + chunk * 4;
        }
        wold[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if ((apply || push.fused) && e[u] >= 0)
            wold[u] = *reinterpret_cast<const float4*>(e[u] < kGradB0 ? W0T + e[u] : (e[u] < kGradW1 ? b0 + (e[u] - kGradB0) : W1 + (e[u] - kGradW1)));
    }
    const int bt = threadIdx.x - 128;
    if (warp >= 4)                                             // the one-hot stages start from all-zero
        for (int u = bt; u < (int)(kDwStages * kDwABytes / 16); u += 256) reinterpret_cast<uint4*>(sA)[u] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x < 2 * BM) s_db1[threadIdx.x] = 0.0f;
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    tc::pdl_wait();
    tc::pdl_launch_dependents();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) XQ_TL(1, 1);

    if (warp == 0) {
        if (lane == 0) {   // ===== TMA producer: board words + delta0^T hi / lo tiles =====
            for (int i = kDwStages; i < my_kb; ++i) {
                tc::mbar_wait(empty + i % kDwStages, ((i / kDwStages) & 1) ^ 1);
                issue_stage(i);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer: M128 x N256 (hi | lo) x K16, the one-hot operand is read once per step =====
            constexpr uint32_t idesc = tc::umma_idesc_bf16(BM, 2 * kHid);
            for (int i = 0; i < my_kb; ++i) {
                const int st = i % kDwStages;
                tc::mbar_wait(full + st, (i / kDwStages) & 1);
                if (i < 8) XQ_TL(1, 4 + i);
                tc::tc_fence_after();
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) {
                    const uint64_t da = tc::umma_desc_sw128(tc::smem_u32(sA + st * kDwABytes) + k * 32);
                    const uint64_t db = tc::umma_desc_sw128(tc::smem_u32(sB + st * kDwBBytes) + k * 32);
                    tc::umma_bf16(tmem_base, da, db, idesc, (i | k) != 0);
                }
                tc::umma_commit(empty + st);
            }
            if (my_kb > 0) tc::umma_commit(acc_full);
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===== one-hot^T builders: thread = (sample of the k-block, group of <= 3 squares of this feature tile).  A thread owns
        // column `sample` of its squares' feature rows in every stage: it clears the (<= 3) ones it set kDwStages k-blocks ago and
        // sets the new ones -- no tile-wide zeroing, no barrier between the warps.  The stage is free for rewriting once its board
        // words have landed: the producer issued them only after the MMAs of the stage's previous use had completed.
        const int sample = bt & 63, grp = bt >> 6;
        const int q0 = f0 / 14;
        uint32_t prev[kDwStages][3];
#pragma unroll
        for (int a = 0; a < kDwStages; ++a) prev[a][0] = prev[a][1] = prev[a][2] = 0xFFFFFFFFu;
        for (int i0 = 0; i0 < my_kb; i0 += kDwStages) {
#pragma unroll
            for (int st = 0; st < kDwStages; ++st) {
                const int i = i0 + st;
                if (i >= my_kb) break;
                const int b = (ks + i * kDwSplits) * BK + sample;
                const uint32_t* words = reinterpret_cast<const uint32_t*>(sC + st * kDwCStride) + sample;     // word w at words[w * 64]
                tc::mbar_wait(cfull + st, (i / kDwStages) & 1);
                uint32_t off[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
                if (b < n && w1_tile) {
                    if (grp == 0) off[0] = sw128_offset((int)XQ_ACTION_TO(words[12 * BK] & 0xFFFFu), sample);      // row = action.to (< 128)
                } else if (b < n) {
#pragma unroll
                    for (int u = 0; u < 3; ++u) {
                        const int q = q0 + grp + 4 * u;
                        if (q < XQ_SQUARES) {
                            const int code = (words[(q >> 3) * BK] >> (4 * (q & 7))) & 15;
                            const int f = q * 14 + code - 1 - f0;
                            if (code >= 1 && code <= 14 && f >= 0 && f < BM) off[u] = sw128_offset(f, sample);
                        }
                    }
                    if (mt == kDwMTiles - 2 && grp == 3) off[2] = sw128_offset(kBiasFeat - f0, sample);      // constant-one feature -> db0
                }
                if (w1_tile && grp == 0) {      // db1[to] += delta1 (src/dqn.cu:310-319): lanes with equal `to` are summed in lane order, the lowest
                    const int to = (int)XQ_ACTION_TO(words[12 * BK] & 0xFFFFu);          // lane of a group adds to this WARP's row -> deterministic, no atomics
                    const float d1 = b < n ? __uint_as_float(words[14 * BK]) : 0.0f;
                    const unsigned peers = __match_any_sync(0xFFFFFFFFu, to);
                    float sum = 0.0f;
#pragma unroll
                    for (int k = 0; k < 32; ++k) { const float v = __shfl_sync(0xFFFFFFFFu, d1, k); if (peers >> k & 1u) sum += v; }
                    if (lane == __ffs((int)peers) - 1) s_db1[(warp - 4) * BM + to] += sum;
                    __syncwarp();
                }
                if (bt == 0 && i < 8) XQ_TL(1, 12 + i);
                uint8_t* tile = sA + st * kDwABytes;
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    if (prev[st][u] != 0xFFFFFFFFu) *reinterpret_cast<uint16_t*>(tile + prev[st][u]) = 0;
                    if (off[u] != 0xFFFFFFFFu) *reinterpret_cast<uint16_t*>(tile + off[u]) = 0x3F80;        // BF16 1.0
                    prev[st][u] = off[u];
                }
                tc::fence_proxy_async();                                             // generic-proxy stores -> visible to the tensor core
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(full + st);
                if (bt == 0 && i < 8) XQ_TL(1, 20 + i);
            }
        }
        if (warp < 8) {   // ===== epilogue: hi + lo halves out of TMEM -> this warp's 32 rows staged in shared memory (16-byte chunks
                          // XOR-swizzled by row); the whole CTA then writes coalesced 512-byte rows of the FP32 partial =====
            const int quarter = warp & 3, row = quarter * 32 + lane;
            if (my_kb > 0) { tc::mbar_wait(acc_full, 0); tc::tc_fence_after(); }
            if (bt == 0) XQ_TL(1, 2);
#pragma unroll
            for (int c0 = 0; c0 < kHid; c0 += 32) {
                uint32_t rh[32], rlo[32];
                if (my_kb > 0) {
                    tc::tmem_ld32_nowait(tmem_base + ((uint32_t)(quarter * 32) << 16) + c0, rh);
                    tc::tmem_ld32_nowait(tmem_base + ((uint32_t)(quarter * 32) << 16) + kHid + c0, rlo);
                    tc::tmem_wait_ld();
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) rh[j] = rlo[j] = 0u;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<float4*>(smem + row * (kHid * 4) + (((c0 / 4 + j) ^ row) & 31) * 16) =
                        make_float4(__uint_as_float(rh[4 * j]) + __uint_as_float(rlo[4 * j]), __uint_as_float(rh[4 * j + 1]) + __uint_as_float(rlo[4 * j + 1]),
                                    __uint_as_float(rh[4 * j + 2]) + __uint_as_float(rlo[4 * j + 2]), __uint_as_float(rh[4 * j + 3]) + __uint_as_float(rlo[4 * j + 3]));
            }
            if (bt == 0) XQ_TL(1, 38);
        }
    }
    __syncthreads();               // the FP32 tile is staged
    {   // all 12 warps push it to L2 (a warp keeps only a few stores in flight: the more warps, the shorter this phase)
        float* out = part + (size_t)(mt * kDwSplits + ks) * BM * kHid;
#pragma unroll 4
        for (int rr = warp; rr < BM; rr += kDwThreads / 32)     // lane = 16-byte chunk of row rr
            reinterpret_cast<float4*>(out + rr * kHid)[lane] = *reinterpret_cast<const float4*>(smem + rr * (kHid * 4) + ((lane ^ rr) & 31) * 16);
        if (w1_tile && threadIdx.x < BM) dbpart[ks * BM + threadIdx.x] = s_db1[threadIdx.x] + s_db1[BM + threadIdx.x];
    }
    if (threadIdx.x == 128) XQ_TL(1, 40);
    // ===== cluster reduction + SGD: this CTA owns rows [16 ks, 16 ks + 16) of the tile =====
    tc::tc_fence_before();
    __syncwarp();
    cluster_sync_all();            // all 8 partials of the row tile are visible (release / acquire at cluster scope); also a CTA-wide barrier
    if (threadIdx.x == 0) XQ_TL(1, 3);
    if (warp == 2) { tc::tc_fence_after(); tc::tmem_dealloc<256>(tmem_base); }
    float4 acc[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (e[u] >= 0) {
#pragma unroll
            for (int p = 0; p < kDwSplits; ++p) {               // fixed order: the sum is deterministic
                const float4 v = __ldcg(reinterpret_cast<const float4*>(src[u] + (size_t)p * BM * kHid));
                acc[u].x += v.x; acc[u].y += v.y; acc[u].z += v.z; acc[u].w += v.w;
            }
        }
    }
    bool exch_ok = true;           // false: a peer never arrived -- this thread's part of the update is skipped and *push.status is raised
    float db1 = 0.0f;
    const bool owns_db1 = push.fused && w1_tile && ks == 0 && threadIdx.x < kQRows;
    if (owns_db1) {
#pragma unroll
        for (int p = 0; p < kDwSplits; ++p) db1 += __ldcg(dbpart + p * BM + threadIdx.x);      // the 8 per-CTA sums in fixed order
    }
    if (push.fused) {
        // ===== multi-GPU, ONE kernel: contraction -> reduce-scatter -> all-gather -> SGD, row block by row block, over peer memory =====
        // Block blk (the 16 rows this CTA reduced) is OWNED by rank blk % world.  The same CTA (mt, ks) of every rank handles the same block and
        // the same thread the same elements, so the exchange is thread to thread:
        //   non-owner: 3 flag-in-data lines per thread into the owner's inbox 1 (posted 16-byte stores over NVLink 5 / NVSwitch, a warp
        //              covers 512 contiguous bytes per store instruction), then polls its own inbox 2 for the owner's sum;
        //   owner:     polls inbox 1 for the `world - 1` other copies (the loads of up to eight source ranks in flight together), adds the
        //              copies IN RANK ORDER (its own from registers) -- every rank applies the very same bits -- and stores the sum into
        //              inbox 2 of every other rank.
        // No fence, no flag array, no barrier: a line is valid when its check word matches the epoch.  Traffic per rank and update:
        // 2 x (world - 1) / world x 0.69 MB x 4/3 (line format) instead of (world - 1) x 0.69 MB -- 1.6 MB instead of 4.8 MB at 8 GPUs, and the
        // critical path is two one-way NVLink hops instead of [stores -> system-scope fence -> flag -> acquire].
        // Slot reuse: a rank writes epoch e + 2 into the slots of epoch e only after it completed update e + 1, for which it needed every
        // rank's lines of epoch e + 1, which they sent after completing update e, i.e. after their last read of the epoch-e slots.
        const int blk = mt * kDwSplits + ks, owner = blk % push.world, tid = threadIdx.x;
        const uint32_t flag = push.epoch;
        // line k of a thread = values 3k .. 3k + 2 of (acc[0], acc[1], db1); it travels if any of them is a real gradient entry
        const bool line[kLLLinesPerThread] = {e[0] >= 0, e[0] >= 0 || e[1] >= 0, e[1] >= 0 || owns_db1};
        const float mine[9] = {acc[0].x, acc[0].y, acc[0].z, acc[0].w, acc[1].x, acc[1].y, acc[1].z, acc[1].w, db1};
        const long long t0 = clock64();
        float g[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (threadIdx.x == 0) { XQ_TL(1, 41); XQ_TLV(1, 45, owner == push.rank ? 1 : 0); }
        if (owner == push.rank) {
            const uint8_t* inbox = push.peers.p[push.rank] + (size_t)tid * 16;
            constexpr int kG = 8;                                   // source ranks polled together: all 24 line loads of a thread in flight at once
            for (int r0 = 0; r0 < push.world; r0 += kG) {
                uint4 l[kG][kLLLinesPerThread];
                bool ready;
                do {
                    ready = true;
#pragma unroll
                    for (int j = 0; j < kG; ++j) {
                        const int r = r0 + j;
                        if (r >= push.world || r == push.rank) continue;
                        const uint8_t* src = inbox + exch_ll1_off(push.parity, r, blk);
#pragma unroll
                        for (int k = 0; k < kLLLinesPerThread; ++k)
                            if (line[k]) l[j][k] = ll_load(src + (size_t)k * 256 * 16);
                    }
#pragma unroll
                    for (int j = 0; j < kG; ++j) {
                        const int r = r0 + j;
                        if (r >= push.world || r == push.rank) continue;
#pragma unroll
                        for (int k = 0; k < kLLLinesPerThread; ++k)
                            if (line[k] && !ll_valid(l[j][k], flag)) ready = false;
                    }
                } while (!ready && clock64() - t0 < push.timeout);
                if (!ready) exch_ok = false;
                if (threadIdx.x == 0) XQ_TL(1, 48 + (r0 >> 3));     // sources r0 .. r0 + 7 are in
#pragma unroll
                for (int j = 0; j < kG; ++j) {                      // rank order
                    const int r = r0 + j;
                    if (r >= push.world) break;
#pragma unroll
                    for (int k = 0; k < kLLLinesPerThread; ++k) {
                        if (!line[k]) continue;
                        g[3 * k] += r == push.rank ? mine[3 * k] : __uint_as_float(l[j][k].x);
                        g[3 * k + 1] += r == push.rank ? mine[3 * k + 1] : __uint_as_float(l[j][k].y);
                        g[3 * k + 2] += r == push.rank ? mine[3 * k + 2] : __uint_as_float(l[j][k].z);
                    }
                }
            }
            if (exch_ok)
                for (int r = 0; r < push.world; ++r) {
                    if (r == push.rank) continue;
                    uint8_t* dst = push.peers.p[r] + exch_ll2_off(push.parity, blk) + (size_t)tid * 16;
#pragma unroll
                    for (int k = 0; k < kLLLinesPerThread; ++k)
                        if (line[k]) ll_store(dst + (size_t)k * 256 * 16, g[3 * k], g[3 * k + 1], g[3 * k + 2], flag);
                }
            if (threadIdx.x == 0) XQ_TL(1, 43);                     // owner: the sum is on its way to the peers
        } else {
            uint8_t* dst = push.peers.p[owner] + exch_ll1_off(push.parity, push.rank, blk) + (size_t)tid * 16;
#pragma unroll
            for (int k = 0; k < kLLLinesPerThread; ++k)
                if (line[k]) ll_store(dst + (size_t)k * 256 * 16, mine[3 * k], mine[3 * k + 1], mine[3 * k + 2], flag);
            if (threadIdx.x == 0) XQ_TL(1, 42);                     // non-owner: my copy is on its way to the owner
            const uint8_t* src = push.peers.p[push.rank] + exch_ll2_off(push.parity, blk) + (size_t)tid * 16;
            uint4 l[kLLLinesPerThread];
            bool ready;
            do {
                ready = true;
#pragma unroll
                for (int k = 0; k < kLLLinesPerThread; ++k)
                    if (line[k]) l[k] = ll_load(src + (size_t)k * 256 * 16);
#pragma unroll
                for (int k = 0; k < kLLLinesPerThread; ++k)
                    if (line[k] && !ll_valid(l[k], flag)) ready = false;
            } while (!ready && clock64() - t0 < push.timeout);
            if (!ready) exch_ok = false;
            if (threadIdx.x == 0) XQ_TL(1, 44);                     // non-owner: the owner's sum is in
#pragma unroll
            for (int k = 0; k < kLLLinesPerThread; ++k)
                if (line[k]) { g[3 * k] = __uint_as_float(l[k].x); g[3 * k + 1] = __uint_as_float(l[k].y); g[3 * k + 2] = __uint_as_float(l[k].z); }
        }
        if (!exch_ok) { *push.status = flag; __threadfence_system(); }
        acc[0] = make_float4(g[0], g[1], g[2], g[3]); acc[1] = make_float4(g[4], g[5], g[6], g[7]);
        if (owns_db1 && exch_ok) b1[threadIdx.x] -= lr * g[8];
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        if (e[u] < 0) continue;
        if (!apply && !push.fused) {
            if (push.world > 0) {      // multi-GPU: the finished rows go straight into slot (parity, my rank) of EVERY rank's exchange buffer (posted NVLink stores)
                const size_t off = sizeof(float) * (exch_slot_floats(push.parity, push.rank) + (size_t)e[u]);
                for (int r = 0; r < push.world; ++r) *reinterpret_cast<float4*>(push.peers.p[r] + off) = acc[u];
            } else {
                *reinterpret_cast<float4*>(grad + e[u]) = acc[u];
            }
            continue;
        }
        if (!exch_ok) continue;
        float* dst = e[u] < kGradB0 ? W0T + e[u] : (e[u] < kGradW1 ? b0 + (e[u] - kGradB0) : W1 + (e[u] - kGradW1));
        float4 w = wold[u];
        w.x -= lr * acc[u].x; w.y -= lr * acc[u].y; w.z -= lr * acc[u].z; w.w -= lr * acc[u].w;
        *reinterpret_cast<float4*>(dst) = w;
        if (e[u] >= kGradW1) {                                  // refresh the BF16 operand copy of the touched W1 row
            __nv_bfloat162 p0 = __floats2bfloat162_rn(w.x, w.y), p1 = __floats2bfloat162_rn(w.z, w.w);
            uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
            *reinterpret_cast<uint2*>(W1bf + (e[u] - kGradW1)) = pk;
            __nv_bfloat162 q0 = __floats2bfloat162_rn(w.x - __bfloat162float(p0.x), w.y - __bfloat162float(p0.y));
            __nv_bfloat162 q1 = __floats2bfloat162_rn(w.z - __bfloat162float(p1.x), w.w - __bfloat162float(p1.y));
            pk.x = *reinterpret_cast<uint32_t*>(&q0); pk.y = *reinterpret_cast<uint32_t*>(&q1);
            *reinterpret_cast<uint2*>(W1lo + (e[u] - kGradW1)) = pk;       // rows 0..89 < 96: the acting path's residual operand
        }
    }
    if (w1_tile && ks == 0) {
        if (threadIdx.x < kQRows && !push.fused) {              // db1: the 8 per-CTA sums in fixed order
            float g = 0.0f;
#pragma unroll
            for (int p = 0; p < kDwSplits; ++p) g += __ldcg(dbpart + p * BM + threadIdx.x);
            if (!apply && push.world > 0) {
                const size_t off = sizeof(float) * (exch_slot_floats(push.parity, push.rank) + (size_t)(kGradB1 + threadIdx.x));
                for (int r = 0; r < push.world; ++r) *reinterpret_cast<float*>(push.peers.p[r] + off) = g;
            } else {
                grad[kGradB1 + threadIdx.x] = g;
            }
            if (apply) b1[threadIdx.x] -= lr * g;
        } else if (threadIdx.x >= 128 && threadIdx.x < 131) {   // loss statistics: fold the slots td_delta_kernel accumulated into
            float a = 0.0f;
            for (int p = 0; p < kInfoSlots; ++p) a += __ldcg(info_slots + p * 4 + (threadIdx.x - 128));
            info[threadIdx.x - 128] = a;
        }
    }
    if (threadIdx.x == 32) XQ_TL(1, 37);
    if (!apply && push.world > 0 && !push.fused) {
        // "gradient `epoch` of this rank has landed everywhere": every CTA fences its stores at system scope and counts itself; the last one
        // raises this rank's flag in every rank's buffer (release, system scope) -- grad_exchange_apply_kernel spins on those flags locally
        __shared__ int s_last;
        __threadfence_system();
        __syncthreads();
        unsigned* counter = reinterpret_cast<unsigned*>(push.peers.p[push.rank] + kExchFlagsOff) + kMaxRanks + 1;
        if (threadIdx.x == 0) {
            const unsigned prev = atomicAdd(counter, 1u);
            s_last = prev == gridDim.x * gridDim.y - 1u;
        }
        __syncthreads();
        if (s_last) {
            __threadfence_system();
            if ((int)threadIdx.x < push.world) {
                uint32_t* f = reinterpret_cast<uint32_t*>(push.peers.p[threadIdx.x] + kExchFlagsOff) + push.rank;
                asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(push.epoch) : "memory");
            }
            if (threadIdx.x == 0) *counter = 0u;
        }
    }
}

// SGD: W -= lr * grad on the compact gradient (src/dqn.cu:310-319), refresh the BF16 operand rows, clear the gradient
__global__ void __launch_bounds__(256) apply_kernel(float* __restrict__ W0T, float* __restrict__ b0, float* __restrict__ W1, float* __restrict__ b1,
                                                   __nv_bfloat16* __restrict__ W1bf, __nv_bfloat16* __restrict__ W1lo, float* __restrict__ grad, float lr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kGradSize) return;
    const float g = grad[i];
    grad[i] = 0.0f;
    if (g == 0.0f) return;
    if (i < kGradB0) W0T[i] -= lr * g;
    else if (i < kGradW1) b0[i - kGradB0] -= lr * g;
    else if (i < kGradB1) {
        const int e = i - kGradW1; const float v = W1[e] - lr * g; W1[e] = v;
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        W1bf[e] = hi; W1lo[e] = __float2bfloat16_rn(v - __bfloat162float(hi));
    }
    else b1[i - kGradB1] -= lr * g;
}

// ---------------------------------------------------------------------------------------------
// Multi-GPU TD update, the ONE exchange step of the path, fused on both sides: the gradient contraction (dw_gemm_kernel, apply = 0) PUSHES every
// finished 16-row block of its compact gradient into slot (parity, its rank) of EVERY rank's exchange buffer -- posted stores over NVLink 5 /
// NVSwitch while the other row tiles are still being reduced -- and its last CTA raises "gradient `epoch` of rank r has landed" in every
// rank's flag array (fence + release at system scope).  This kernel (same launch on every rank, programmatic dependent launch)
//   1. waits until all `world` flags in its OWN memory carry `epoch` (acquire, system scope; the spin and everything after it is local),
//   2. sums the `world` slots in rank order -- the same order on every rank, so the replicas stay bit-identical -- and applies W -= lr * g.
// Two parities alternate: a rank can only push epoch e+1 after its own kernel of epoch e has finished, i.e. after every rank's flag of epoch e
// was in, i.e. after every rank's kernel of epoch e-1 had finished reading slot parity (e-1)&1 == (e+1)&1.  No NCCL call, no remote loads,
// no separate apply.

__global__ void __launch_bounds__(256) grad_exchange_apply_kernel(PeerPtrs peers, int rank, int world, int parity, uint32_t epoch,
                                                                 float* __restrict__ W0T, float* __restrict__ b0, float* __restrict__ W1,
                                                                 float* __restrict__ b1, __nv_bfloat16* __restrict__ W1bf,
                                                                 __nv_bfloat16* __restrict__ W1lo, float lr, long long timeout, uint32_t* __restrict__ status) {
    uint32_t* my_flags = reinterpret_cast<uint32_t*>(peers.p[rank] + kExchFlagsOff);
    __shared__ int s_timed_out;
    if (threadIdx.x == 0) s_timed_out = 0;
    tc::pdl_wait();                                            // launched under the tail of the gradient contraction (programmatic dependent launch)
    tc::pdl_launch_dependents();                               // the next update's layer-0 kernel waits for this grid's completion before it reads W0T
    __syncthreads();
    if ((int)threadIdx.x < world) {                            // 2. all gradients of this epoch are complete
        const long long t0 = clock64();
        uint32_t v;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(my_flags + threadIdx.x) : "memory");
            if ((int32_t)(v - epoch) >= 0) break;
            if (clock64() - t0 > timeout) { s_timed_out = 1; *status = epoch; __threadfence_system(); break; }   // a peer never arrived: sticky, nothing is applied
        } while (true);
    }
    __syncthreads();
    if (s_timed_out) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;       // 3. float4 index over the compact gradient
    if (i >= kGradPad / 4) return;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = 0; r < world; ++r) {                          // slot (parity, r) of MY buffer: pushed by rank r's contraction
        const float4 v = ld_peer_f4(reinterpret_cast<const float*>(peers.p[rank]) + exch_slot_floats(parity, r) + 4 * (size_t)i);
        g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
    }
    const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {                              // the segment boundaries of the compact layout are not all multiples of 4
        const int e = 4 * i + k;
        if (e >= kGradSize) break;
        if (e < kGradB0) W0T[e] -= lr * gv[k];
        else if (e < kGradW1) b0[e - kGradB0] -= lr * gv[k];
        else if (e < kGradB1) {
            const int j = e - kGradW1;
            const float v = W1[j] - lr * gv[k];
            W1[j] = v;
            const __nv_bfloat16 hi = __float2bfloat16_rn(v);
            W1bf[j] = hi; W1lo[j] = __float2bfloat16_rn(v - __bfloat162float(hi));
        } else b1[e - kGradB1] -= lr * gv[k];
    }
}

// Host-level all-gather of one small message per rank (the multi-GPU episode driver's round totals and finished-game events): every rank
// stores its message into inbox (parity, its rank) of every rank, fences at system scope, releases its sequence number into every rank's
// flag array and waits for all `world` flags in its own memory.  One CTA; same double-buffering argument as the gradient slots.
__global__ void __launch_bounds__(256) host_gather_kernel(PeerPtrs peers, int rank, int world, int parity, uint32_t seq, const uint4* __restrict__ src,
                                                         int n16, long long timeout, uint32_t* __restrict__ status) {
    const size_t off = kExchHgOff + ((size_t)parity * kMaxRanks + (size_t)rank) * kHgCap;
    for (int r = 0; r < world; ++r) {
        uint4* dst = reinterpret_cast<uint4*>(peers.p[r] + off);
        for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = src[i];
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < world) {
        uint32_t* f = reinterpret_cast<uint32_t*>(peers.p[threadIdx.x] + kExchHgFlagsOff) + rank;
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(seq) : "memory");
        const uint32_t* mine = reinterpret_cast<const uint32_t*>(peers.p[rank] + kExchHgFlagsOff) + threadIdx.x;
        const long long t0 = clock64();
        uint32_t v;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
            if ((int32_t)(v - seq) >= 0) break;
            if (clock64() - t0 > timeout) { *status = 0x80000000u | seq; __threadfence_system(); break; }
        } while (true);
    }
}

// ---- FP64 (reference layout) <-> fast-path layouts ----------------------------------------------
__global__ void f64_to_fast_kernel(const double* __restrict__ w, const double* __restrict__ b, float* __restrict__ W0T, float* __restrict__ b0,
                                   float* __restrict__ W1, float* __restrict__ b1, __nv_bfloat16* __restrict__ W1bf, __nv_bfloat16* __restrict__ W1lo) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (int64_t)kIn * kHid) { const int o = (int)(i / kIn), in = (int)(i % kIn); W0T[(size_t)in * kHid + o] = (float)w[i]; }   // W0[o][in] -> W0T[in][o]
    if (i < (int64_t)kOut * kHid) {
        const float v = (float)w[(size_t)kIn * kHid + i]; W1[i] = v;
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        W1bf[i] = hi;
        if (W1lo && i < (int64_t)QN * kHid) W1lo[i] = __float2bfloat16_rn(v - __bfloat162float(hi));
    }
    if (i < kHid) b0[i] = (float)b[i];
    if (i < kOut) b1[i] = (float)b[kHid + i];
}
__global__ void fast_to_f64_kernel(double* __restrict__ w, double* __restrict__ b, const float* __restrict__ W0T, const float* __restrict__ b0,
                                   const float* __restrict__ W1, const float* __restrict__ b1) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (int64_t)kIn * kHid) { const int o = (int)(i / kIn), in = (int)(i % kIn); w[i] = (double)W0T[(size_t)in * kHid + o]; }
    if (i < (int64_t)kOut * kHid) w[(size_t)kIn * kHid + i] = (double)W1[i];
    if (i < kHid) b[i] = (double)b0[i];
    if (i < kOut) b[kHid + i] = (double)b1[i];
}

// ---- host side ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}
// [rows][128] BF16 row-major, box = 64 columns x box_rows, 128-byte swizzle, out-of-range rows read as zero
static int make_tmap(CUtensorMap* m, const void* base, int64_t rows, int box_rows, int64_t cols = kHid, int64_t ld = kHid) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(XQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(XQ_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return XQ_OK;
}

// compact batch [15 words][ld samples] u32, box = 64 samples x 15 words, no swizzle, out-of-range samples read as zero
static int make_tmap_cb(CUtensorMap* m, const void* base, int64_t n, int64_t ld) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(XQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)kCbRows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)kCbRows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(XQ_ERR_CUDA, "cuTensorMapEncodeTiled (compact batch) failed with CUresult %d", (int)r);
    return XQ_OK;
}

// launch with programmatic stream serialization (PDL), optionally as thread-block clusters along y
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, int cluster_y, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at[2];
    int na = 0;
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[na].val.programmaticStreamSerializationAllowed = 1; ++na;
    if (cluster_y > 1) { at[na].id = cudaLaunchAttributeClusterDimension; at[na].val.clusterDim.x = 1; at[na].val.clusterDim.y = cluster_y; at[na].val.clusterDim.z = 1; ++na; }
    cfg.attrs = at; cfg.numAttrs = na;
    ++g_launches;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// where the compact gradient of the current update goes: the rank's exchange slot once xq_dqn_dist_connect has run
static inline float* cur_grad(Fast* f) { return f->connected ? reinterpret_cast<float*>(f->exch) + exch_slot_floats(f->parity, f->rank) : f->grad; }
// multi-GPU: the contraction of an update whose SGD step is left to the exchange pushes its gradient to every rank (epoch = the one
// the following grad_exchange_apply_kernel waits for)
static inline DwPush dw_push(Fast* f, bool apply, bool fused = false) {
    DwPush p;
    if (!apply && f->connected) {
        for (int r = 0; r < kMaxRanks; ++r) p.peers.p[r] = f->peer[r];
        p.rank = f->rank; p.world = f->world; p.parity = f->parity; p.epoch = f->epoch + 1; p.fused = fused;
        p.timeout = f->timeout_ticks; p.status = f->status_dev;
    } else {
        for (int r = 0; r < kMaxRanks; ++r) p.peers.p[r] = nullptr;
    }
    return p;
}

static inline unsigned blocks(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

void dqn_fast_destroy(xq_dqn_s* h) {
    Fast* f = h->fast;
    if (!f) return;
    for (int r = 0; r < f->world; ++r) if (f->connected && r != f->rank && f->peer[r]) cudaIpcCloseMemHandle(f->peer[r]);
    cudaFree(f->exch); cudaFree(f->hg_stage);
    if (f->status_host) cudaFreeHost(f->status_host);
    if (f->hg_pin) cudaFreeHost(f->hg_pin);
    cudaFree(f->H2bf_b); cudaFree(f->zpart_b);
    if (f->aux) cudaStreamDestroy(f->aux);
    if (f->main_hi) cudaStreamDestroy(f->main_hi);
    if (f->ev_join) cudaEventDestroy(f->ev_join);
    if (f->ev_fork) cudaEventDestroy(f->ev_fork);
    for (int i = 0; i < 2; ++i) { if (f->ev_aux[i]) cudaEventDestroy(f->ev_aux[i]); if (f->ev_td[i]) cudaEventDestroy(f->ev_td[i]); }
    cudaFree(f->W0T); cudaFree(f->b0); cudaFree(f->W1); cudaFree(f->b1); cudaFree(f->W1bf); cudaFree(f->W1lo); cudaFree(f->actHhi); cudaFree(f->actHlo);
    cudaFree(f->W0Q); cudaFree(f->b0Q); cudaFree(f->zOpen); cudaFree(f->actMax); cudaFree(f->actZ); cudaFree(f->actPrev);
    cudaFree(f->tW0T); cudaFree(f->tb0); cudaFree(f->tW1); cudaFree(f->tb1); cudaFree(f->tW1bf);
    cudaFree(f->grad); cudaFree(f->boards); cudaFree(f->Hbf); cudaFree(f->H2bf); cudaFree(f->Hf); cudaFree(f->zpart);
    cudaFree(f->cb); cudaFree(f->d0hi); cudaFree(f->d0lo); cudaFree(f->ghi); cudaFree(f->glo); cudaFree(f->q); cudaFree(f->part); cudaFree(f->dbpart); cudaFree(f->info_slots);
    delete f;
    h->fast = nullptr;
}

static int fast_init_alloc(xq_dqn_s* h, Fast* f);
static int fast_init(xq_dqn_s* h) {
    if (h->fast) return XQ_OK;
    if (h->layers.size() != 3 || h->layers[0] != kIn || h->layers[1] != kHid || h->layers[2] != kOut)
        return fail(XQ_ERR_INVALID, "the batched tensor-core path is specialised to the {1260,128,8100} network (src/chessai.cpp:395-404)");
    Fast* f = new (std::nothrow) Fast();
    if (!f) return fail(XQ_ERR_NOMEM, "out of host memory");
    h->fast = f;
    if (int rc = fast_init_alloc(h, f)) { dqn_fast_destroy(h); return rc; }      // never leave a half-built object behind: later calls would launch on null pointers
    return XQ_OK;
}
static int fast_init_alloc(xq_dqn_s* h, Fast* f) {
    XQ_CUDA(cudaMalloc(&f->W0T, sizeof(float) * (kIn + 1) * kHid)); XQ_CUDA(cudaMalloc(&f->b0, sizeof(float) * kHid));
    XQ_CUDA(cudaMalloc(&f->W1, sizeof(float) * kOut * kHid)); XQ_CUDA(cudaMalloc(&f->b1, sizeof(float) * kOut));
    XQ_CUDA(cudaMalloc(&f->W1bf, sizeof(__nv_bfloat16) * kOut * kHid));
    XQ_CUDA(cudaMalloc(&f->W1lo, sizeof(__nv_bfloat16) * QN * kHid));
    XQ_CUDA(cudaMalloc(&f->tW0T, sizeof(float) * (kIn + 1) * kHid)); XQ_CUDA(cudaMalloc(&f->tb0, sizeof(float) * kHid));
    XQ_CUDA(cudaMalloc(&f->tW1, sizeof(float) * kOut * kHid)); XQ_CUDA(cudaMalloc(&f->tb1, sizeof(float) * kOut));
    XQ_CUDA(cudaMalloc(&f->tW1bf, sizeof(__nv_bfloat16) * kOut * kHid));
    XQ_CUDA(cudaMalloc(&f->grad, sizeof(float) * (kGradSize + 8)));      // + 4 floats of loss statistics right behind db1
    f->info = f->grad + kGradSize;
    XQ_CUDA(cudaMemsetAsync(f->grad, 0, sizeof(float) * (kGradSize + 8), h->stream));
    XQ_CUDA(cudaMemsetAsync(f->W0T + (size_t)kIn * kHid, 0, sizeof(float) * kHid, h->stream));      // row kIn = zeros: the padding row of the gather lists
    XQ_CUDA(cudaMemsetAsync(f->tW0T + (size_t)kIn * kHid, 0, sizeof(float) * kHid, h->stream));
    if (int rc = make_tmap(&f->tmW1, f->W1bf, kOut, BN)) return rc;
    if (int rc = make_tmap(&f->tmTW1, f->tW1bf, kOut, BN)) return rc;
    if (int rc = make_tmap(&f->tmW1q, f->W1bf, QN, QN)) return rc;
    if (int rc = make_tmap(&f->tmW1loq, f->W1lo, QN, QN)) return rc;
    XQ_CUDA(cudaFuncSetAttribute(q90_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kQSmem));
    XQ_CUDA(cudaFuncSetAttribute(l1_gemm_kernel<EPI_ROWMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmem));
    XQ_CUDA(cudaFuncSetAttribute(l1_gemm_kernel<EPI_STORE_TANH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmem));
    XQ_CUDA(cudaFuncSetAttribute(dw_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDwSmem));
    XQ_CUDA(cudaMalloc(&f->part, sizeof(float) * kDwMTiles * kDwSplits * BM * kHid));
    XQ_CUDA(cudaMalloc(&f->dbpart, sizeof(float) * kDwSplits * BM));
    XQ_CUDA(cudaMalloc(&f->info_slots, sizeof(float) * kInfoSlots * 4));
    return XQ_OK;
}

static int fast_reserve(xq_dqn_s* h, int64_t n) {
    Fast* f = h->fast;
    if (n <= f->cap) return XQ_OK;
    cudaFree(f->boards); cudaFree(f->Hbf); cudaFree(f->H2bf); cudaFree(f->Hf); cudaFree(f->zpart); cudaFree(f->cb);
    cudaFree(f->H2bf_b); cudaFree(f->zpart_b); f->H2bf_b = nullptr; f->zpart_b = nullptr;
    cudaFree(f->d0hi); cudaFree(f->d0lo); cudaFree(f->ghi); cudaFree(f->glo);
    f->boards = nullptr; f->Hbf = f->H2bf = nullptr; f->Hf = f->zpart = nullptr; f->cb = nullptr; f->d0hi = f->d0lo = f->ghi = f->glo = nullptr; f->cap = 0;
    const int64_t rows = (n + BM - 1) / BM * BM;
    XQ_CUDA(cudaMalloc(&f->boards, sizeof(Transition) * n));
    XQ_CUDA(cudaMalloc(&f->Hbf, sizeof(__nv_bfloat16) * rows * kHid)); XQ_CUDA(cudaMalloc(&f->H2bf, sizeof(__nv_bfloat16) * rows * kHid));
    XQ_CUDA(cudaMalloc(&f->Hf, sizeof(float) * rows * kHid)); XQ_CUDA(cudaMalloc(&f->zpart, sizeof(float) * kPartsPad * rows));
    XQ_CUDA(cudaMalloc(&f->H2bf_b, sizeof(__nv_bfloat16) * rows * kHid)); XQ_CUDA(cudaMalloc(&f->zpart_b, sizeof(float) * kPartsPad * rows));
    XQ_CUDA(cudaMalloc(&f->cb, sizeof(uint32_t) * kCbRows * rows));
    XQ_CUDA(cudaMalloc(&f->d0hi, sizeof(__nv_bfloat16) * rows * kHid)); XQ_CUDA(cudaMalloc(&f->d0lo, sizeof(__nv_bfloat16) * rows * kHid));
    XQ_CUDA(cudaMalloc(&f->ghi, sizeof(__nv_bfloat16) * rows * kHid)); XQ_CUDA(cudaMalloc(&f->glo, sizeof(__nv_bfloat16) * rows * kHid));
    f->cap = n; f->tm_rows = 0;
    return XQ_OK;
}

// tensor maps whose extents follow the batch size (out-of-range rows / samples read as zero)
static int fast_maps(xq_dqn_s* h, int64_t n) {
    Fast* f = h->fast;
    if (n == f->tm_rows) return XQ_OK;
    const int64_t ld = (f->cap + BM - 1) / BM * BM;
    if (int rc = make_tmap(&f->tmH, f->Hbf, n, BM)) return rc;
    if (int rc = make_tmap(&f->tmH2, f->H2bf, n, BM)) return rc;
    if (int rc = make_tmap(&f->tmH2_b, f->H2bf_b, n, BM)) return rc;
    if (int rc = make_tmap(&f->tmD0hi, f->d0hi, kHid, kHid, n, ld)) return rc;     // delta0^T [128 hidden][n samples], row stride ld
    if (int rc = make_tmap(&f->tmD0lo, f->d0lo, kHid, kHid, n, ld)) return rc;
    if (int rc = make_tmap(&f->tmGhi, f->ghi, kHid, kHid, n, ld)) return rc;
    if (int rc = make_tmap(&f->tmGlo, f->glo, kHid, kHid, n, ld)) return rc;
    if (int rc = make_tmap_cb(&f->tmCb, f->cb, n, ld)) return rc;
    f->tm_rows = n;
    return XQ_OK;
}

// the fast path's copies follow the FP64 parameters whenever those were modified last
static int ensure_fast(xq_dqn_s* h) {
    if (int rc = fast_init(h)) return rc;
    Fast* f = h->fast;
    if (!h->fast_current) {
        f64_to_fast_kernel<<<blocks((int64_t)kOut * kHid, 256), 256, 0, h->stream>>>(h->d_w, h->d_b, f->W0T, f->b0, f->W1, f->b1, f->W1bf, f->W1lo);
        XQ_LAUNCH_CHECK();
        h->fast_current = true; ++f->w_version;
    }
    if (!f->target_current) {
        f64_to_fast_kernel<<<blocks((int64_t)kOut * kHid, 256), 256, 0, h->stream>>>(h->d_tw, h->d_tb, f->tW0T, f->tb0, f->tW1, f->tb1, f->tW1bf, (__nv_bfloat16*)nullptr);
        XQ_LAUNCH_CHECK();
        f->target_current = true;
    }
    return XQ_OK;
}

int dqn_ensure_f64(xq_dqn_s* h) {
    if (h->f64_current || !h->fast) return XQ_OK;
    Fast* f = h->fast;
    fast_to_f64_kernel<<<blocks((int64_t)kOut * kHid, 256), 256, 0, h->stream>>>(h->d_w, h->d_b, f->W0T, f->b0, f->W1, f->b1);
    XQ_LAUNCH_CHECK();
    h->f64_current = true;
    return XQ_OK;
}
int dqn_fast_weights(xq_dqn_s* h, FastWeights* out) {
    if (int rc = ensure_fast(h)) return rc;
    out->W0T = h->fast->W0T; out->b0 = h->fast->b0; out->W1 = h->fast->W1; out->b1 = h->fast->b1;
    return XQ_OK;
}
void dqn_target_changed(xq_dqn_s* h) { if (h->fast) h->fast->target_current = false; }

// the n rows of the batch, cut into row_splits CTAs per column tile
static int launch_gemm(xq_dqn_s* h, int mode, const CUtensorMap& tmA, const CUtensorMap& tmB, const float* b1, int64_t n, float* q,
                       cudaStream_t stream = nullptr, float* zpart = nullptr, int row_splits = 0) {
    Fast* f = h->fast;
    if (!stream) stream = h->stream;
    if (!zpart) zpart = f->zpart;
    const int m_tiles = (int)((n + BM - 1) / BM);
    int n_splits = row_splits > 0 ? row_splits : 148 / kNTiles;      // default: 4 row splits x 37 column tiles = 148 CTAs
    if (n_splits > m_tiles) n_splits = m_tiles;
    const dim3 grid(kNTiles, n_splits);
    const int64_t zstride = (f->cap + BM - 1) / BM * BM;
    if (mode == EPI_ROWMAX)
        XQ_CUDA(launch_pdl(l1_gemm_kernel<EPI_ROWMAX>, grid, dim3(kGemmThreads), kGemmSmem, stream, 1, tmA, tmB, b1, (int)n, m_tiles, n_splits,
                           zpart, zstride, (float*)nullptr));
    else
        XQ_CUDA(launch_pdl(l1_gemm_kernel<EPI_STORE_TANH>, grid, dim3(kGemmThreads), kGemmSmem, stream, 1, tmA, tmB, b1, (int)n, m_tiles, n_splits,
                           (float*)nullptr, zstride, q));
    return XQ_OK;
}

// Q(s)[0..95] (row-major [n][96] FP32, device) for n env records resident on the device, on `stream`:
// layer-0 gather (FP32) + split-precision tensor-core contraction with W1 rows 0..95
int dqn_q90_device(xq_dqn_s* h, const xq_env_rec* envs_dev, int64_t n, float* q90_dev, cudaStream_t stream, bool carried, ActCarry* carry) {
    if (int rc = ensure_fast(h)) return rc;
    Fast* f = h->fast;
    if (n > f->act_cap) {
        cudaFree(f->actHhi); cudaFree(f->actHlo); cudaFree(f->actZ); cudaFree(f->actPrev);
        f->actHhi = f->actHlo = nullptr; f->actZ = nullptr; f->actPrev = nullptr; f->act_cap = 0; f->act_rows = 0; f->actz_version = 0;
        const int64_t rows = (n + BM - 1) / BM * BM;
        XQ_CUDA(cudaMalloc(&f->actHhi, sizeof(__nv_bfloat16) * rows * kHid)); XQ_CUDA(cudaMalloc(&f->actHlo, sizeof(__nv_bfloat16) * rows * kHid));
        XQ_CUDA(cudaMalloc(&f->actZ, sizeof(int32_t) * n * kHid)); XQ_CUDA(cudaMalloc(&f->actPrev, sizeof(uint32_t) * n * 12));
        f->act_cap = n;
    }
    if (n != f->act_rows) {
        if (int rc = make_tmap(&f->tmActHi, f->actHhi, n, BM)) return rc;
        if (int rc = make_tmap(&f->tmActLo, f->actHlo, n, BM)) return rc;
        f->act_rows = n;
    }
    if (!f->W0Q) {
        XQ_CUDA(cudaMalloc(&f->W0Q, sizeof(int32_t) * (kIn + 1) * kHid)); XQ_CUDA(cudaMalloc(&f->b0Q, sizeof(int32_t) * kHid)); XQ_CUDA(cudaMalloc(&f->zOpen, sizeof(int32_t) * kHid));
        XQ_CUDA(cudaMalloc(&f->actMax, sizeof(uint32_t) * 4));
        XQ_CUDA(cudaMemsetAsync(f->actMax, 0, sizeof(uint32_t) * 4, stream));
    }
    if (f->actq_version != f->w_version) {       // the online W0 / b0 changed: new fixed-point table (scale from max |w|), every sum starts over
        act_quant_max_kernel<<<148, 256, 0, stream>>>(f->W0T, f->b0, f->actMax + f->act_slot);
        XQ_LAUNCH_CHECK();
        act_quant_kernel<<<148, 256, 0, stream>>>(f->W0T, f->b0, f->actMax + f->act_slot, f->actMax + (f->act_slot ^ 1), f->W0Q, f->b0Q,
                                                  reinterpret_cast<float*>(f->actMax + 2));
        XQ_LAUNCH_CHECK();
        act_zopen_kernel<<<1, kHid, 0, stream>>>(f->W0Q, f->b0Q, f->zOpen);
        XQ_LAUNCH_CHECK();
        f->act_slot ^= 1;
        f->actq_version = f->w_version;
    }
    const int fresh_all = f->actz_version != f->w_version ? 1 : 0;
    // `carried`: the caller's act_team_kernel has already brought the sums, the remembered boards and h(s) of these n envs up to date
    // (tail of the previous ply of the same xq_selfplay_collect call); only valid while nothing else could have touched them
    if (!(carried && !fresh_all && n == f->act_carried_n)) {
        l0_act_kernel<<<blocks(n, 32), 256, 0, stream>>>(envs_dev, n, f->W0Q, f->b0Q, reinterpret_cast<const float*>(f->actMax + 2), f->actZ, f->actPrev, fresh_all,
                                                        f->actHhi, f->actHlo);
        XQ_LAUNCH_CHECK();
    }
    f->actz_version = f->w_version;
    f->act_carried_n = n;
    if (carry) {
        carry->W0Q = f->W0Q; carry->zOpen = f->zOpen; carry->inv_scale = reinterpret_cast<const float*>(f->actMax + 2);
        carry->Z = f->actZ; carry->Prev = f->actPrev; carry->Hhi = f->actHhi; carry->Hlo = f->actHlo;
    }
    const int m_tiles = (int)((n + BM - 1) / BM);
    XQ_CUDA(launch_pdl(q90_gemm_kernel, dim3(m_tiles < 148 ? m_tiles : 148), dim3(kGemmThreads), kQSmem, stream, 1, f->tmActHi, f->tmActLo, f->tmW1q,
                       f->tmW1loq, (const float*)f->b1, (int)n, m_tiles, q90_dev));
    return XQ_OK;
}

// Half `half` (0 or 1) of the n envs of a collector call whose layer-0 sums are carried by the act kernel (dqn_q90_device has run for the
// whole range in this call): only the contraction, on `stream`, with tensor maps over the half's rows of h(s).  The first half is a multiple
// of the 128-env tile, the second takes the rest; *off / *m return the half's env range.
int dqn_q90_half(xq_dqn_s* h, int64_t n, int half, float* q90_dev, cudaStream_t stream, ActCarry* carry, int64_t* off_out, int64_t* m_out) {
    Fast* f = h->fast;
    if (!f || n != f->act_rows || n != f->act_carried_n) return fail(XQ_ERR_STATE, "dqn_q90_half: the whole range has not been prepared");
    if (half < 0 || half > 1) return fail(XQ_ERR_INVALID, "dqn_q90_half: bad half");
    const int64_t size = ((n + 1) / 2 + BM - 1) / BM * BM;
    if (size >= n) return fail(XQ_ERR_INVALID, "dqn_q90_half: too few envs for two halves");
    if (f->act_sub_n != n) {
        for (int k = 0; k < 2; ++k) {
            const int64_t o = k * size, m = std::min<int64_t>(size, n - o);
            if (int rc = make_tmap(&f->tmActHiS[k], f->actHhi + o * kHid, m, BM)) return rc;
            if (int rc = make_tmap(&f->tmActLoS[k], f->actHlo + o * kHid, m, BM)) return rc;
        }
        f->act_sub_n = n;
    }
    const int64_t off = half * size, m = std::min<int64_t>(size, n - off);
    if (carry) {
        carry->W0Q = f->W0Q; carry->zOpen = f->zOpen; carry->inv_scale = reinterpret_cast<const float*>(f->actMax + 2);
        carry->Z = f->actZ + off * kHid; carry->Prev = f->actPrev + off * 12; carry->Hhi = f->actHhi + off * kHid; carry->Hlo = f->actHlo + off * kHid;
    }
    const int m_tiles = (int)((m + BM - 1) / BM);
    XQ_CUDA(launch_pdl(q90_gemm_kernel, dim3(m_tiles < 148 ? m_tiles : 148), dim3(kGemmThreads), kQSmem, stream, 1, f->tmActHiS[half], f->tmActLoS[half], f->tmW1q,
                       f->tmW1loq, (const float*)f->b1, (int)m, m_tiles, q90_dev + off * QN));
    *off_out = off; *m_out = m;
    return XQ_OK;
}

}  // namespace xq

using namespace xq;

#define XQ_DQN_ENTER(h)                                                      \
    if (!(h)) return fail(XQ_ERR_INVALID, "%s: null handle", __func__);      \
    XQ_CUDA(cudaSetDevice((h)->device))

extern "C" {

int xq_dqn_forward_boards(xq_dqn_t h, const xq_env_rec* boards_host, int64_t n, float* q_host) {
    XQ_DQN_ENTER(h);
    if (!boards_host || !q_host || n <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_forward_boards: bad arguments");
    if (int rc = ensure_fast(h)) return rc;
    if (int rc = fast_reserve(h, n)) return rc;
    Fast* f = h->fast;
    if (n > f->q_cap) { cudaFree(f->q); f->q = nullptr; f->q_cap = 0; XQ_CUDA(cudaMalloc(&f->q, sizeof(float) * n * kOut)); f->q_cap = n; }
    XQ_CUDA(cudaMemcpyAsync(f->boards, boards_host, sizeof(xq_env_rec) * n, cudaMemcpyHostToDevice, h->stream));
    l0_forward_kernel<<<blocks(n * 32, 256), 256, 0, h->stream>>>(reinterpret_cast<const uint8_t*>(f->boards), sizeof(xq_env_rec), n, f->W0T, f->b0, f->Hbf, nullptr);
    XQ_LAUNCH_CHECK();
    if (int rc = fast_maps(h, n)) return rc;
    if (int rc = launch_gemm(h, EPI_STORE_TANH, f->tmH, f->tmW1, f->b1, n, f->q)) return rc;
    XQ_CUDA(cudaMemcpyAsync(q_host, f->q, sizeof(float) * n * kOut, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

}  // extern "C" (reopened below)
namespace xq {
// one batched TD update on the batch described by `ref` (contiguous transitions or in-place replay draws): 4 kernels
// a gradient exchange of this handle timed out earlier: the replicas may differ, every later update call fails (sticky)
static int dist_check(xq_dqn_s* h) {
    Fast* f = h->fast;
    if (f && f->status_host && *reinterpret_cast<volatile uint32_t*>(f->status_host) != 0)
        return fail(XQ_ERR_STATE, "multi-GPU gradient exchange %u timed out (a peer never arrived): the update was not applied and the replicas may differ; "
                                  "recreate the handles on every rank", *reinterpret_cast<volatile uint32_t*>(f->status_host));
    return XQ_OK;
}

int td_update_core(xq_dqn_s* h, const BatchRef& ref, int64_t n, int use_target_net, double lr, int apply) {
    if (int rc = ensure_fast(h)) return rc;
    if (int rc = fast_reserve(h, n)) return rc;
    Fast* f = h->fast;
    if (int rc = dist_check(h)) return rc;
    // on a handle connected to its peers EVERY applied update exchanges its gradient (include/xq.h): the contraction itself does it
    const bool exchange = apply && f->connected;
    if (int rc = fast_maps(h, n)) return rc;
    if (lr <= 0) lr = h->lr;
    const int64_t ld = (f->cap + BM - 1) / BM * BM;
    // Four kernels chained with programmatic dependent launch: each one's set-up (barriers, TMEM, operand tiles that do not
    // depend on its predecessor) overlaps the predecessor's tail.
    // 1. h(s) with the online net; h(s') with the online (ChessAI::train) or target (DQN::train) net; compact batch
    XQ_CUDA(launch_pdl(l0_pair_kernel, dim3(blocks(n, kL0Warps)), dim3(kL0Warps * 32), 0, h->stream, 1, ref, n, f->W0T, f->b0,
                       use_target_net ? f->tW0T : f->W0T, use_target_net ? f->tb0 : f->b0, f->Hf, f->H2bf, f->cb, ld, f->info_slots,
                       kInfoSlots * 4, 3));
    // 2. max_a z(s')[a] over all 8100 outputs
    if (int rc = launch_gemm(h, EPI_ROWMAX, f->tmH2, use_target_net ? f->tmTW1 : f->tmW1, use_target_net ? f->tb1 : f->b1, n, nullptr)) return rc;
    // 3. TD error, delta0, delta1 h
    XQ_CUDA(launch_pdl(td_delta_kernel, dim3(blocks(n * 32, 256)), dim3(256), 0, h->stream, 1, f->cb, n, f->Hf, f->W1, f->b1, f->zpart, ld, kParts,
                       (float)h->gamma, h->mode, f->d0hi, f->d0lo, f->ghi, f->glo, ld, f->info_slots));
    // 4. dW0 / db0 / dW1 / db1 contraction, cluster reduction and the SGD step (or the compact gradient)
    XQ_CUDA(launch_pdl(dw_gemm_kernel, dim3(kDwMTiles, kDwSplits), dim3(kDwThreads), kDwSmem, h->stream, kDwSplits, f->tmD0hi, f->tmD0lo, f->tmGhi,
                       f->tmGlo, f->tmCb, (int)n, f->part, f->dbpart, f->info_slots, f->info, cur_grad(f), f->W0T, f->b0, f->W1, f->b1, f->W1bf,
                       f->W1lo, (float)lr, (apply && !exchange) ? 1 : 0, dw_push(f, apply != 0 && !exchange, exchange)));
    if (exchange) { ++f->epoch; f->parity ^= 1; }
    if (apply) { h->f64_current = false; ++f->w_version; }
    return XQ_OK;
}

int dqn_td_update_sampled(xq_dqn_s* h, const void* ring, int64_t size, uint64_t seed, uint32_t counter, int64_t n, int use_target_net,
                          double lr, int apply) {
    const BatchRef ref{reinterpret_cast<const uint8_t*>(ring), size, seed, counter, 1};
    return td_update_core(h, ref, n, use_target_net, lr, apply);
}

int dqn_exchange_apply(xq_dqn_s* h, double lr);

// n_updates sequential TD updates on replay draws (counters counter0, counter0 + 1, ...), bit-identical to n_updates calls of
// dqn_td_update_sampled(..., use_target_net = 1, apply = 1), but software-pipelined over two streams: between two target syncs the
// bootstrap branch of an update -- h(s') with the TARGET net and the [B x 128] x [128 x 8100] row-max GEMM -- does not depend on the
// online weights, so for update i+1 it runs on an auxiliary stream underneath update i's online branch
// [h(s) -> TD error -> gradient contraction + SGD], which alone stays on the critical path.  Two slots of (h(s'), row-max partials).
int dqn_td_update_pipelined(xq_dqn_s* h, const void* ring, int64_t size, uint64_t seed, uint32_t counter0, int64_t n, int n_updates, double lr) {
    if (int rc = ensure_fast(h)) return rc;
    if (int rc = fast_reserve(h, n)) return rc;
    Fast* f = h->fast;
    if (int rc = fast_maps(h, n)) return rc;
    if (int rc = dist_check(h)) return rc;
    if (lr <= 0) lr = h->lr;
    if (!f->aux) {
        int lo = 0, hi = 0;
        XQ_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        XQ_CUDA(cudaStreamCreateWithPriority(&f->aux, cudaStreamNonBlocking, lo));       // lowest priority = the priority of a default-created stream: measured best
                                                                                          // when both branches have EQUAL priority (29.0 us per update; 34.4 with the
                                                                                          // online branch on a higher-priority stream, 41 with the bootstrap branch higher)
        XQ_CUDA(cudaEventCreateWithFlags(&f->ev_fork, cudaEventDisableTiming));
        for (int i = 0; i < 2; ++i) { XQ_CUDA(cudaEventCreateWithFlags(&f->ev_aux[i], cudaEventDisableTiming)); XQ_CUDA(cudaEventCreateWithFlags(&f->ev_td[i], cudaEventDisableTiming)); }
    }
    const int64_t ld = (f->cap + BM - 1) / BM * BM;
    // The online branch (the critical path) can run on a stream of the library with a HIGHER priority than the bootstrap branch.  Measured per
    // update (batch 4096 per GPU, us; equal priorities / online branch higher):  1 GPU 33.5 (29.6 .. 35.5 from call to call) / 34.6;  2 GPUs 36.3 / 38.9;
    // 8 GPUs 47.1 (43.9 .. 48.5) / 42.5 (+- 0.1).  With equal priorities the row-max GEMM of update i+1 and the 88 whole-SM CTAs of the contraction of
    // update i race for SMs; once the contraction also waits for its peers' row blocks (it then holds its SMs for ~17 us instead of ~10) losing that
    // race costs more than the GEMM's loss of the SMs under the h(s) gather, so the rule is: higher priority from 4 ranks on.
    const bool main_prio = f->connected && f->world >= 4;
    if (main_prio && !f->main_hi) {
        int lo = 0, hi = 0;
        XQ_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        XQ_CUDA(cudaStreamCreateWithPriority(&f->main_hi, cudaStreamNonBlocking, hi));
    }
    if (!f->ev_join) XQ_CUDA(cudaEventCreateWithFlags(&f->ev_join, cudaEventDisableTiming));
    cudaStream_t main = main_prio ? f->main_hi : h->stream, aux = f->aux;
    XQ_CUDA(cudaEventRecord(f->ev_fork, h->stream));             // the target net and the ring are final for the other streams
    XQ_CUDA(cudaStreamWaitEvent(aux, f->ev_fork, 0));
    if (main != h->stream) XQ_CUDA(cudaStreamWaitEvent(main, f->ev_fork, 0));
    // bootstrap branch of update i into slot i & 1, in two parts.  h(s') (small CTAs) is enqueued early and runs under the online branch of
    // update i-1; the row-max GEMM needs a whole SM's shared memory per CTA, exactly like the gradient contraction of the online branch, so
    // when it is released decides whether it sits on the critical path (below).
    auto aux_l0 = [&](int i) -> int {
        const int slot = i & 1;
        const BatchRef ref{reinterpret_cast<const uint8_t*>(ring), size, seed, counter0 + (uint32_t)i, 1};
        XQ_CUDA(launch_pdl(l0_pair_kernel, dim3(blocks(n, kL0Warps)), dim3(kL0Warps * 32), 0, aux, 1, ref, n, f->W0T, f->b0, f->tW0T, f->tb0, f->Hf,
                           slot ? f->H2bf_b : f->H2bf, f->cb, ld, f->info_slots, 0, 2));
        return XQ_OK;
    };
    // The row-max GEMM of update i+1 is released when the row-max partials of update i are in, i.e. BEFORE the TD-error kernel of update i:
    // the GEMM's CTAs start under the TD-error kernel (small CTAs, they co-reside), the contraction's 88 CTAs take their SMs as they become
    // free, and the GEMM is (nearly) done when the contraction ends.  It is cut into 5 row splits (185 CTAs instead of 4 x 37 = 148).  Slot
    // reuse: the partials slot of update i+1 was last read by the TD-error kernel of update i-1, which precedes the event in stream order.
    // Measured per update at batch 4096: 29.0 us; 29.6 / 29.0 / 31.1 us with 4 / 6 / 8 splits; released when update i is complete 36.4 us,
    // after its TD-error kernel 34.0 us; enqueued a whole update ahead (no event) 33.4 us.  Same results bit for bit (DESIGN.md section 4).
    auto aux_gemm = [&](int i, cudaEvent_t gate) -> int {
        const int slot = i & 1;
        if (gate) XQ_CUDA(cudaStreamWaitEvent(aux, gate, 0));
        if (int rc = launch_gemm(h, EPI_ROWMAX, slot ? f->tmH2_b : f->tmH2, f->tmTW1, f->tb1, n, nullptr, aux, slot ? f->zpart_b : f->zpart, 5)) return rc;
        XQ_CUDA(cudaEventRecord(f->ev_aux[slot], aux));
        return XQ_OK;
    };
    if (int rc = aux_l0(0)) return rc;
    if (int rc = aux_gemm(0, nullptr)) return rc;
    for (int i = 0; i < n_updates; ++i) {
        const int slot = i & 1;
        const BatchRef ref{reinterpret_cast<const uint8_t*>(ring), size, seed, counter0 + (uint32_t)i, 1};
        if (i + 1 < n_updates) if (int rc = aux_l0(i + 1)) return rc;
        XQ_CUDA(launch_pdl(l0_pair_kernel, dim3(blocks(n, kL0Warps)), dim3(kL0Warps * 32), 0, main, 1, ref, n, f->W0T, f->b0, f->tW0T, f->tb0, f->Hf,
                           f->H2bf, f->cb, ld, f->info_slots, kInfoSlots * 4, 1));
        XQ_CUDA(cudaStreamWaitEvent(main, f->ev_aux[slot], 0));  // the row-max partials of this update
        XQ_CUDA(cudaEventRecord(f->ev_td[slot], main));
        if (i + 1 < n_updates) if (int rc = aux_gemm(i + 1, f->ev_td[slot])) return rc;
        XQ_CUDA(launch_pdl(td_delta_kernel, dim3(blocks(n * 32, 256)), dim3(256), 0, main, 1, f->cb, n, f->Hf, f->W1, f->b1, slot ? f->zpart_b : f->zpart,
                           ld, kParts, (float)h->gamma, h->mode, f->d0hi, f->d0lo, f->ghi, f->glo, ld, f->info_slots));
        // multi-GPU: the contraction exchanges the gradient and applies the SGD step itself
        XQ_CUDA(launch_pdl(dw_gemm_kernel, dim3(kDwMTiles, kDwSplits), dim3(kDwThreads), kDwSmem, main, kDwSplits, f->tmD0hi, f->tmD0lo, f->tmGhi,
                           f->tmGlo, f->tmCb, (int)n, f->part, f->dbpart, f->info_slots, f->info, cur_grad(f), f->W0T, f->b0, f->W1, f->b1, f->W1bf,
                           f->W1lo, (float)lr, f->connected ? 0 : 1, dw_push(f, !f->connected, true)));
        if (f->connected) { ++f->epoch; f->parity ^= 1; }
    }
    if (main != h->stream) {                // the online branch ran on the library's own high-priority stream: join
        XQ_CUDA(cudaEventRecord(f->ev_join, main));
        XQ_CUDA(cudaStreamWaitEvent(h->stream, f->ev_join, 0));
    }
    h->f64_current = false; ++f->w_version;
    return XQ_OK;
}

}  // namespace xq
using namespace xq;
extern "C" {

int xq_dqn_td_update_device(xq_dqn_t h, const void* batch_dev, int64_t n, int use_target_net, double lr, int apply) {
    XQ_DQN_ENTER(h);
    if (!batch_dev || n <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_td_update_device: bad arguments");
    const BatchRef ref{reinterpret_cast<const uint8_t*>(batch_dev), n, 0, 0, 0};
    return td_update_core(h, ref, n, use_target_net, lr, apply);
}

int xq_dqn_td_update(xq_dqn_t h, const xq_transition* batch_host, int64_t n, int use_target_net, double lr, float* info_host) {
    XQ_DQN_ENTER(h);
    if (!batch_host || n <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_td_update: bad arguments");
    if (int rc = ensure_fast(h)) return rc;
    if (int rc = fast_reserve(h, n)) return rc;
    Fast* f = h->fast;
    XQ_CUDA(cudaMemcpyAsync(f->boards, batch_host, sizeof(Transition) * n, cudaMemcpyHostToDevice, h->stream));
    if (int rc = xq_dqn_td_update_device(h, f->boards, n, use_target_net, lr, 1)) return rc;
    if (info_host) XQ_CUDA(cudaMemcpyAsync(info_host, f->info, sizeof(float) * 4, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_dqn_grad_buffer(xq_dqn_t h, void** dev_ptr, int64_t* n_floats) {
    XQ_DQN_ENTER(h);
    if (int rc = ensure_fast(h)) return rc;
    if (dev_ptr) *dev_ptr = cur_grad(h->fast);
    if (n_floats) *n_floats = kGradSize;
    return XQ_OK;
}

int xq_dqn_apply_grads(xq_dqn_t h, double lr) {
    XQ_DQN_ENTER(h);
    if (int rc = ensure_fast(h)) return rc;
    Fast* f = h->fast;
    if (lr <= 0) lr = h->lr;
    apply_kernel<<<blocks(kGradSize, 256), 256, 0, h->stream>>>(f->W0T, f->b0, f->W1, f->b1, f->W1bf, f->W1lo, cur_grad(f), (float)lr);
    XQ_LAUNCH_CHECK();
    h->f64_current = false; ++f->w_version;
    return XQ_OK;
}

int xq_dqn_dist_export(xq_dqn_t h, void* handle_out) {
    XQ_DQN_ENTER(h);
    if (!handle_out) return fail(XQ_ERR_INVALID, "xq_dqn_dist_export: null handle buffer");
    if (int rc = ensure_fast(h)) return rc;
    Fast* f = h->fast;
    if (!f->exch) {
        XQ_CUDA(cudaMalloc(&f->exch, kExchBytes));
        XQ_CUDA(cudaMemset(f->exch, 0, kExchBytes));
        XQ_CUDA(cudaMalloc(&f->hg_stage, kHgCap));
        XQ_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&f->hg_pin), (size_t)(kMaxRanks + 1) * kHgCap, cudaHostAllocDefault));
        XQ_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&f->status_host), 64, cudaHostAllocMapped));
        memset(f->status_host, 0, 64);
        XQ_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&f->status_dev), f->status_host, 0));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == XQ_IPC_HANDLE_BYTES, "CUDA IPC handle size");
    cudaIpcMemHandle_t ipc;
    XQ_CUDA(cudaIpcGetMemHandle(&ipc, f->exch));
    memcpy(handle_out, &ipc, sizeof(ipc));
    return XQ_OK;
}

int xq_dqn_dist_connect(xq_dqn_t h, int rank, int world, const void* handles) {
    XQ_DQN_ENTER(h);
    if (!handles || world < 1 || world > kMaxRanks || rank < 0 || rank >= world)
        return fail(XQ_ERR_INVALID, "xq_dqn_dist_connect: bad arguments (world must be 1..%d)", kMaxRanks);
    if (int rc = ensure_fast(h)) return rc;
    Fast* f = h->fast;
    if (!f->exch) return fail(XQ_ERR_STATE, "xq_dqn_dist_connect: call xq_dqn_dist_export first");
    if (f->connected) return fail(XQ_ERR_STATE, "xq_dqn_dist_connect: already connected");
    for (int r = 0; r < world; ++r) {
        if (r == rank) { f->peer[r] = f->exch; continue; }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, static_cast<const uint8_t*>(handles) + (size_t)r * XQ_IPC_HANDLE_BYTES, sizeof(ipc));
        void* p = nullptr;
        XQ_CUDA(cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
        f->peer[r] = static_cast<uint8_t*>(p);
    }
    f->rank = rank; f->world = world; f->parity = 0; f->epoch = 0; f->connected = true;
    {   // how long a wait for a peer may last (XQ_DIST_TIMEOUT_MS, default 20 s: host-side callbacks, logging, a first-call allocation on a
        // peer are legitimate skew), in clock64 ticks of this device
        const char* e = getenv("XQ_DIST_TIMEOUT_MS");
        const double ms = e && atof(e) > 0 ? atof(e) : 20000.0;
        int khz = 0;
        XQ_CUDA(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device));
        f->timeout_ticks = (long long)(ms * (double)(khz > 0 ? khz : 2000000));
    }
    return XQ_OK;
}

int xq_dqn_dist_allreduce_apply(xq_dqn_t h, double lr) {
    XQ_DQN_ENTER(h);
    if (!h->fast || !h->fast->connected) return fail(XQ_ERR_STATE, "xq_dqn_dist_allreduce_apply: not connected (xq_dqn_dist_connect)");
    if (int rc = dist_check(h)) return rc;
    return dqn_exchange_apply(h, lr);
}

}  // extern "C" (reopened below)
namespace xq {
int dqn_exchange_apply(xq_dqn_s* h, double lr) {
    Fast* f = h->fast;
    if (lr <= 0) lr = h->lr;
    PeerPtrs pp;
    for (int r = 0; r < kMaxRanks; ++r) pp.p[r] = f->peer[r];
    ++f->epoch;
    XQ_CUDA(launch_pdl(grad_exchange_apply_kernel, dim3(blocks(kGradPad / 4, 256)), dim3(256), 0, h->stream, 1, pp, f->rank, f->world, f->parity, f->epoch, f->W0T,
                       f->b0, f->W1, f->b1, f->W1bf, f->W1lo, (float)lr, f->timeout_ticks, f->status_dev));
    f->parity ^= 1;
    h->f64_current = false; ++f->w_version;
    return XQ_OK;
}
}  // namespace xq
extern "C" {

int xq_dqn_dist_info(xq_dqn_t h, int* rank, int* world) {
    if (!h) return fail(XQ_ERR_INVALID, "xq_dqn_dist_info: null handle");
    const bool c = h->fast && h->fast->connected;
    if (rank) *rank = c ? h->fast->rank : 0;
    if (world) *world = c ? h->fast->world : 1;
    return XQ_OK;
}

int xq_dqn_dist_allgather(xq_dqn_t h, const void* send_host, int64_t bytes, void* recv_host) {
    XQ_DQN_ENTER(h);
    if (!h->fast || !h->fast->connected) return fail(XQ_ERR_STATE, "xq_dqn_dist_allgather: not connected (xq_dqn_dist_connect)");
    if (!send_host || !recv_host || bytes <= 0 || bytes > (int64_t)kHgCap) return fail(XQ_ERR_INVALID, "xq_dqn_dist_allgather: 1..%d bytes per rank", (int)kHgCap);
    Fast* f = h->fast;
    if (int rc = dist_check(h)) return rc;
    const int n16 = (int)((bytes + 15) / 16);
    memset(f->hg_pin, 0, (size_t)n16 * 16);            // pinned staging on both sides: one H2D copy, one kernel, one strided D2H copy, one synchronisation
    memcpy(f->hg_pin, send_host, (size_t)bytes);
    XQ_CUDA(cudaMemcpyAsync(f->hg_stage, f->hg_pin, (size_t)n16 * 16, cudaMemcpyHostToDevice, h->stream));
    PeerPtrs pp;
    for (int r = 0; r < kMaxRanks; ++r) pp.p[r] = f->peer[r];
    const uint32_t seq = ++f->hg_seq;
    const int parity = (int)(seq & 1u);
    host_gather_kernel<<<1, 256, 0, h->stream>>>(pp, f->rank, f->world, parity, seq, reinterpret_cast<const uint4*>(f->hg_stage), n16, f->timeout_ticks, f->status_dev);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaMemcpy2DAsync(f->hg_pin + kHgCap, (size_t)n16 * 16, f->exch + kExchHgOff + (size_t)parity * kMaxRanks * kHgCap, kHgCap, (size_t)n16 * 16, (size_t)f->world,
                              cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    for (int r = 0; r < f->world; ++r) memcpy(static_cast<uint8_t*>(recv_host) + (size_t)r * (size_t)bytes, f->hg_pin + kHgCap + (size_t)r * (size_t)n16 * 16, (size_t)bytes);
    return dist_check(h);
}

int xq_dqn_dist_status(xq_dqn_t h, int* timed_out) {
    XQ_DQN_ENTER(h);
    if (!h->fast || !h->fast->exch || !timed_out) return fail(XQ_ERR_STATE, "xq_dqn_dist_status: no exchange buffer");
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    *timed_out = (int)*reinterpret_cast<volatile uint32_t*>(h->fast->status_host);      // epoch of the first exchange that timed out, 0 = none
    return XQ_OK;
}

#ifdef XQ_TIMELINE
int xq_debug_timeline(long long* out_host, int64_t n) {   // profiling builds only
    if (n > (int64_t)(sizeof(long long) * 2 * 160 * 64)) n = sizeof(long long) * 2 * 160 * 64;
    XQ_CUDA(cudaDeviceSynchronize());
    XQ_CUDA(cudaMemcpyFromSymbol(out_host, g_tl, (size_t)n));
    return XQ_OK;
}
#endif

}  // extern "C"
