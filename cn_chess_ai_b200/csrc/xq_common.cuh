// xq_common.cuh -- shared host/device plumbing of libxq_b200 (error handling, launch counter,
// the shared-memory board accessor used by the thread-per-board kernels).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/xq.h"
#include "xq_rules.cuh"

namespace xq {

// ---- error plumbing: no exception crosses the C ABI ------------------------------------------
std::string& last_error();
int fail(int code, const char* fmt, ...);
extern unsigned long long g_launches;   // kernels launched by this library (xq_launch_count)

#define XQ_CUDA(call)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return ::xq::fail(XQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

#define XQ_LAUNCH_CHECK()                                                                      \
    do {                                                                                       \
        ++::xq::g_launches;                                                                    \
        cudaError_t e_ = cudaGetLastError();                                                   \
        if (e_ != cudaSuccess)                                                                 \
            return ::xq::fail(XQ_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ---- cross-module accessors (handles are opaque outside their own translation unit) ------------
struct EnvInfo {
    int64_t n; int device; uint64_t seed, env_id0; cudaStream_t stream; xq_env_rec* d_envs; xq_env_stats* d_stats;
    xq_game_event* d_events; unsigned long long* d_event_count; int64_t event_cap; uint32_t event_ply;     // finished-game ring (optional)
    uint8_t* d_nonstd; bool maybe_nonstd;      // per-env flags of the team kernels (board left to the generic kernel); boards were injected
};
int env_info(xq_env_t h, EnvInfo* out);
void env_advance_event_ply(xq_env_t h, uint32_t plies);   // the collector applied `plies` more plies
void** env_scratch_slot(xq_env_t h, void (*free_fn)(void*));   // the env handle's slot for the collector's scratch; free_fn runs when the handle is destroyed
// what the example buffer (xq_examples.cu) reads of a search (xq_search.cu): the root rows of its slab
struct SearchRoots {
    int64_t n; int cap;              // node j of tree t at g = t * cap + j; edge k of node g at g * 128 + k
    const xq_env_rec* rec; const uint8_t *nedges, *expanded; const int32_t* N; const float* W; const int16_t* act;
};
// the roots of search s for the caller fn, which records them for the envs of `env`: the search must be on `env`, reset, and have no
// selection pending
int search_roots(xq_search_t s, xq_env_t env, const char* fn, SearchRoots* out);
// xq_examples_record_gumbel_device: the call checks of a begun Gumbel search on env `env`, its roots, and the improved-policy weights of
// every root ([n][128], edge k at t * 128 + k) launched on the env's stream
int gumbel_weights(xq_gumbel_t g, xq_env_t env, SearchRoots* roots, const uint32_t** w);
// the same two for a reader of a search on any env handle of `device` (XQ_ERR_INVALID on another device), with the same call-order
// checks; the weights are launched on `stream`, the reader's
int search_roots_on(xq_search_t s, int device, const char* fn, SearchRoots* out);
int gumbel_weights_on(xq_gumbel_t g, int device, cudaStream_t stream, const char* fn, SearchRoots* roots, const uint32_t** w);
void env_boards_injected(xq_env_t h);      // boards were written from outside the env's own calls (xq_env_set_boards' after-effect)

// ---- host helpers of the C ABI -----------------------------------------------------------------
inline unsigned grid_of(int64_t n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }
inline bool valid_view(int view) { return view == XQ_VIEW_ABSOLUTE || view == XQ_VIEW_SIDE_TO_MOVE; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// A handle's device slab, carved into arrays that each start on a 256-byte boundary.  A handle lays its slab out in one function, run
// first with base nullptr to count the bytes and then on the allocation to set its pointers, so the size and the offsets agree.
struct Slab {
    char* base;
    size_t bytes = 0;
    template <class T> T* take(size_t count) {
        T* p = reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(base) + bytes);
        bytes += (sizeof(T) * count + 255) & ~(size_t)255;
        return p;
    }
};

// ---- device helpers ---------------------------------------------------------------------------
#if defined(__CUDACC__)
// One board per thread in shared memory, word-interleaved: word w of thread t lives at
// smem[w*blockDim.x + t], i.e. always in bank (t & 31): any mix of squares across the lanes
// of a warp is bank-conflict free.
struct SmemBoard {
    uint32_t* base;   // &smem[threadIdx.x]
    int stride;       // blockDim.x
    __device__ __forceinline__ int get(int s) const { return (base[(s >> 3) * stride] >> ((s & 7) * 4)) & 15; }
    __device__ __forceinline__ void set(int s, int code) {
        uint32_t& w = base[(s >> 3) * stride];
        const int sh = (s & 7) * 4;
        w = (w & ~(15u << sh)) | ((uint32_t)code << sh);
    }
    __device__ __forceinline__ void load(const xq_env_rec* rec) {
        const uint4* p = reinterpret_cast<const uint4*>(rec);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const uint4 v = p[i];
            base[(4 * i + 0) * stride] = v.x; base[(4 * i + 1) * stride] = v.y;
            base[(4 * i + 2) * stride] = v.z; base[(4 * i + 3) * stride] = v.w;
        }
    }
    __device__ __forceinline__ void store(xq_env_rec* rec) const {
        uint4* p = reinterpret_cast<uint4*>(rec);
#pragma unroll
        for (int i = 0; i < 3; ++i)
            p[i] = make_uint4(base[(4 * i + 0) * stride], base[(4 * i + 1) * stride], base[(4 * i + 2) * stride],
                              base[(4 * i + 3) * stride]);
    }
};

// The opening position as 12 packed words (ChessBoard::initializeBoard, src/chessboard.cpp:8-29):
// row 0 = R,H,E,A,G,A,E,H,R (codes 5,4,3,2,1,2,3,4,5), cannons (2,1),(2,7), soldiers row 3 even cols;
// Black mirrored on rows 9,7,6 with codes +7.
static __constant__ uint32_t kOpening[12] = {0x43212345u, 0x00000005u, 0x00006000u, 0x70707060u, 0x00007070u, 0x00000000u,
                                            0x0E000000u, 0x0E0E0E0Eu, 0x0D00000Du, 0x00000000u, 0xA989ABC0u, 0x000000CBu};
#endif

}  // namespace xq
