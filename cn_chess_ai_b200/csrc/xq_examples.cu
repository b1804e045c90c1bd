// xq_examples.cu -- device-resident self-play example buffer for policy/value training (include/xq.h: xq_examples_*): per move the
// searched roots' records and sparse visit counts, per finished game the result, per training step a sampled batch of observations, policy
// and value targets and legal masks.  No call synchronises with the host except info / get.
//
// Layout (one slab): the ring of `capacity` examples (xq_example, 864 B), the staging area of max_game_examples examples per env (env e's
// example p at e * max_game_examples + p), per env the staged count, the game count and two commit scratch words, and the counters
// (total committed, dropped, stale, and the base / count of the last commit).  The ring head is total % capacity.
// examples_record_kernel: one warp per tree, as search_root_kernel reads a root: the lanes compare the root record with the env's, read the
//   root's act / N / W rows coalesced, sum q in list order with s_add / s_div exactly as search_root_kernel, build the example in shared
//   memory and store it with 16-byte stores.
// examples_scan_kernel: one CTA; each thread sums the counts of a contiguous segment of envs, the segment sums are scanned across the CTA
//   (warp shuffles, then the 32 warp totals), and each thread writes the commit numbers of its envs in env order (ex_commit_offsets).
// examples_commit_kernel: persistent warps over the commit numbers in contiguous chunks; a warp finds the env of its first number by
//   binary search over the offsets, moves to the next env at its end, and copies one 864-byte example per step with z and game stamped.
// examples_sample_kernel: one CTA per sample: the draw, the policy row and the packed mask built in shared memory and streamed out with
//   16-byte (policy) and 8-byte (mask) stores, the record gathered for observe_kernel (launch_observe, xq_policy.cu).
#include <stddef.h>

#include <algorithm>
#include <new>
#include <vector>

#include "xq_common.cuh"
#include "xq_env_dev.cuh"
#include "xq_examples.cuh"

static_assert(sizeof(xq_example) == xq::kExampleBytes && sizeof(xq_example) % 32 == 0, "include/xq.h documents 864 B");
static_assert(offsetof(xq_example, game) == 72 && offsetof(xq_example, z) == 80 && offsetof(xq_example, action) == 96 &&
              offsetof(xq_example, visits) == 352, "examples_commit_kernel stamps game in word 4 and z in word 5");

namespace xq {

cudaError_t launch_observe(const xq_env_rec* recs, int64_t n, void* planes, int dtype, int view, int32_t* aux, cudaStream_t stream);

constexpr int kRecWarps = 4;          // trees per CTA of the record kernel
constexpr int kScanThreads = 1024;    // the one CTA of the commit scan
constexpr int kCopyThreads = 256;
constexpr int kSmpThreads = 256;

struct ExCounters {
    unsigned long long total, dropped, stale;       // committed since create, counted since create
    long long commit_base, commit_count;            // the last end_games: commit number of its first example, examples committed
};

struct ExDev {
    int64_t n, capacity; int maxg;
    xq_example *ring, *staging;
    uint32_t *staged, *games, *game_at;             // per env: staged examples, ended games, the game number of the last commit
    int64_t* off;                                    // per env: commit number of its first example in the last commit
    ExCounters* ctr;
};

// WEIGHTS: the visits field takes the Gumbel improved-policy weights wts[t * 128 + k] instead of N (xq_examples_record_gumbel_device)
template <bool WEIGHTS>
__global__ void __launch_bounds__(32 * kRecWarps) examples_record_kernel(ExDev b, SearchRoots r, const xq_env_rec* __restrict__ envs,
                                                                        const uint8_t* __restrict__ mask, uint64_t env_id0,
                                                                        const uint32_t* __restrict__ wts) {
    __shared__ __align__(16) xq_example s_ex[kRecWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * kRecWarps + warp;
    if (t >= b.n || (mask && !mask[t])) return;
    const int64_t g = t * r.cap, eb = g * kSearchEdges;
    xq_example& x = s_ex[warp];
    // 1. the root is the env's current board, all 64 bytes
    if (root_stale_warp(r.rec + g, envs + t, lane, reinterpret_cast<uint4*>(&x.rec))) {
        if (lane == 0) atomicAdd(&b.ctr->stale, 1ull);
        return;
    }
    const uint32_t slot = b.staged[t];
    if (slot >= (uint32_t)b.maxg) {
        if (lane == 0) atomicAdd(&b.ctr->dropped, 1ull);
        return;
    }
    // 2. the edges, coalesced; q summed in list order as search_root_kernel sums it
    const int ne = r.expanded[g] ? r.nedges[g] : 0;
    float w[kSearchEdges / 32];
    uint32_t tot = 0, sn = 0;           // sum of visits[], and sum of N for q (the same sum unless WEIGHTS)
#pragma unroll
    for (int i = 0; i < kSearchEdges / 32; ++i) {
        const int k = lane + 32 * i;
        const bool live = k < ne;
        const uint32_t nk = live ? (uint32_t)r.N[eb + k] : 0u;
        const uint32_t v = WEIGHTS ? (live ? wts[t * kSearchEdges + k] : 0u) : nk;
        w[i] = live ? r.W[eb + k] : 0.f;
        x.action[k] = live ? r.act[eb + k] : (int16_t)-1;
        x.visits[k] = v;
        tot += v;
        if (WEIGHTS) sn += nk;
    }
    tot = __reduce_add_sync(0xFFFFFFFFu, tot);
    if (WEIGHTS) sn = __reduce_add_sync(0xFFFFFFFFu, sn);
    const uint32_t qn = WEIGHTS ? sn : tot;
    float sw = 0.f;
#pragma unroll
    for (int i = 0; i < kSearchEdges / 32; ++i) {
        if (32 * i >= ne) break;
        for (int j = 0; j < 32; ++j) {
            const float v = __shfl_sync(0xFFFFFFFFu, w[i], j);
            if (32 * i + j < ne) sw = s_add(sw, v);
        }
    }
    if (lane == 0) {
        x.env = env_id0 + (uint64_t)t; x.game = 0; x.ply = (uint16_t)slot; x.n_edges = (uint8_t)ne; x.reserved0 = 0;
        x.z = 0.f; x.q = qn > 0 ? s_div(sw, (float)(int)qn) : NAN; x.total_visits = tot; x.reserved1 = 0;
        b.staged[t] = slot + 1;
    }
    __syncwarp();
    // 3. the example, 54 16-byte stores
    uint4* dst = reinterpret_cast<uint4*>(b.staging + t * b.maxg + slot);
    const uint4* src = reinterpret_cast<const uint4*>(&x);
    for (int c = lane; c < kExampleVecs; c += 32) dst[c] = src[c];
}

__global__ void __launch_bounds__(kScanThreads) examples_scan_kernel(ExDev b, const uint8_t* __restrict__ ended) {
    __shared__ long long s_warp[kScanThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int64_t lo, hi;
    ex_segment(b.n, kScanThreads, tid, lo, hi);
    long long sum = 0;
    for (int64_t e = lo; e < hi; ++e) sum += ex_count(ended[e], b.staged[e]);
    long long incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        long long v = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += y;
        }
        s_warp[lane] = v;
    }
    __syncthreads();
    const long long base = (long long)b.ctr->total;
    long long run = base + (warp ? s_warp[warp - 1] : 0) + incl - sum;
    for (int64_t e = lo; e < hi; ++e) {
        const uint8_t end = ended[e];
        b.off[e] = run;
        run += ex_count(end, b.staged[e]);
        if (end) { b.game_at[e] = b.games[e]; b.games[e] += 1; b.staged[e] = 0; }
    }
    __syncthreads();                                  // every thread has read the old total
    if (tid == 0) {
        const long long c = s_warp[kScanThreads / 32 - 1];
        b.ctr->commit_base = base; b.ctr->commit_count = c;
        b.ctr->total = (unsigned long long)(base + c);
    }
}

__global__ void __launch_bounds__(kCopyThreads) examples_commit_kernel(ExDev b, const float* __restrict__ result) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * kCopyThreads + threadIdx.x) >> 5, warps = ((int64_t)gridDim.x * kCopyThreads) >> 5;
    const int64_t base = b.ctr->commit_base, cnt = b.ctr->commit_count;
    const int64_t first = cnt > b.capacity ? cnt - b.capacity : 0;      // the older ones would be overwritten within this commit
    const int64_t per = (cnt - first + warps - 1) / warps;
    const int64_t i0 = first + warp * per, i1 = min(cnt, i0 + per);
    int64_t e = -1, end = 0;
    uint32_t game = 0;
    float z_red = 0.f;
    for (int64_t i = i0; i < i1; ++i) {
        const int64_t pos = base + i;
        if (pos >= end) {
            e = ex_find_env(b.off, b.n, pos);
            end = e + 1 < b.n ? b.off[e + 1] : base + cnt;
            game = b.game_at[e];
            z_red = result[e];
        }
        const uint4* src = reinterpret_cast<const uint4*>(b.staging + e * b.maxg + (pos - b.off[e]));
        uint4* dst = reinterpret_cast<uint4*>(b.ring + pos % b.capacity);
        uint4 v = src[lane];
        const int player = (int)((__shfl_sync(0xFFFFFFFFu, v.x, 3) >> 16) & 0xFFu);
        if (lane == 4) v.z = game;
        if (lane == 5) v.x = __float_as_uint(ex_z(z_red, player));
        dst[lane] = v;
        if (lane < kExampleVecs - 32) dst[32 + lane] = src[32 + lane];
    }
}

__global__ void __launch_bounds__(256) examples_discard_kernel(ExDev b, const uint8_t* __restrict__ mask) {
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e < b.n && (!mask || mask[e])) b.staged[e] = 0;
}

__global__ void __launch_bounds__(kSmpThreads) examples_sample_kernel(ExDev b, uint64_t seed, uint32_t counter, int view, xq_env_rec* __restrict__ recs,
                                                                    float* __restrict__ policy, float* __restrict__ value, float* __restrict__ q,
                                                                    uint32_t* __restrict__ mask, int64_t* __restrict__ index) {
    __shared__ __align__(16) float s_p[XQ_POLICY_ACTIONS];
    __shared__ __align__(16) uint32_t s_m[XQ_MASK_WORDS + 2];
    const int tid = threadIdx.x;
    const int64_t i = blockIdx.x;
    const int64_t total = (int64_t)b.ctr->total, size = total < b.capacity ? total : b.capacity;
    const int64_t idx = ex_sample_index(seed, i, counter, size);
    const xq_example* x = idx >= 0 ? b.ring + idx : nullptr;
    for (int c = tid; c < XQ_POLICY_ACTIONS / 4; c += kSmpThreads) reinterpret_cast<float4*>(s_p)[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid < XQ_MASK_WORDS + 2) s_m[tid] = 0u;
    if (tid < 4) reinterpret_cast<uint4*>(recs + i)[tid] = x ? reinterpret_cast<const uint4*>(&x->rec)[tid] : make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    if (x) {
        const int player = x->rec.player, ne = x->n_edges;
        const uint32_t tot = x->total_visits;
        for (int k = tid; k < ne; k += kSmpThreads) {
            const int pi = ex_view_index(x->action[k], player, view);
            s_p[pi] = ex_policy(x->visits[k], tot);
            atomicOr(&s_m[pi >> 5], 1u << (pi & 31));
        }
    }
    __syncthreads();
    float4* dp = reinterpret_cast<float4*>(policy + i * XQ_POLICY_ACTIONS);
    for (int c = tid; c < XQ_POLICY_ACTIONS / 4; c += kSmpThreads) dp[c] = reinterpret_cast<const float4*>(s_p)[c];
    if (mask && tid < XQ_MASK_WORDS / 2)
        reinterpret_cast<uint2*>(mask + i * XQ_MASK_WORDS)[tid] = reinterpret_cast<const uint2*>(s_m)[tid];
    if (tid == 0) {
        if (value) value[i] = x ? x->z : NAN;
        if (q) q[i] = x ? x->q : NAN;
        if (index) index[i] = idx;
    }
}

}  // namespace xq

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace xq;

struct xq_examples_s {
    xq_env_t env = nullptr;
    int device = 0, sms = 1;
    void* slab = nullptr;
    ExDev d{};
    xq_env_rec* recs = nullptr; int64_t recs_cap = 0;     // sampling scratch, grown as needed
};

namespace {

// the slab of an example buffer for n envs (Slab); false when it does not fit in memory
bool ex_slab(ExDev& d, void* base, int64_t n, int64_t capacity, int maxg, size_t* bytes) {
    const double ex = ((double)capacity + (double)n * (double)maxg) * kExampleBytes;
    if (ex > 9.0e18) return false;
    Slab b{static_cast<char*>(base)};
    d.ring = b.take<xq_example>((size_t)capacity);
    d.staging = b.take<xq_example>((size_t)n * (size_t)maxg);
    d.staged = b.take<uint32_t>(n); d.games = b.take<uint32_t>(n); d.game_at = b.take<uint32_t>(n);
    d.off = b.take<int64_t>(n);
    d.ctr = b.take<ExCounters>(1);
    *bytes = b.bytes;
    return true;
}
int enter(xq_examples_t b, EnvInfo* E, const char* fn) {
    if (!b) return fail(XQ_ERR_INVALID, "%s: null handle", fn);
    if (int rc = env_info(b->env, E)) return rc;
    XQ_CUDA(cudaSetDevice(E->device));
    return XQ_OK;
}
}  // namespace

extern "C" {

int xq_examples_bytes(int64_t n_envs, int64_t capacity, int max_game_examples, int64_t* bytes) {
    size_t s = 0;
    ExDev d;
    if (!bytes || n_envs < 1 || capacity < 1 || max_game_examples < 1 || max_game_examples > 65535 ||
        !ex_slab(d, nullptr, n_envs, capacity, max_game_examples, &s))
        return fail(XQ_ERR_INVALID, "xq_examples_bytes: bad arguments");
    *bytes = (int64_t)s;
    return XQ_OK;
}

int xq_examples_create(xq_env_t env, int64_t capacity, int max_game_examples, xq_examples_t* out) {
    if (!out || !env) return fail(XQ_ERR_INVALID, "xq_examples_create: null env or out");
    if (capacity < 1) return fail(XQ_ERR_INVALID, "xq_examples_create: capacity %lld (>= 1)", (long long)capacity);
    if (max_game_examples < 1 || max_game_examples > 65535)
        return fail(XQ_ERR_INVALID, "xq_examples_create: max_game_examples %d (1 .. 65535)", max_game_examples);
    EnvInfo E;
    if (int rc = env_info(env, &E)) return rc;
    size_t bytes = 0;
    ExDev d{};
    if (!ex_slab(d, nullptr, E.n, capacity, max_game_examples, &bytes)) return fail(XQ_ERR_NOMEM, "xq_examples_create: the buffer does not fit in memory");
    XQ_CUDA(cudaSetDevice(E.device));
    xq_examples_s* b = new (std::nothrow) xq_examples_s();
    if (!b) return fail(XQ_ERR_NOMEM, "xq_examples_create: out of host memory");
    b->env = env; b->device = E.device;
    cudaDeviceGetAttribute(&b->sms, cudaDevAttrMultiProcessorCount, E.device);
    if (b->sms < 1) b->sms = 1;
    if (cudaMalloc(&b->slab, bytes) != cudaSuccess) {
        cudaGetLastError();
        delete b;
        return fail(XQ_ERR_NOMEM, "xq_examples_create: %.2f GB of device memory not available", bytes / 1e9);
    }
    ex_slab(d, b->slab, E.n, capacity, max_game_examples, &bytes);
    d.n = E.n; d.capacity = capacity; d.maxg = max_game_examples;
    b->d = d;
    // the ring reads back as zeros before it is written; the counters and per-env words start at 0
    cudaError_t e = cudaMemsetAsync(b->slab, 0, bytes, E.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(E.stream);
    if (e != cudaSuccess) {
        cudaFree(b->slab);
        delete b;
        return fail(XQ_ERR_CUDA, "xq_examples_create: %s", cudaGetErrorString(e));
    }
    *out = b;
    return XQ_OK;
}

int xq_examples_destroy(xq_examples_t b) {
    if (!b) return XQ_OK;
    cudaSetDevice(b->device);
    cudaFree(b->slab);             // synchronises with the work still queued on the env's stream
    cudaFree(b->recs);
    delete b;
    return XQ_OK;
}

int xq_examples_record_device(xq_examples_t b, xq_search_t s, const uint8_t* mask_dev) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_record_device")) return rc;
    if (!s) return fail(XQ_ERR_INVALID, "xq_examples_record_device: null search");
    SearchRoots r;
    if (int rc = search_roots(s, b->env, "xq_examples_record_device", &r)) return rc;
    examples_record_kernel<false><<<grid_of(b->d.n, kRecWarps), 32 * kRecWarps, 0, E.stream>>>(b->d, r, E.d_envs, mask_dev, E.env_id0, nullptr);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_examples_record_gumbel_device(xq_examples_t b, xq_gumbel_t g, const uint8_t* mask_dev) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_record_gumbel_device")) return rc;
    if (!g) return fail(XQ_ERR_INVALID, "xq_examples_record_gumbel_device: null Gumbel state");
    SearchRoots r;
    const uint32_t* w = nullptr;
    if (int rc = gumbel_weights(g, b->env, &r, &w)) return rc;
    examples_record_kernel<true><<<grid_of(b->d.n, kRecWarps), 32 * kRecWarps, 0, E.stream>>>(b->d, r, E.d_envs, mask_dev, E.env_id0, w);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_examples_end_games_device(xq_examples_t b, const uint8_t* ended_dev, const float* result_dev) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_end_games_device")) return rc;
    if (!ended_dev || !result_dev) return fail(XQ_ERR_INVALID, "xq_examples_end_games_device: ended and result are required");
    examples_scan_kernel<<<1, kScanThreads, 0, E.stream>>>(b->d, ended_dev);
    XQ_LAUNCH_CHECK();
    const int64_t most = b->d.n * (int64_t)b->d.maxg;      // no more examples can be staged
    const int64_t grid = std::min<int64_t>(std::max<int64_t>(1, (most + kCopyThreads / 32 - 1) / (kCopyThreads / 32)), (int64_t)b->sms * 8);
    examples_commit_kernel<<<(unsigned)grid, kCopyThreads, 0, E.stream>>>(b->d, result_dev);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_examples_discard_device(xq_examples_t b, const uint8_t* mask_dev) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_discard_device")) return rc;
    examples_discard_kernel<<<grid_of(b->d.n, 256), 256, 0, E.stream>>>(b->d, mask_dev);
    XQ_LAUNCH_CHECK();
    return XQ_OK;
}

int xq_examples_sample_device(xq_examples_t b, int64_t batch, uint64_t seed, uint32_t counter, int view, void* planes_dev, int dtype,
                              float* policy_dev, float* value_dev, float* q_dev, uint32_t* mask_dev, int64_t* index_dev) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_sample_device")) return rc;
    if (batch <= 0 || batch > 0x7FFFFFFF) return fail(XQ_ERR_INVALID, "xq_examples_sample_device: batch %lld", (long long)batch);
    if (!valid_view(view)) return fail(XQ_ERR_INVALID, "xq_examples_sample_device: view %d", view);
    if (dtype < XQ_DTYPE_F32 || dtype > XQ_DTYPE_U8) return fail(XQ_ERR_INVALID, "xq_examples_sample_device: dtype %d", dtype);
    if (!planes_dev || !policy_dev) return fail(XQ_ERR_INVALID, "xq_examples_sample_device: planes and policy are required");
    if (!aligned16(planes_dev) || !aligned16(policy_dev) || (reinterpret_cast<uintptr_t>(mask_dev) & 7u))
        return fail(XQ_ERR_INVALID, "xq_examples_sample_device: planes and policy must be 16-byte aligned, mask 8-byte aligned");
    if (batch > b->recs_cap) {      // grows on the env's stream; cudaFree waits for the work that used the old scratch
        cudaFree(b->recs); b->recs = nullptr; b->recs_cap = 0;
        XQ_CUDA(cudaMalloc(&b->recs, sizeof(xq_env_rec) * (size_t)batch));
        b->recs_cap = batch;
    }
    examples_sample_kernel<<<(unsigned)batch, kSmpThreads, 0, E.stream>>>(b->d, seed, counter, view, b->recs, policy_dev, value_dev, q_dev, mask_dev,
                                                                         index_dev);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(launch_observe(b->recs, batch, planes_dev, dtype, view, nullptr, E.stream));
    return XQ_OK;
}

int xq_examples_info(xq_examples_t b, int64_t* size, int64_t* capacity, int64_t* total_committed, int64_t* pending, int64_t* dropped,
                     int64_t* stale) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_info")) return rc;
    ExCounters c;
    std::vector<uint32_t> staged((size_t)b->d.n);
    XQ_CUDA(cudaMemcpyAsync(&c, b->d.ctr, sizeof(c), cudaMemcpyDeviceToHost, E.stream));
    XQ_CUDA(cudaMemcpyAsync(staged.data(), b->d.staged, 4 * staged.size(), cudaMemcpyDeviceToHost, E.stream));
    XQ_CUDA(cudaStreamSynchronize(E.stream));
    int64_t p = 0;
    for (uint32_t v : staged) p += v;
    const int64_t total = (int64_t)c.total;
    if (size) *size = total < b->d.capacity ? total : b->d.capacity;
    if (capacity) *capacity = b->d.capacity;
    if (total_committed) *total_committed = total;
    if (pending) *pending = p;
    if (dropped) *dropped = (int64_t)c.dropped;
    if (stale) *stale = (int64_t)c.stale;
    return XQ_OK;
}

int xq_examples_get(xq_examples_t b, int64_t first, int64_t n, xq_example* out_host) {
    EnvInfo E;
    if (int rc = enter(b, &E, "xq_examples_get")) return rc;
    if (!out_host || first < 0 || n < 0 || first + n > b->d.capacity) return fail(XQ_ERR_INVALID, "xq_examples_get: bad range");
    XQ_CUDA(cudaMemcpyAsync(out_host, b->d.ring + first, sizeof(xq_example) * (size_t)n, cudaMemcpyDeviceToHost, E.stream));
    XQ_CUDA(cudaStreamSynchronize(E.stream));
    return XQ_OK;
}

}  // extern "C"
