// xq_dqn_internal.cuh -- the DQN handle shared by the FP64 reference-semantics path (xq_dqn.cu)
// and the batched BF16 tensor-core path (xq_dqn_fast.cu).
#pragma once
#include <cuda_bf16.h>

#include <vector>

#include "xq_common.cuh"

namespace xq { struct Fast; struct ActCarry; }

struct xq_dqn_s {
    std::vector<int> layers;          // layerSizes (include/dqn.h:77)
    int L = 0;                        // number of weight layers = layers.size()-1
    std::vector<size_t> wofs, bofs;   // weightOffsets / biasOffsets (src/dqn.cu:125-140)
    size_t nw = 0, nb = 0;
    double lr = 0.001, gamma = 0.99;  // include/chessai.h:48-49
    int device = 0, mode = XQ_DQN_AS_WRITTEN;
    uint64_t seed = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;

    // FP64 parameters: online + target (DQN::qNetwork / targetNetwork, include/dqn.h:112-113)
    double *d_w = nullptr, *d_b = nullptr, *d_tw = nullptr, *d_tb = nullptr;
    // FP64 scratch: activations / pre-activations / deltas for `cap` samples
    int64_t cap = 0;
    size_t act_stride = 0;            // sum of all layer sizes
    double *d_act = nullptr, *d_z = nullptr, *d_delta = nullptr, *d_target = nullptr, *d_tmp = nullptr;
    int* d_sel = nullptr;
    double* d_scalar = nullptr;
    uint16_t* d_actions = nullptr;

    // which copy of the parameters is current (the two numeric paths keep their own master copy)
    bool f64_current = true, fast_current = false;

    // ---- batched BF16 path, {1260,128,8100} only (xq_dqn_fast.cu) ----
    xq::Fast* fast = nullptr;
    // the acting state of the tensor-core path (carried layer-0 sums, h(s) operands) belongs to the network handle and is written on the
    // ENV's stream: collectors / xq_dqn_act calls that share this network are ordered one after the other across env handles and streams
    cudaEvent_t act_ev = nullptr;
    cudaStream_t act_stream = nullptr;
    bool act_pending = false;
};

namespace xq {
int dqn_ensure_f64(xq_dqn_s* h);      // refresh the FP64 parameters from the fast path's FP32 master if it is newer
void dqn_fast_destroy(xq_dqn_s* h);
void dqn_target_changed(xq_dqn_s* h);
struct FastWeights { const float *W0T, *b0, *W1, *b1; };
// bracket every use of the network's acting state on `stream`: enter waits for the previous user (if it ran on another stream), leave records
inline int dqn_act_enter(xq_dqn_s* h, cudaStream_t stream) {
    if (h->act_pending && h->act_stream != stream) XQ_CUDA(cudaStreamWaitEvent(stream, h->act_ev, 0));
    return XQ_OK;
}
inline int dqn_act_leave(xq_dqn_s* h, cudaStream_t stream) {
    if (!h->act_ev) XQ_CUDA(cudaEventCreateWithFlags(&h->act_ev, cudaEventDisableTiming));
    XQ_CUDA(cudaEventRecord(h->act_ev, stream));
    h->act_stream = stream; h->act_pending = true;
    return XQ_OK;
}
int dqn_fast_weights(xq_dqn_s* h, FastWeights* out);
// Q(s)[0..95] ([n][96] FP32 on the device) for n resident env records: the acting path of the self-play collector
// `carried`: skip the layer-0 kernel because the caller's act_team_kernel kept the per-env sums and h(s) current; `carry` receives what it needs to do so
int dqn_q90_device(xq_dqn_s* h, const xq_env_rec* envs_dev, int64_t n, float* q90_dev, cudaStream_t stream, bool carried = false, ActCarry* carry = nullptr);
// the contraction for part `part` of `n_parts` of a prepared, carried env range (multi-stream collector plies)
int dqn_q90_half(xq_dqn_s* h, int64_t n, int half, float* q90_dev, cudaStream_t stream, xq::ActCarry* carry, int64_t* off_out, int64_t* m_out);
// TD update on n uniform draws from a replay ring, resolved in place (no gather pass)
int dqn_td_update_sampled(xq_dqn_s* h, const void* ring, int64_t size, uint64_t seed, uint32_t counter, int64_t n, int use_target_net,
                          double lr, int apply);   // brings the FP32 copies up to date and returns them   // the FP64 target parameters were rewritten
// n_updates sequential target-net TD updates on replay draws, software-pipelined over two streams (same results as n_updates single calls)
int dqn_td_update_pipelined(xq_dqn_s* h, const void* ring, int64_t size, uint64_t seed, uint32_t counter0, int64_t n, int n_updates, double lr);
}
