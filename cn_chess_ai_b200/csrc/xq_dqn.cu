// xq_dqn.cu -- DQN / NeuralNetwork with the reference's per-sample FP64 semantics, any layer sizes.
//
// Replaces src/dqn.cu:184-319 (the six one-thread-per-neuron kernels, each wrapped in
// cudaMalloc/H2D/launch/cudaDeviceSynchronize/D2H/cudaFree by NeuralNetwork::forward/backpropagate
// :199-260,:323-467) and src/dqn.cpp (selectAction, getQValues, backpropagate, train,
// updateTargetNetwork, saveModel/loadModel).  Here activations live in a persistent device
// workspace, launches are stream-ordered without host synchronisation, dot products are
// warp-per-neuron with coalesced weight rows, and one D2H copy ends a call.
// Numerics: FP64; results agree with the reference's kernels to ~1e-16 relative (different
// summation order); tests hold 1e-12 abs.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <random>

#include "xq_dqn_internal.cuh"

namespace xq {

// out[s][o] = tanh(z), z = b[o] + sum_i in[s][i] * W[o][i]   (forwardKernel, src/dqn.cu:184-195 / :275-286)
__global__ void __launch_bounds__(256) fwd_layer_f64(const double* __restrict__ W, const double* __restrict__ b,
                                                    const double* __restrict__ in, int64_t in_stride, double* __restrict__ out,
                                                    double* __restrict__ z, int64_t out_stride, int in_size, int out_size, int64_t n) {
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n * out_size) return;
    const int64_t s = warp / out_size;
    const int o = (int)(warp - s * out_size);
    const double* w = W + (size_t)o * in_size;
    const double* x = in + s * in_stride;
    double sum = 0.0;
    for (int i = lane; i < in_size; i += 32) sum += x[i] * w[i];
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, k);
    if (lane == 0) {
        sum += b[o];
        if (z) z[s * out_stride + o] = sum;
        out[s * out_stride + o] = tanh(sum);
    }
}

// delta[o] = (a[o] - t[o]) * (1 - tanh(z[o])^2)   (outputLayerDeltaKernel, src/dqn.cu:288-295)
__global__ void out_delta_f64(const double* __restrict__ a, const double* __restrict__ t, const double* __restrict__ z,
                              double* __restrict__ delta, int size) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= size) return;
    const double th = tanh(z[i]);
    delta[i] = (a[i] - t[i]) * (1.0 - th * th);
}

// hiddenLayerDeltaKernel exactly as the reference launches it (src/dqn.cu:297-308 via :406-423):
// "inputSize" = width of THIS layer, "outputSize" = width of the PREVIOUS layer, index i*outputSize+idx into
// the next layer's weights (SURVEY F7).  Only idx < width is consumed by the update; out-of-range reads of the
// reference (undefined there) contribute 0 here.
__global__ void hidden_delta_as_written_f64(const double* __restrict__ Wn, size_t wn_size, const double* __restrict__ dn, int dn_size,
                                            const double* __restrict__ z, double* __restrict__ delta, int width, int prev_width) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= width) return;
    double sum = 0.0;
    if (idx < prev_width)
        for (int i = 0; i < width; ++i) {
            const size_t wi = (size_t)i * prev_width + idx;
            if (wi < wn_size && i < dn_size) sum += Wn[wi] * dn[i];
        }
    const double th = tanh(z[idx]);
    delta[idx] = idx < prev_width ? sum * (1.0 - th * th) : 0.0;
}

// corrected hidden delta: pre[j] = sum_o W_next[o][j] * delta_next[o]; one CTA = 32 rows of W_next x all columns
__global__ void __launch_bounds__(256) hidden_delta_partial_f64(const double* __restrict__ Wn, const double* __restrict__ dn,
                                                               double* __restrict__ pre, int width, int next_width) {
    const int o0 = blockIdx.x * 32;
    for (int j = threadIdx.x; j < width; j += blockDim.x) {
        double sum = 0.0;
        for (int o = o0; o < min(o0 + 32, next_width); ++o) sum += Wn[(size_t)o * width + j] * dn[o];
        atomicAdd(&pre[j], sum);
    }
}
__global__ void hidden_delta_finish_f64(const double* __restrict__ pre, const double* __restrict__ z, double* __restrict__ delta, int width) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= width) return;
    const double th = tanh(z[j]);
    delta[j] = pre[j] * (1.0 - th * th);
}

// W[o][i] -= lr*delta[o]*a[i]; b[o] -= lr*delta[o]   (updateWeightsBiasesKernel, src/dqn.cu:310-319)
__global__ void __launch_bounds__(256) update_f64(double* __restrict__ W, double* __restrict__ b, const double* __restrict__ a,
                                                 const double* __restrict__ delta, double lr, int in_size, int out_size) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)in_size * out_size) return;
    const int o = (int)(e / in_size), i = (int)(e - (int64_t)o * in_size);
    const double g = lr * delta[o];
    W[e] -= g * a[i];
    if (i == 0) b[o] -= g;
}

// max over a vector (std::max_element, src/chessai.cpp:127 / src/dqn.cpp:167), single CTA
__global__ void __launch_bounds__(256) vec_max_f64(const double* __restrict__ v, int n, double* __restrict__ out) {
    __shared__ double s[8];
    double m = -INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) m = fmax(m, v[i]);
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) m = fmax(m, __shfl_xor_sync(0xFFFFFFFFu, m, k));
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) { for (int k = 1; k < 8; ++k) m = fmax(m, s[k]); *out = m; }
}
// target = q; target[a] = done ? r : r + gamma * max_next   (src/chessai.cpp:122-128)
__global__ void td_target_f64(double* __restrict__ target, int a, double reward, int done, double gamma, const double* __restrict__ max_next) {
    if (threadIdx.x == 0 && blockIdx.x == 0) target[a] = done ? reward : reward + gamma * (*max_next);
}
// greedy branch of DQN::selectAction (src/dqn.cpp:39-54): FIRST action maximising q[action.to] (strict >, from -inf)
__global__ void __launch_bounds__(128) select_greedy_f64(const double* __restrict__ q, int q_size, const uint16_t* __restrict__ actions, int n,
                                                        int* __restrict__ out) {
    __shared__ double sv[128];
    __shared__ int si[128];
    double best = -INFINITY;
    int bi = 0x7FFFFFFF;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int to = XQ_ACTION_TO(actions[i]);
        if (to >= q_size) continue;                              // "Action.to index out of bounds" is skipped (:43-46)
        const double v = q[to];
        if (v > best) { best = v; bi = i; }
    }
    sv[threadIdx.x] = best; si[threadIdx.x] = bi;
    __syncthreads();
    if (threadIdx.x == 0) {
        double b = -INFINITY;
        int idx = 0x7FFFFFFF;
        for (int t = 0; t < 128; ++t)
            if (si[t] != 0x7FFFFFFF && (sv[t] > b || (sv[t] == b && si[t] < idx))) { b = sv[t]; idx = si[t]; }
        *out = idx == 0x7FFFFFFF ? 0 : idx;                      // bestAction = validActions[0] when nothing beats -inf (:40)
    }
}


static int dqn_reserve(xq_dqn_s* h, int64_t n) {
    if (n <= h->cap) return XQ_OK;
    cudaFree(h->d_act); cudaFree(h->d_z); cudaFree(h->d_target);
    h->d_act = h->d_z = h->d_target = nullptr; h->cap = 0;
    XQ_CUDA(cudaMalloc(&h->d_act, sizeof(double) * h->act_stride * n));
    XQ_CUDA(cudaMalloc(&h->d_z, sizeof(double) * h->act_stride * n));
    XQ_CUDA(cudaMalloc(&h->d_target, sizeof(double) * (size_t)h->layers.back() * n));
    h->cap = n;
    return XQ_OK;
}

// forward of n samples already in d_act (layer 0 slice); act/z layout: sample-major, per sample the layers concatenated
static int dqn_forward_dev(xq_dqn_s* h, const double* W, const double* B, int64_t n, bool keep_z) {
    size_t ofs = 0;
    for (int l = 0; l < h->L; ++l) {
        const int in = h->layers[l], on = h->layers[l + 1];
        fwd_layer_f64<<<grid_of(n * on * 32, 256), 256, 0, h->stream>>>(W + h->wofs[l], B + h->bofs[l], h->d_act + ofs, (int64_t)h->act_stride,
                                                                       h->d_act + ofs + in, keep_z ? h->d_z + ofs + in : nullptr,
                                                                       (int64_t)h->act_stride, in, on, n);
        XQ_LAUNCH_CHECK();
        ofs += in;
    }
    return XQ_OK;
}

// one reference backpropagate() on the sample in slot 0 of the workspace, target in d_target (device)
static int dqn_backprop_dev(xq_dqn_s* h, double lr) {
    if (int rc = dqn_forward_dev(h, h->d_w, h->d_b, 1, true)) return rc;
    std::vector<size_t> aofs(h->L + 1);
    size_t o = 0;
    for (int l = 0; l <= h->L; ++l) { aofs[l] = o; o += h->layers[l]; }
    const int Lo = h->L - 1;
    double* delta = h->d_delta;   // deltas use the same per-layer offsets as activations
    out_delta_f64<<<grid_of(h->layers[Lo + 1], 256), 256, 0, h->stream>>>(h->d_act + aofs[Lo + 1], h->d_target, h->d_z + aofs[Lo + 1],
                                                                         delta + aofs[Lo + 1], h->layers[Lo + 1]);
    XQ_LAUNCH_CHECK();
    for (int l = Lo - 1; l >= 0; --l) {
        const int width = h->layers[l + 1], prev = h->layers[l], next = h->layers[l + 2];
        const double* Wn = h->d_w + h->wofs[l + 1];
        if (h->mode == XQ_DQN_AS_WRITTEN) {
            hidden_delta_as_written_f64<<<grid_of(width, 128), 128, 0, h->stream>>>(Wn, (size_t)width * next, delta + aofs[l + 2], next,
                                                                                   h->d_z + aofs[l + 1], delta + aofs[l + 1], width, prev);
            XQ_LAUNCH_CHECK();
        } else {
            XQ_CUDA(cudaMemsetAsync(h->d_tmp, 0, sizeof(double) * width, h->stream));
            hidden_delta_partial_f64<<<grid_of(next, 32), 256, 0, h->stream>>>(Wn, delta + aofs[l + 2], h->d_tmp, width, next);
            XQ_LAUNCH_CHECK();
            hidden_delta_finish_f64<<<grid_of(width, 128), 128, 0, h->stream>>>(h->d_tmp, h->d_z + aofs[l + 1], delta + aofs[l + 1], width);
            XQ_LAUNCH_CHECK();
        }
    }
    for (int l = 0; l < h->L; ++l) {   // every delta was taken from the pre-update weights (src/dqn.cu:429-447)
        const int in = h->layers[l], on = h->layers[l + 1];
        update_f64<<<grid_of((int64_t)in * on, 256), 256, 0, h->stream>>>(h->d_w + h->wofs[l], h->d_b + h->bofs[l], h->d_act + aofs[l],
                                                                         delta + aofs[l + 1], lr, in, on);
        XQ_LAUNCH_CHECK();
    }
    h->fast_current = false;
    return XQ_OK;
}

}  // namespace xq

using namespace xq;

#define XQ_DQN_ENTER(h)                                                      \
    if (!(h)) return fail(XQ_ERR_INVALID, "%s: null handle", __func__);      \
    XQ_CUDA(cudaSetDevice((h)->device))

extern "C" {

int xq_dqn_destroy(xq_dqn_t h) {
    if (!h) return XQ_OK;
    cudaSetDevice(h->device);
    dqn_fast_destroy(h);
    if (h->act_ev) cudaEventDestroy(h->act_ev);
    cudaFree(h->d_w); cudaFree(h->d_b); cudaFree(h->d_tw); cudaFree(h->d_tb); cudaFree(h->d_act); cudaFree(h->d_z);
    cudaFree(h->d_delta); cudaFree(h->d_target); cudaFree(h->d_tmp); cudaFree(h->d_sel); cudaFree(h->d_actions); cudaFree(h->d_scalar);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return XQ_OK;
}

int xq_dqn_create(const int32_t* layer_sizes, int n_layers, double lr, double gamma, int device, uint64_t seed, int mode, xq_dqn_t* out) {
    if (!out || !layer_sizes) return fail(XQ_ERR_INVALID, "xq_dqn_create: null pointer");
    // std::invalid_argument of NeuralNetwork::NeuralNetwork (src/dqn.cu:17-19)
    if (n_layers < 2) return fail(XQ_ERR_INVALID, "NeuralNetwork must have at least two layers (input and output).");
    for (int i = 0; i < n_layers; ++i) if (layer_sizes[i] <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_create: layer %d has size %d", i, layer_sizes[i]);
    if (mode != XQ_DQN_AS_WRITTEN && mode != XQ_DQN_CORRECTED) return fail(XQ_ERR_INVALID, "xq_dqn_create: unknown mode %d", mode);
    int ndev = 0;
    XQ_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(XQ_ERR_INVALID, "xq_dqn_create: device %d out of range (%d devices)", device, ndev);
    XQ_CUDA(cudaSetDevice(device));
    xq_dqn_s* h = new (std::nothrow) xq_dqn_s();
    if (!h) return fail(XQ_ERR_NOMEM, "xq_dqn_create: out of host memory");
    h->layers.assign(layer_sizes, layer_sizes + n_layers);
    h->L = n_layers - 1; h->lr = lr; h->gamma = gamma; h->device = device; h->mode = mode; h->seed = seed;
    h->wofs.resize(h->L); h->bofs.resize(h->L);
    size_t maxw = 0;
    for (int l = 0; l < h->L; ++l) {
        h->wofs[l] = h->nw; h->bofs[l] = h->nb;
        h->nw += (size_t)h->layers[l] * h->layers[l + 1]; h->nb += h->layers[l + 1];
    }
    for (int v : h->layers) { h->act_stride += v; if ((size_t)v > maxw) maxw = v; }
    // initializeHostWeightsAndBiases (src/dqn.cu:96-123) with a caller-supplied seed instead of random_device
    std::vector<double> w(h->nw), b(h->nb, 0.0);
    std::mt19937 gen((uint32_t)(seed ^ (seed >> 32)));
    std::uniform_real_distribution<> dis(-0.05, 0.05);
    for (auto& v : w) v = dis(gen);
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    h->own_stream = e == cudaSuccess;
    if (e == cudaSuccess) e = cudaMalloc(&h->d_w, sizeof(double) * h->nw);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_b, sizeof(double) * h->nb);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_tw, sizeof(double) * h->nw);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_tb, sizeof(double) * h->nb);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_delta, sizeof(double) * h->act_stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_tmp, sizeof(double) * (maxw + 8));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_sel, sizeof(int) * 4);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_scalar, sizeof(double) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_actions, sizeof(uint16_t) * 1024);
    if (e != cudaSuccess) { xq_dqn_destroy(h); return fail(XQ_ERR_CUDA, "xq_dqn_create: %s", cudaGetErrorString(e)); }
    if (int rc = dqn_reserve(h, 2)) { xq_dqn_destroy(h); return rc; }
    *out = h;
    return xq_dqn_set_params(h, w.data(), b.data());
}

int xq_dqn_set_stream(xq_dqn_t h, void* s) {
    XQ_DQN_ENTER(h);
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    if (h->own_stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    h->stream = (cudaStream_t)s;
    return XQ_OK;
}
int xq_dqn_sync(xq_dqn_t h) { XQ_DQN_ENTER(h); XQ_CUDA(cudaStreamSynchronize(h->stream)); return XQ_OK; }

int xq_dqn_num_params(xq_dqn_t h, int64_t* nw, int64_t* nb) {
    if (!h) return fail(XQ_ERR_INVALID, "xq_dqn_num_params: null handle");
    if (nw) *nw = (int64_t)h->nw;
    if (nb) *nb = (int64_t)h->nb;
    return XQ_OK;
}

int xq_dqn_set_params(xq_dqn_t h, const double* w, const double* b) {
    XQ_DQN_ENTER(h);
    if (!w || !b) return fail(XQ_ERR_INVALID, "xq_dqn_set_params: null pointer");
    XQ_CUDA(cudaMemcpyAsync(h->d_w, w, sizeof(double) * h->nw, cudaMemcpyHostToDevice, h->stream));
    XQ_CUDA(cudaMemcpyAsync(h->d_b, b, sizeof(double) * h->nb, cudaMemcpyHostToDevice, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    h->f64_current = true; h->fast_current = false;
    return xq_dqn_sync_target(h);
}

int xq_dqn_get_params(xq_dqn_t h, double* w, double* b) {
    XQ_DQN_ENTER(h);
    if (int rc = dqn_ensure_f64(h)) return rc;
    if (w) XQ_CUDA(cudaMemcpyAsync(w, h->d_w, sizeof(double) * h->nw, cudaMemcpyDeviceToHost, h->stream));
    if (b) XQ_CUDA(cudaMemcpyAsync(b, h->d_b, sizeof(double) * h->nb, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_dqn_sync_target(xq_dqn_t h) {
    XQ_DQN_ENTER(h);
    if (int rc = dqn_ensure_f64(h)) return rc;
    XQ_CUDA(cudaMemcpyAsync(h->d_tw, h->d_w, sizeof(double) * h->nw, cudaMemcpyDeviceToDevice, h->stream));
    XQ_CUDA(cudaMemcpyAsync(h->d_tb, h->d_b, sizeof(double) * h->nb, cudaMemcpyDeviceToDevice, h->stream));
    dqn_target_changed(h);
    return XQ_OK;
}

int xq_dqn_forward(xq_dqn_t h, const double* states, int64_t n, double* q) {
    XQ_DQN_ENTER(h);
    if (!states || !q || n <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_forward: bad arguments");
    if (int rc = dqn_ensure_f64(h)) return rc;
    if (int rc = dqn_reserve(h, n)) return rc;
    const int in = h->layers[0], on = h->layers.back();
    XQ_CUDA(cudaMemcpy2DAsync(h->d_act, sizeof(double) * h->act_stride, states, sizeof(double) * in, sizeof(double) * in, (size_t)n,
                              cudaMemcpyHostToDevice, h->stream));
    if (int rc = dqn_forward_dev(h, h->d_w, h->d_b, n, false)) return rc;
    XQ_CUDA(cudaMemcpy2DAsync(q, sizeof(double) * on, h->d_act + (h->act_stride - on), sizeof(double) * h->act_stride, sizeof(double) * on,
                              (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_dqn_backprop(xq_dqn_t h, const double* states, const double* targets, int64_t n, double lr) {
    XQ_DQN_ENTER(h);
    if (!states || !targets || n <= 0) return fail(XQ_ERR_INVALID, "xq_dqn_backprop: bad arguments");
    if (int rc = dqn_ensure_f64(h)) return rc;
    const int in = h->layers[0], on = h->layers.back();
    for (int64_t s = 0; s < n; ++s) {   // n sequential SGD steps, each one reference backpropagate() call
        XQ_CUDA(cudaMemcpyAsync(h->d_act, states + s * in, sizeof(double) * in, cudaMemcpyHostToDevice, h->stream));
        XQ_CUDA(cudaMemcpyAsync(h->d_target, targets + s * on, sizeof(double) * on, cudaMemcpyHostToDevice, h->stream));
        if (int rc = dqn_backprop_dev(h, lr)) return rc;
    }
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_dqn_select_action(xq_dqn_t h, const double* state, double eps, const xq_action* actions, int n_actions, uint32_t coin31,
                         uint32_t idx31, int* index_out) {
    XQ_DQN_ENTER(h);
    if (!state || !actions || !index_out) return fail(XQ_ERR_INVALID, "xq_dqn_select_action: null pointer");
    if (n_actions <= 0) return fail(XQ_ERR_INVALID, "No valid actions available.");              // std::runtime_error, src/dqn.cpp:26-28
    if (n_actions > 1024) return fail(XQ_ERR_INVALID, "xq_dqn_select_action: at most 1024 actions");
    if ((double)coin31 / 2147483647.0 < eps) { *index_out = (int)(idx31 % (uint32_t)n_actions); return XQ_OK; }   // :30-34
    if (int rc = dqn_ensure_f64(h)) return rc;
    const int in = h->layers[0], on = h->layers.back();
    XQ_CUDA(cudaMemcpyAsync(h->d_act, state, sizeof(double) * in, cudaMemcpyHostToDevice, h->stream));
    XQ_CUDA(cudaMemcpyAsync(h->d_actions, actions, sizeof(uint16_t) * n_actions, cudaMemcpyHostToDevice, h->stream));
    if (int rc = dqn_forward_dev(h, h->d_w, h->d_b, 1, false)) return rc;
    select_greedy_f64<<<1, 128, 0, h->stream>>>(h->d_act + (h->act_stride - on), on, h->d_actions, n_actions, h->d_sel);
    XQ_LAUNCH_CHECK();
    XQ_CUDA(cudaMemcpyAsync(index_out, h->d_sel, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

int xq_dqn_train(xq_dqn_t h, const double* state, int action, double reward, const double* next_state, int done, int use_target_net,
                 double lr) {
    XQ_DQN_ENTER(h);
    const int in = h->layers[0], on = h->layers.back();
    if (!state || (!done && !next_state)) return fail(XQ_ERR_INVALID, "xq_dqn_train: null state");
    if (action < 0 || action >= on) return fail(XQ_ERR_INVALID, "xq_dqn_train: action %d outside [0,%d)", action, on);
    if (int rc = dqn_ensure_f64(h)) return rc;
    if (lr <= 0) lr = h->lr;
    if (!done) {
        XQ_CUDA(cudaMemcpyAsync(h->d_act, next_state, sizeof(double) * in, cudaMemcpyHostToDevice, h->stream));
        if (int rc = dqn_forward_dev(h, use_target_net ? h->d_tw : h->d_w, use_target_net ? h->d_tb : h->d_b, 1, false)) return rc;
        vec_max_f64<<<1, 256, 0, h->stream>>>(h->d_act + (h->act_stride - on), on, h->d_scalar);
        XQ_LAUNCH_CHECK();
    }
    XQ_CUDA(cudaMemcpyAsync(h->d_act, state, sizeof(double) * in, cudaMemcpyHostToDevice, h->stream));
    if (int rc = dqn_forward_dev(h, h->d_w, h->d_b, 1, false)) return rc;      // targetQ = getQValues(state)
    XQ_CUDA(cudaMemcpyAsync(h->d_target, h->d_act + (h->act_stride - on), sizeof(double) * on, cudaMemcpyDeviceToDevice, h->stream));
    td_target_f64<<<1, 32, 0, h->stream>>>(h->d_target, action, reward, done, h->gamma, h->d_scalar);
    XQ_LAUNCH_CHECK();
    if (int rc = dqn_backprop_dev(h, lr)) return rc;
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    return XQ_OK;
}

static void put_be(FILE* f, uint64_t v, int bytes) { for (int i = bytes - 1; i >= 0; --i) fputc((int)((v >> (8 * i)) & 0xFF), f); }
static bool get_be(FILE* f, uint64_t* v, int bytes) { *v = 0; for (int i = 0; i < bytes; ++i) { int c = fgetc(f); if (c == EOF) return false; *v = (*v << 8) | (uint64_t)c; } return true; }

int xq_dqn_save(xq_dqn_t h, const char* path) {
    XQ_DQN_ENTER(h);
    if (!path) return fail(XQ_ERR_INVALID, "xq_dqn_save: null path");
    std::vector<double> w(h->nw), b(h->nb);
    if (int rc = xq_dqn_get_params(h, w.data(), b.data())) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(XQ_ERR_IO, "Unable to open file for saving model.");                      // src/dqn.cpp:79-81
    bool ok = fwrite(w.data(), sizeof(double), w.size(), f) == w.size() && fwrite(b.data(), sizeof(double), b.size(), f) == b.size();
    put_be(f, (uint64_t)h->layers.size(), 8);                                                     // quint64, big-endian (QDataStream)
    for (int v : h->layers) put_be(f, (uint32_t)v, 4);                                            // int -> qint32, big-endian
    ok = ok && !ferror(f);
    fclose(f);
    return ok ? XQ_OK : fail(XQ_ERR_IO, "Error writing weights to model file.");
}

int xq_dqn_load(xq_dqn_t h, const char* path) {
    XQ_DQN_ENTER(h);
    if (!path) return fail(XQ_ERR_INVALID, "xq_dqn_load: null path");
    FILE* f = fopen(path, "rb");
    if (!f) return fail(XQ_ERR_IO, "Unable to open file for loading model.");                     // src/dqn.cpp:114-116
    std::vector<double> w(h->nw), b(h->nb);
    if (fread(w.data(), sizeof(double), w.size(), f) != w.size()) { fclose(f); return fail(XQ_ERR_IO, "Error reading weights from model file."); }
    if (fread(b.data(), sizeof(double), b.size(), f) != b.size()) { fclose(f); return fail(XQ_ERR_IO, "Error reading biases from model file."); }
    uint64_t nl = 0;
    bool ok = get_be(f, &nl, 8) && nl == h->layers.size();
    for (size_t i = 0; ok && i < h->layers.size(); ++i) { uint64_t v; ok = get_be(f, &v, 4) && (int32_t)v == h->layers[i]; }
    fclose(f);
    if (!ok) return fail(XQ_ERR_IO, "Layer sizes in the model file do not match the current network architecture.");   // :146-148
    // loadModel re-uploads the online network only (qNetwork->copyToDevice, :152-153); the target keeps its weights
    XQ_CUDA(cudaMemcpyAsync(h->d_w, w.data(), sizeof(double) * h->nw, cudaMemcpyHostToDevice, h->stream));
    XQ_CUDA(cudaMemcpyAsync(h->d_b, b.data(), sizeof(double) * h->nb, cudaMemcpyHostToDevice, h->stream));
    XQ_CUDA(cudaStreamSynchronize(h->stream));
    h->f64_current = true; h->fast_current = false;
    return XQ_OK;
}

}  // extern "C"
