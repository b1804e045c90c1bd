"""FP64 restatement of the Q(s)[0..95] the acting path computes (xq_dqn_act, xq_selfplay_collect: l0_act_kernel / the tail of the act
kernels for layer 0, q90_gemm_kernel for layer 1), vectorised over packed env records, and the error bound of the device result.

Q[o] = tanh(W1[o] . tanh(W0 x + b0) + b1[o]), o < 96, x = the one-hot state of ChessAI::getStateRepresentation (index square * 14 +
code - 1; code 15 is not a piece and selects nothing).  Parameters use the reference layout: w = [W0 (128 x 1260) | W1 (8100 x 128)],
each [out][in] row-major, b = [b0 (128) | b1 (8100)].  The layer-0 sum goes through a sparse one-hot matrix, so 65,536 envs cost a few
MB rather than the gigabytes of a dense [n, 1260] state.

Error bound (`bound`), per env and output o, for the device Q against this FP64 Q.  u = 2^-24 is the FP32 unit roundoff.
  Layer 0, per hidden unit j (dz_j):
    - the FP32 copies of W0 and b0: u x S_j, S_j = |b0_j| + sum of |W0[j, i]| over the selected inputs i;
    - the fixed-point table W0Q = rint(W0 * 2^k), k as act_quant_shift (k = 30 - e, 92 max |W0|, |b0| < 2^e): 2^-(k+1) per term,
      (occupied squares + 1) terms;
    - the int32 -> FP32 conversion of the sum: u x S_j.
  h_j = act_tanh(z_j) on the SFU: |error| <= TANH_ABS (ex2.approx and rcp.approx are good to ~2^-22 and ~2^-23 relative: ~2e-7,
  taken twice).  tanh is 1-Lipschitz, so dh_j = dz_j + TANH_ABS and |h_dev| <= H_j = min(1, |h_j| + dh_j).
  Layer 1: the device forms hi_h W_hi + lo_h W_hi + hi_h W_lo in BF16 with FP32 accumulation.  With h_dev = hi_h + lo_h + r_h and
  W = hi_W + lo_W + dW, z1_dev - h_dev . W = -(r_h . W) - ((hi_h + lo_h) . dW) - lo_h . lo_W + accumulation error, so
    - sum_j |W1[o, j]| dh_j                             the error of h;
    - 2^-17 sum_j H_j |W1[o, j]|                         the hi + lo split of h (|r_h| <= 2^-17 |h|: lo is rounded in a binade
                                                         at least 2^8 below h's);
    - sum_j H_j |dW[o, j]|                               the split of W1, computed exactly here (FP32 copy, BF16 hi, BF16 lo);
    - 2^-8 (1 + 2^-8) sum_j H_j |lo_W[o, j]|             the dropped lo_h lo_W product (|lo_h| <= 2^-8 |h|(1 + 2^-8));
    - 64 u sum_j H_j |W1[o, j]|                          FP32 accumulation: 24 MMAs (3 parts x 8 k-steps of 16) each round the
                                                         running sum once and add 16 products in a tree of depth 4: <= 28
                                                         roundings of at most 2 u (truncation) each of the running magnitude;
    - 2 u |b1[o]|                                        the FP32 copy of b1 and the bias add;
    - TANH_ABS                                           the output tanh, 1-Lipschitz like the rest.
  At the reference initialisation U(-0.05, 0.05) this bound stays below 2e-5 for every position (k = 27, about 1e-5 typical), and it
  grows with the weights: k follows max |W0|, |b0|, the split terms follow |h| |W1|."""
import numpy as np
import scipy.sparse as sp

N_IN, N_HID, N_Q = 1260, 128, 96
U32 = 2.0 ** -24
TANH_ABS = 2.0 ** -21


def codes(recs):
    """[n, 90] square codes of packed records"""
    sq = np.ascontiguousarray(recs["sq"], dtype=np.uint32)
    nib = (sq[:, :, None] >> (4 * np.arange(8, dtype=np.uint32))[None, None, :]) & np.uint32(15)
    return nib.reshape(len(recs), 96)[:, :90].astype(np.int64)


def onehot(recs):
    """sparse [n, 1260] state (getStateRepresentation) and the number of occupied squares per env"""
    c = codes(recs)
    live = (c > 0) & (c < 15)
    env, sq = np.nonzero(live)
    x = sp.csr_matrix((np.ones(len(env)), (env, sq * 14 + c[env, sq] - 1)), shape=(len(recs), N_IN))
    return x, live.sum(axis=1)


def layers(w, b):
    w = np.asarray(w, np.float64)
    b = np.asarray(b, np.float64)
    return w[:N_IN * N_HID].reshape(N_HID, N_IN), b[:N_HID], w[N_IN * N_HID:].reshape(-1, N_HID)[:N_Q], b[N_HID:N_HID + N_Q]


def forward(recs, w, b):
    """FP64 Q(s)[0..95] [n, 96] and h(s) [n, 128]"""
    W0, b0, W1, b1 = layers(w, b)
    x, _ = onehot(recs)
    h = np.tanh(np.asarray(x @ W0.T) + b0)
    return np.tanh(h @ W1.T + b1), h


def act_quant_shift(w, b):
    """k of act_quant_shift for the FP32 copies of W0, b0 (finite weights)"""
    W0, b0, _, _ = layers(w, b)
    m = max(np.abs(W0.astype(np.float32)).max(), np.abs(b0.astype(np.float32)).max())
    top = np.float32(92.0) * np.float32(m)
    e = int(np.frexp(top)[1]) if top > 0 else -60
    return min(max(30 - e, -100), 124)


def bf16(x):
    """round-to-nearest-even FP32 -> BF16, returned as FP32"""
    bits = np.asarray(x, np.float32).view(np.uint32)
    r = (bits + np.uint32(0x7FFF) + ((bits >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)
    return r.view(np.float32)


def w1_split(W1):
    """the device's split W1 ~ hi + lo (f64_to_fast_kernel): returns lo and dW = W1 - hi - lo, both float64"""
    v = W1.astype(np.float32)
    hi = bf16(v)
    lo = bf16(v - hi)
    return lo.astype(np.float64), W1 - hi.astype(np.float64) - lo.astype(np.float64)


def bound(recs, w, b, h=None):
    """per-entry bound [n, 96] of |Q_device - Q_fp64| (module docstring)"""
    W0, b0, W1, b1 = layers(w, b)
    x, occ = onehot(recs)
    if h is None:
        h = np.tanh(np.asarray(x @ W0.T) + b0)
    k = act_quant_shift(w, b)
    S = np.asarray(x @ np.abs(W0).T) + np.abs(b0)
    dh = 2 * U32 * S + 2.0 ** -(k + 1) * (occ[:, None] + 1) + TANH_ABS
    H = np.minimum(1.0, np.abs(h) + dh)
    aW = np.abs(W1)
    lo, dW = w1_split(W1)
    return (dh @ aW.T + (2.0 ** -17 + 64 * U32) * (H @ aW.T) + H @ (np.abs(dW) + 2.0 ** -8 * (1 + 2.0 ** -8) * np.abs(lo)).T
            + 2 * U32 * np.abs(b1) + TANH_ABS)


def greedy_check(counts, acts, q_dev_actions, q64, bnd):
    """eps = 0 choice against the FP64 first maximum of Q[to] over the oracle's list (envs with 0 < count < 128).
    Returns (mismatches, near_ties, checked): near ties are envs whose best and another listed `to` lie within the sum of their bounds
    of each other; there any of the near-tied actions is a correct FP32 answer.  Actions sharing a `to` tie exactly and list order
    decides them on both sides (first maximum)."""
    sel = np.nonzero((counts > 0) & (counts < 128))[0]
    to = (acts[sel].astype(np.int64) & 127)
    pos = np.arange(128)[None, :] < counts[sel, None]
    tq = np.where(pos, np.take_along_axis(q64[sel], np.minimum(to, 95), axis=1), -np.inf)
    tb = np.where(pos, np.take_along_axis(bnd[sel], np.minimum(to, 95), axis=1), 0.0)
    best = np.argmax(tq, axis=1)
    r = np.arange(len(sel))
    near = pos & (tq >= (tq[r, best] - tb[r, best])[:, None] - tb) & (to != to[r, best][:, None])
    is_near = near.any(axis=1)
    want = acts[sel, best]
    got = np.asarray(q_dev_actions)[sel]
    ok_near = (near | (to == to[r, best][:, None])) & pos & (acts[sel] == got[:, None])
    bad = np.where(is_near, ~ok_near.any(axis=1), got != want)
    return sel[bad], int(is_near.sum()), len(sel)
