"""The batched tensor-core TD update (l0_pair_kernel -> l1_gemm_kernel<EPI_ROWMAX> -> td_delta_kernel -> dw_gemm_kernel) and
forward_boards (l1_gemm_kernel<EPI_STORE_TANH>) against the FP64 oracle, entry by entry, beyond the benchmarked configuration:
both hidden-delta modes x both bootstraps, ragged batch sizes, one handle whose batch size grows and shrinks, boards with up to
90 pieces, db1 collision patterns, the bootstrap maximum sample by sample (with weights that put it at the padded columns' doorstep
and at tile edges), the applied SGD step on every parameter, and Q at every row and column.

Every tolerance is either the rule of test_dqn_fast_gpu.py::test_td_gradient_batch_4096_vs_fp64_oracle (RULE A below, unchanged) or
a bound derived per element from the operands (D, H); each derivation sits next to the code that computes it."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

from conftest import recs_from_codes
from test_dqn_fast_gpu import LA, LAYERS, make_batch, rand_params, states_of

pytestmark = pytest.mark.gpu

GAMMA = 0.99
NW0, NW1 = 1260 * 128, 128 * 8100
G_B0 = NW0                       # compact gradient: [dW0^T 1260x128 | db0 128 | dW1 rows 0..89 | db1 0..89]
G_W1 = G_B0 + 128
G_B1 = G_W1 + 90 * 128
G_SIZE = G_B1 + 90               # 173,018
U32 = 2.0 ** -24                 # unit roundoff of FP32, round to nearest (CUDA cores)
U_TC = 2.0 ** -23                # FP32 accumulation inside the tensor core: its rounding mode is not documented, so truncation is assumed
U_BF = 2.0 ** -8                 # unit roundoff of BF16 (8 significant bits)
TANHF = 2.0 ** -23               # |tanhf(x) - tanh(x)|: CUDA documents at most 2 ulp, and |tanh| <= 1 has an ulp of at most 2^-24


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch_dev():
    import torch
    return torch, torch.device("cuda", 0)


@pytest.fixture(scope="module")
def pool(xq, O, oracle_lib):
    """4097 transitions of oracle-driven random play (desynchronised games, mixed `done`), their FP64 states, the boards of s"""
    batch, before, after = make_batch(O, oracle_lib, xq, 4097, seed=2024, train_done=True)
    x = np.ascontiguousarray(states_of(O, oracle_lib, before))
    x2 = np.ascontiguousarray(states_of(O, oracle_lib, after))
    return batch, x, x2, before


def split_params(w, b):
    """reference layout -> W0 [128][1260], b0, W1 [8100][128], b1 (views)"""
    return w[:NW0].reshape(128, 1260), b[:128], w[NW0:].reshape(8100, 128), b[128:]


def make_net(xq, w, b, tw=None, tb=None, mode=0):
    """a handle with online parameters (w, b) and, when given, target parameters (tw, tb)"""
    net = xq.DQN(LAYERS, lr=1e-3, gamma=GAMMA, mode=mode)
    if tw is None:
        net.set_params(w, b)
        return net
    net.set_params(tw, tb)                       # set_params refreshes the target too ...
    net.update_target_network()
    with tempfile.TemporaryDirectory() as d:     # ... so the online parameters come in through load_model, which leaves the target alone
        tmp = xq.DQN(LAYERS)
        tmp.set_params(w, b)
        tmp.save_model(os.path.join(d, "m.bin"))
        tmp.close()
        net.load_model(os.path.join(d, "m.bin"))
    return net


def device_grad(torch_dev, net, batch, use_target):
    """the compact gradient of one td_update_device(..., apply=False) call, float64 [173018]"""
    torch, dev = torch_dev
    from cn_chess_ai_b200.dist import grad_tensor
    n = len(batch)
    stage = torch.from_numpy(np.ascontiguousarray(batch).view(np.uint8).reshape(n, 128)).to(dev)
    torch.cuda.synchronize(dev)                  # the handle's stream reads what torch's stream wrote
    net.td_update_device(stage.data_ptr(), n, use_target_net=use_target, lr=1e-3, apply=False)
    net.sync()
    g = grad_tensor(net, dev).double().cpu().numpy().copy()
    del stage
    return g


def oracle_grad(L, w, b, tw, tb, batch, x, x2, mode):
    """xqo_td_batch_grad (per sample: getQValues(s) online, getQValues(s') with the bootstrap net, TD target, gradient at frozen weights;
    summed, FP64) mapped to the compact layout of the device gradient"""
    n = len(batch)
    gw, gb = np.zeros_like(w), np.zeros_like(b)
    loss = C.c_double()
    L.xqo_td_batch_grad(LA, 3, w, b, tw, tb, np.ascontiguousarray(x), np.ascontiguousarray(x2),
                        np.ascontiguousarray(batch["action"] & 127, dtype=np.int32), np.ascontiguousarray(batch["reward"], dtype=np.int32),
                        np.ascontiguousarray(batch["done"], dtype=np.uint8), GAMMA, mode, n, os.cpu_count() or 8, gw, gb, C.byref(loss))
    ref = np.concatenate([gw[:NW0].reshape(128, 1260).T.ravel(), gb[:128], gw[NW0:NW0 + 90 * 128], gb[128:128 + 90]])
    scale = np.abs(ref).max()
    # outside the compact layout the reference holds summation-order noise only (Q is indexed by action.to < 90)
    assert np.abs(gw[NW0 + 90 * 128:]).max() <= 1e-9 * scale and np.abs(gb[128 + 90:]).max() <= 1e-9 * scale
    return ref


def check_rule_a(g, ref, what=""):
    """RULE A, the tolerance of the batch-4096 oracle test, for every configuration (BF16 MMA operands split hi + lo, FP32 accumulation,
    BF16 h(s') under the bootstrap max):
      * every entry within 2e-3 of its row's largest reference entry + 2e-5 of the largest reference entry overall
        (rows: the 1260 features of dW0^T, the 90 destinations of dW1; db0 / db1 are judged by the global bound);
      * every entry within 1e-3 of the largest reference entry overall;
      * rows the batch never touches (no sample sets the feature / moves to the destination) are exactly 0.
    Returns the worst global and row-relative error ratios (<= 1 passes)."""
    assert g.shape == ref.shape == (G_SIZE,)
    assert np.isfinite(g).all(), what
    scale = np.abs(ref).max()
    assert scale > 0, what
    err = np.abs(g - ref)
    worst_global = err.max() / (1e-3 * scale)
    assert worst_global <= 1.0, (what, "global error", err.max(), scale)
    worst_row = 0.0
    for lo, hi in ((0, G_B0), (G_W1, G_B1)):
        e2, r2 = err[lo:hi].reshape(-1, 128), np.abs(ref[lo:hi]).reshape(-1, 128)
        bound = 2e-3 * r2.max(1) + 2e-5 * scale
        worst_row = max(worst_row, float((e2.max(1) / bound).max()))
        dead = r2.max(1) < 1e-12 * scale
        assert (g[lo:hi].reshape(-1, 128)[dead] == 0).all(), (what, "an untouched row is not exactly 0")
    assert worst_row <= 1.0, (what, "row-relative error", worst_row)
    return worst_global, worst_row


def with_to(batch, to):
    """the same transitions with action.to replaced (action.from kept): the TD update is defined for any transition"""
    out = batch.copy()
    out["action"] = (out["action"] & np.uint16(0xFF80)) | np.asarray(to, np.uint16)
    return out


# ---- A + B: the configuration matrix -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1000, 4097])
@pytest.mark.parametrize("use_target", [False, True], ids=["online", "target"])
@pytest.mark.parametrize("mode", [0, 1], ids=["as_written", "corrected"])
def test_td_gradient_modes_x_bootstraps(xq, oracle_lib, pool, torch_dev, mode, use_target, n):
    batch, x, x2, _ = pool
    w, b = rand_params(41)
    tw, tb = rand_params(42) if use_target else (w, b)
    net = make_net(xq, w, b, tw if use_target else None, tb if use_target else None, mode)
    g = device_grad(torch_dev, net, batch[:n], use_target)
    net.close()
    ref = oracle_grad(oracle_lib, w, b, tw, tb, batch[:n], x[:n], x2[:n], mode)
    worst = check_rule_a(g, ref, (mode, use_target, n))
    # how much a single 1 % tolerance over the whole update (test_dqn_fast_gpu.py::test_td_update_vs_fp64_oracle) could miss: the
    # dW0^T / db0 block's largest entry against 1 % of the largest entry overall.  Below 1, an error that wiped out that whole block
    # would still pass the single tolerance; rule A judges every row on its own scale.
    scale = np.abs(ref).max()
    block = np.abs(ref[:G_W1]).max() / (1e-2 * scale)
    block_err = np.abs(g - ref)[:G_W1].max() / (1e-2 * scale)
    print(f"\nmode={mode} target={use_target} n={n}: rule A worst global {worst[0]:.3f}, worst row {worst[1]:.3f}; "
          f"largest dW0^T/db0 entry = {block:.3f} x the 1% line, its error = {block_err:.2e} x the 1% line")


@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 129, 448, 449, 4095])
def test_td_gradient_batch_size_sweep(xq, oracle_lib, pool, torch_dev, n):
    """ChessAI::train's semantics (corrected delta, online bootstrap) at sizes around the 64-sample k-block, the 128-row tile, the 8
    sample splits of the gradient contraction (<= 448 samples leave some splits without a k-block) and the group of 8 of td_delta_kernel"""
    batch, x, x2, _ = pool
    first = (n * 7) % (len(batch) - n + 1)
    sl = slice(first, first + n)
    w, b = rand_params(43)
    net = make_net(xq, w, b, mode=xq.CORRECTED)
    g = device_grad(torch_dev, net, batch[sl], False)
    net.close()
    check_rule_a(g, oracle_grad(oracle_lib, w, b, w, b, batch[sl], x[sl], x2[sl], 1), n)


@pytest.mark.parametrize("done", ["none", "all", "mixed"])
def test_td_gradient_done_patterns(xq, oracle_lib, pool, torch_dev, done):
    batch, x, x2, _ = pool
    n = 1000
    bt = batch[1500:1500 + n].copy()
    bt["done"] = {"none": np.zeros(n), "all": np.ones(n), "mixed": np.random.default_rng(5).integers(0, 2, n)}[done].astype(np.uint8)
    w, b = rand_params(44)
    tw, tb = rand_params(45)
    net = make_net(xq, w, b, tw, tb, xq.AS_WRITTEN)
    g = device_grad(torch_dev, net, bt, True)
    net.close()
    check_rule_a(g, oracle_grad(oracle_lib, w, b, tw, tb, bt, x[1500:1500 + n], x2[1500:1500 + n], 0), done)


# ---- C: one handle, changing sizes --------------------------------------------------------------------------------------------------
def test_td_gradient_one_handle_growing_and_shrinking(xq, oracle_lib, pool, torch_dev):
    """4097 -> 65 -> 1 -> 4096 -> 129 on ONE handle (the workspace keeps its 4097 capacity and row stride; the tensor maps follow n),
    each against the oracle, then bit-identical to a fresh handle sized for that batch: the reduction order does not depend on the
    capacity, so only stale workspace state could make the two differ"""
    batch, x, x2, _ = pool
    w, b = rand_params(46)
    tw, tb = rand_params(47)
    slices = [slice(0, 4097), slice(1000, 1065), slice(7, 8), slice(1, 4097), slice(2000, 2129)]
    net = make_net(xq, w, b, tw, tb, xq.AS_WRITTEN)
    grads = []
    for sl in slices:
        g = device_grad(torch_dev, net, batch[sl], True)
        check_rule_a(g, oracle_grad(oracle_lib, w, b, tw, tb, batch[sl], x[sl], x2[sl], 0), sl)
        grads.append(g)
    net.close()
    for sl, g in zip(slices, grads):
        fresh = make_net(xq, w, b, tw, tb, xq.AS_WRITTEN)
        g2 = device_grad(torch_dev, fresh, batch[sl], True)
        fresh.close()
        assert g2.tobytes() == g.tobytes(), ("gradient depends on the handle's history", sl, np.abs(g2 - g).max())


# ---- D: the bootstrap maximum, sample by sample -------------------------------------------------------------------------------------
def hidden_f64(w, b, x):
    """h = tanh(W0 x + b0) in FP64, and a bound on |h_device - h| per entry: the device sums b0 and the <= 90 selected FP32 rows of
    W0^T sequentially in FP32 (each of the k + 1 weights rounded to FP32 once, k additions: (k + 2) u |terms| to first order, doubled to
    cover the second-order remainder) and takes tanhf (TANHF); tanh is 1-Lipschitz"""
    W0, b0 = split_params(w, b)[:2]
    h = np.tanh(x @ W0.T + b0)
    k = x.sum(1, keepdims=True)
    dh = 2.0 * (k + 2) * U32 * (x @ np.abs(W0).T + np.abs(b0)) + TANHF
    return h, dh


def layer1_bound(h, dh, W1, b1):
    """|z_device - z| per output of the tensor-core contraction z = bf16(h) . bf16(W1)^T + (b1 as BF16 hi + lo + lo2), FP32 accumulation:
      * products: bf16(h~) bf16(f32(w)) = h w (1 + a)(1 + b)(1 + c) with |a|, |b| <= 2^-8 (BF16), |c| <= 2^-24 (FP32 master copy), h~ = h +- dh:
        |error| <= (2^-7 + 2^-15) |h| |w| + (1 + 2^-6) |w| dh;
      * 131 FP32 accumulations (128 products + 3 bias terms) in the tensor core: 131 U_TC (1 + 2^-6) (sum |h w| + sum |w| dh + |b|);
      * the bias: FP32 rounding of b1 plus a 24-bit three-term split: 2^-22 |b|.
    Returns (z, dz) for rows of h."""
    A = np.abs(h) @ np.abs(W1).T
    B = dh @ np.abs(W1).T
    z = h @ W1.T + b1
    dz = (2.0 ** -7 + 2.0 ** -15) * A + (1 + 2.0 ** -6) * B + 131 * U_TC * (1 + 2.0 ** -6) * (A + B + np.abs(b1)) + 2.0 ** -22 * np.abs(b1)
    return z, dz


def sech2_sup(z, dz):
    """sup of tanh' = 1 - tanh^2 over [z - dz, z + dz] (mean value theorem: |tanh(z~) - tanh(z)| <= sech2_sup * |z~ - z|)"""
    return 1.0 - np.tanh(np.maximum(np.abs(z) - dz, 0.0)) ** 2


def weight_set(kind, seed, hot=None):
    w, b = rand_params(seed)
    b1 = b[128:]
    if kind == "ii":                  # every z(s') < 0: a padded output leaking a 0 into the max would move delta1 by ~ gamma (1 - q^2) 0.99
        b1[:] = -3.0
    elif kind == "iii":               # the maximum at one chosen output (tile / half / padding edges)
        b1[:] = -1.0
        b1[hot] = 2.0
    elif kind == "iv":                # tanh saturates
        w[NW0:] *= 20.0
        b1 *= 20.0
    return w, b


HOT = [0, 111, 112, 223, 224, 4031, 8063, 8064, 8099]     # first / last output of a 112-column half and a 224-column tile, the last tile


@pytest.mark.parametrize("use_target", [False, True], ids=["online", "target"])
@pytest.mark.parametrize("kind,hot", [("i", None), ("ii", None), ("iv", None)] + [("iii", c) for c in HOT],
                         ids=["uniform", "all_negative", "saturated"] + [f"hot{c}" for c in HOT])
def test_bootstrap_max_sample_by_sample(xq, oracle_lib, pool, torch_dev, kind, hot, use_target):
    """90 transitions with action.to = 0..89 and done = 0: db1[to] is exactly one sample's delta1 (a single summand everywhere on its way),
    compared with the oracle's (q(s)[to] - r - gamma max q(s')) (1 - q(s)[to]^2) from xqo_nn_forward, against a bound derived per sample:
      delta1 = (q - t)(1 - q^2) with q = tanhf(z_q), z_q an FP32 dot product of h(s) with W1[to] (+ b1[to]), and t = r + gamma tanhf(max z(s'))
      |dq| <= sech2_sup(z_q) dz_q + TANHF,   dz_q = 11 u (|h| . |W1[to]| + |b1[to]|) (4 products, 5 shuffle levels, 1 bias add) + u |h| . |W1[to]|
              + |W1[to]| . dh                 (FP32 rounding of W1, h error)
      |dt| <= gamma (sech2_sup(m) dm + TANHF) + u gamma + 2 u (|r| + gamma),   dm = max_c dz_c of layer1_bound (|max a - max b| <= max |a - b|)
      |d delta1| <= (1 - q^2)(dq + dt + u |q - t|) + |q - t| (2 |q| dq + dq^2 + 2u) + (dq + dt)(2 |q| dq + dq^2) + u |delta1|"""
    batch, x, x2, _ = pool
    n = 90
    sl = slice(100, 100 + n)
    bt = with_to(batch[sl], np.arange(n))
    bt["done"] = 0
    bt["reward"] = np.arange(n) % 5 - 2
    if use_target:
        w, b = rand_params(48)
        tw, tb = weight_set(kind, 49, hot)
    else:
        w, b = tw, tb = weight_set(kind, 49, hot)
    net = make_net(xq, w, b, tw if use_target else None, tb if use_target else None, xq.CORRECTED)
    g = device_grad(torch_dev, net, bt, use_target)
    net.close()
    d1_dev = g[G_B1:G_B1 + n]
    xs, xs2 = x[sl], x2[sl]
    r = bt["reward"].astype(np.float64)
    # the oracle's delta1
    qs, qn = np.zeros(8100), np.zeros(8100)
    d1_ref, q_ref, t_ref = np.zeros(n), np.zeros(n), np.zeros(n)
    for i in range(n):
        oracle_lib.xqo_nn_forward(LA, 3, w, b, xs[i], qs)
        oracle_lib.xqo_nn_forward(LA, 3, tw, tb, xs2[i], qn)
        q_ref[i], t_ref[i] = qs[i], r[i] + GAMMA * qn.max()
        d1_ref[i] = (q_ref[i] - t_ref[i]) * (1 - q_ref[i] ** 2)
    # the bound, from a float64 restatement pinned to the oracle
    W1, b1 = split_params(w, b)[2:]
    h, dh = hidden_f64(w, b, xs)
    A_q = (np.abs(h) * np.abs(W1[:n])).sum(1)
    z_q = (h * W1[:n]).sum(1) + b1[:n]
    assert np.allclose(np.tanh(z_q), q_ref, rtol=0, atol=1e-12)
    dz_q = 11 * U32 * (A_q + np.abs(b1[:n])) + U32 * A_q + (dh * np.abs(W1[:n])).sum(1)
    dq = sech2_sup(z_q, dz_q) * dz_q + TANHF
    th, dth = hidden_f64(tw, tb, xs2)
    z2, dz2 = layer1_bound(th, dth, *split_params(tw, tb)[2:])
    m, dm = z2.max(1), dz2.max(1)
    assert np.allclose(r + GAMMA * np.tanh(m), t_ref, rtol=0, atol=1e-12)
    if kind == "iii":
        assert (z2.argmax(1) == hot).all()
    if kind == "ii":
        assert (m < 0).all()
    dt = GAMMA * (sech2_sup(m, dm) * dm + TANHF) + U32 * GAMMA + 2 * U32 * (np.abs(r) + GAMMA)
    e1, e2 = dq + dt, 2 * np.abs(q_ref) * dq + dq ** 2
    bound = ((1 - q_ref ** 2) * (e1 + U32 * np.abs(q_ref - t_ref)) + np.abs(q_ref - t_ref) * (e2 + 2 * U32) + e1 * e2
             + U32 * np.abs(d1_ref) + 1e-12)
    err = np.abs(d1_dev - d1_ref)
    worst = int(np.argmax(err / bound))
    print(f"\n{kind} {hot} target={use_target}: max |d delta1| = {err.max():.3e}, worst err / bound = {err[worst] / bound[worst]:.3f} "
          f"(bound {bound[worst]:.3e}, dm {dm[worst]:.3e})")
    assert (err <= bound).all(), ("delta1 outside its derived bound", worst, d1_dev[worst], d1_ref[worst], bound[worst])


# ---- E: boards with up to 90 pieces -------------------------------------------------------------------------------------------------
def full_boards(O, m, seed):
    """arbitrary boards with 60..90 occupied squares (every fourth one completely filled), random piece codes 1..14"""
    rng = np.random.default_rng(seed)
    codes = np.zeros((m, 90), np.uint8)
    for i in range(m):
        k = 90 if i % 4 == 0 else int(rng.integers(60, 91))
        codes[i, rng.choice(90, k, replace=False)] = rng.integers(1, 15, k)
    meta = np.stack([rng.integers(0, 199, m), rng.integers(0, 2, m), rng.integers(0, 500, m), rng.integers(0, 500, m)], 1).astype(np.int32)
    return recs_from_codes(O, codes, meta)


@pytest.fixture(scope="module")
def full_batch(xq, O, oracle_lib):
    n = 1000
    s, s2 = full_boards(O, n, 61), full_boards(O, n, 62)
    rng = np.random.default_rng(63)
    bt = np.zeros(n, xq.TRANSITION_DTYPE)
    bt["s"], bt["s2"] = s["sq"], s2["sq"]
    bt["action"] = (rng.integers(0, 90, n) << 7) | rng.integers(0, 90, n)
    bt["mover"] = s["player"]
    bt["reward"] = rng.integers(-50, 51, n)
    bt["done"] = rng.integers(0, 2, n)
    x, x2 = states_of(O, oracle_lib, s), states_of(O, oracle_lib, s2)
    assert (x.sum(1) >= 60).all() and (x.sum(1) == 90).any()
    return bt, np.ascontiguousarray(x), np.ascontiguousarray(x2), s


@pytest.mark.parametrize("mode,use_target", [(0, True), (1, False)], ids=["as_written_target", "corrected_online"])
def test_td_gradient_full_boards(xq, oracle_lib, full_batch, torch_dev, mode, use_target):
    bt, x, x2, _ = full_batch
    w, b = rand_params(64)
    tw, tb = rand_params(65) if use_target else (w, b)
    net = make_net(xq, w, b, tw if use_target else None, tb if use_target else None, mode)
    g = device_grad(torch_dev, net, bt, use_target)
    net.close()
    check_rule_a(g, oracle_grad(oracle_lib, w, b, tw, tb, bt, x, x2, mode), (mode, use_target))


# ---- F: db1 collision patterns ------------------------------------------------------------------------------------------------------
def to_pattern(kind, n):
    if kind == "one_to":                  # the whole batch on one destination: one match group per warp, every k-block, every split
        return np.full(n, 37)
    if kind == "alternating":             # two destinations interleaved within every warp
        return np.where(np.arange(n) % 2 == 0, 5, 77)
    # runs of equal destinations with lengths 1..700, placed so that they straddle 32-sample warps, 64-sample k-blocks and the
    # 512-sample rounds of the 8 sample splits
    lengths = np.random.default_rng(71).integers(1, 700, n)
    run = np.repeat(np.arange(n), lengths)[:n]
    return (run * 37 + 11) % 90


@pytest.mark.parametrize("kind", ["one_to", "alternating", "runs"])
def test_td_gradient_db1_collisions(xq, oracle_lib, pool, torch_dev, kind):
    batch, x, x2, _ = pool
    n = 4097
    bt = with_to(batch, to_pattern(kind, n))
    w, b = rand_params(72)
    tw, tb = rand_params(73)
    net = make_net(xq, w, b, tw, tb, xq.AS_WRITTEN)
    g = device_grad(torch_dev, net, bt, True)
    net.close()
    check_rule_a(g, oracle_grad(oracle_lib, w, b, tw, tb, bt, x, x2, 0), kind)
    used = np.unique(to_pattern(kind, n))
    assert (g[G_B1:G_B1 + 90][np.setdiff1d(np.arange(90), used)] == 0).all()


# ---- G: the applied step, every parameter -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [65, 4097])
@pytest.mark.parametrize("mode", [0, 1], ids=["as_written", "corrected"])
def test_applied_step_every_parameter(xq, O, pool, torch_dev, mode, n):
    """Twin handles with the same parameters: A computes g (apply=False), B applies the step to the same batch (apply=True).  Each of the
    173,018 compact entries of B moves to w32 - f32(lr) g within 1 FP32 ulp (one fused multiply-add rounds once: 1/2 ulp); everything
    else keeps its bits.  Afterwards B's forward_boards and act Q equal, bit for bit, those of a fresh handle given B.get_params(): the BF16
    operand copies of the touched W1 rows (and the acting path's residual copy) were refreshed from the FP32 master, not approximated."""
    torch, dev = torch_dev
    batch, _, _, before = pool
    bt = batch[:n]
    w, b = rand_params(81)
    tw, tb = rand_params(82)
    lr = 3e-5
    A = make_net(xq, w, b, tw, tb, mode)
    B = make_net(xq, w, b, tw, tb, mode)
    g = device_grad(torch_dev, A, bt, True)
    A.close()
    stage = torch.from_numpy(np.ascontiguousarray(bt).view(np.uint8).reshape(n, 128)).to(dev)
    torch.cuda.synchronize(dev)
    B.td_update_device(stage.data_ptr(), n, use_target_net=True, lr=lr, apply=True)
    B.sync()
    del stage
    w1, b1 = B.get_params()
    w32, b32 = w.astype(np.float32).astype(np.float64), b.astype(np.float32).astype(np.float64)
    old = np.concatenate([w32[:NW0].reshape(128, 1260).T.ravel(), b32[:128], w32[NW0:NW0 + 90 * 128], b32[128:128 + 90]])
    new = np.concatenate([w1[:NW0].reshape(128, 1260).T.ravel(), b1[:128], w1[NW0:NW0 + 90 * 128], b1[128:128 + 90]])
    expect = old - float(np.float32(lr)) * g
    ulp = np.spacing(np.maximum(np.abs(old), np.abs(expect)).astype(np.float32)).astype(np.float64)
    assert (np.abs(new - expect) <= ulp).all(), ("applied step", int(np.argmax(np.abs(new - expect) / ulp)))
    assert (new != old).sum() > 1000                                    # the step is visible in FP32
    assert w1[NW0 + 90 * 128:].tobytes() == w32[NW0 + 90 * 128:].tobytes() and b1[128 + 90:].tobytes() == b32[128 + 90:].tobytes()
    fresh = xq.DQN(LAYERS, lr=1e-3, gamma=GAMMA, mode=mode)
    fresh.set_params(w1, b1)
    recs = np.concatenate([before[:200], full_boards(O, 56, 83)])
    assert B.forward_boards(recs).tobytes() == fresh.forward_boards(recs).tobytes()
    env = xq.BatchedEnv(1000, seed=84)
    env.rollout_random(30)
    a1, q1 = xq.act(B, env, eps=0.0, want_q=True)
    a2, q2 = xq.act(fresh, env, eps=0.0, want_q=True)
    assert q1.tobytes() == q2.tobytes() and (a1 == a2).all()
    B.close()
    fresh.close()


# ---- H: forward_boards at every row and column --------------------------------------------------------------------------------------
def check_forward_every_entry(xq, L, recs, x, w, b, what):
    """Q = tanhf(z~) of EPI_STORE_TANH against tanh(z) in FP64, every row and column: |Q - tanh(z)| <= sech2_sup(z, dz) dz + TANHF with
    dz from layer1_bound (h(s) enters the contraction as BF16, as h(s') does in the TD update).  The float64 restatement is pinned to
    xqo_nn_forward on a few rows."""
    net = xq.DQN(LAYERS)
    net.set_params(w, b)
    q = net.forward_boards(recs).astype(np.float64)
    net.close()
    n = len(recs)
    assert q.shape == (n, 8100) and np.isfinite(q).all()
    W1, b1 = split_params(w, b)[2:]
    worst, worst_at = 0.0, None
    for r0 in range(0, n, 512):
        h, dh = hidden_f64(w, b, x[r0:r0 + 512])
        z, dz = layer1_bound(h, dh, W1, b1)
        err = np.abs(q[r0:r0 + 512] - np.tanh(z))
        ratio = err / (sech2_sup(z, dz) * dz + TANHF)
        k = np.unravel_index(np.argmax(ratio), ratio.shape)
        if ratio[k] > worst:
            worst, worst_at = float(ratio[k]), (r0 + int(k[0]), int(k[1]))
        if r0 == 0 or r0 + 512 >= n:                                 # pin the restatement on the first and last rows of the batch
            ref = np.zeros(8100)
            for i in sorted({0, len(h) - 1}):
                L.xqo_nn_forward(LA, 3, w, b, x[r0 + i], ref)
                assert np.abs(np.tanh(z[i]) - ref).max() <= 1e-12
    print(f"\n{what}: worst |Q - Q64| / bound = {worst:.3f} at {worst_at}")
    assert worst <= 1.0, (what, worst, worst_at)


def forward_weights(kind):
    w, b = rand_params(91)
    if kind == "all_negative":
        b[128:] = -3.0
    elif kind == "last_columns":          # outputs 8064..8099 (the 36 real columns of the last tile) carry distinct, recognisable values
        W1 = w[NW0:].reshape(8100, 128)
        W1[8064:] *= 0.01
        b[128 + 8064:] = np.linspace(-0.9, 0.85, 36)
    return w, b


@pytest.mark.parametrize("kind", ["uniform", "all_negative", "last_columns"])
@pytest.mark.parametrize("n", [129, 4097])
def test_forward_boards_every_entry(xq, oracle_lib, pool, n, kind):
    _, x, _, before = pool
    w, b = forward_weights(kind)
    check_forward_every_entry(xq, oracle_lib, before[:n], x[:n], w, b, (n, kind))


def test_forward_boards_full_boards(xq, oracle_lib, full_batch):
    _, x, _, s = full_batch
    w, b = forward_weights("uniform")
    check_forward_every_entry(xq, oracle_lib, s, x, w, b, "full boards")
