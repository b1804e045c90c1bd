"""GPU parity tests of the FP64 DQN path (through the C ABI) against the FP64 oracle and against
tests/golden/nn_refcuda.npz, which was produced ON A B200 by the reference's OWN CUDA network
(src/dqn.cu compiled unmodified, tests/golden/make_golden.py --nn-gpu).  Tolerance: 1e-12 abs
(FP64; only the summation order / FMA contraction differ)."""
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-12
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def nn_golden():
    """the reference's outputs, with the inputs it was given regenerated from their seed (checked against the stored digest)"""
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    g = dict(np.load(os.path.join(GOLDEN, "nn_refcuda.npz")))
    _, w, b, xs, ts = mg.nn_cases(np.random.default_rng(mg.NN_SEED))[0]
    assert mg.nn_inputs_digest(w, b, xs, ts) == str(g["inputs_sha256"]), "regenerated inputs differ from the reference's"
    g.update(w0=w, b0=b, x0=xs, t0=ts)
    return g


def rand_net(rng, layers):
    nw = sum(layers[i] * layers[i + 1] for i in range(len(layers) - 1))
    return rng.uniform(-0.05, 0.05, nw), rng.uniform(-0.02, 0.02, sum(layers[1:]))


def test_forward_backprop_vs_reference_cuda_golden(xq, nn_golden):
    g = nn_golden
    layers = g["layers0"]
    assert list(layers) == [1260, 128, 8100]
    net = xq.DQN(layers, mode=xq.AS_WRITTEN)
    net.set_params(g["w0"], g["b0"])
    q = net.get_q_values(g["x0"])
    assert q.shape == (3, 8100) and np.abs(q.ravel()[g["q0_idx"]] - g["q0_at"]).max() < TOL
    net.backpropagate(g["x0"], g["t0"], lr=0.001)        # three sequential reference steps
    w, b = net.get_params()
    idx = g["w_after0_idx"]
    want = g["w0"].copy()
    want[idx] = g["w_after0_at"]
    n0 = 1260 * 128                                        # layer 0 in full: the entries not stored kept w0 in the reference
    assert np.abs(w[:n0] - want[:n0]).max() < TOL and np.abs(w[idx] - want[idx]).max() < TOL
    assert np.abs(b - g["b_after0"]).max() < TOL
    assert np.abs(w - g["w0"]).max() > 1e-5


@pytest.mark.parametrize("layers,mode", [([1260, 128, 8100], 0), ([1260, 128, 8100], 1), ([12, 8, 30], 0), ([12, 8, 30], 1),
                                          ([40, 16, 24, 50], 1), ([7, 5], 0)])
def test_forward_backprop_vs_oracle(xq, O, oracle_lib, layers, mode):
    rng = np.random.default_rng(sum(layers) + mode)
    w, b = rand_net(rng, layers)
    la = np.array(layers, np.int32)
    net = xq.DQN(layers, mode=mode)
    net.set_params(w, b)
    xs = (rng.random((4, layers[0])) < 0.1).astype(np.float64) if layers[0] > 100 else rng.uniform(-1, 1, (4, layers[0]))
    ts = rng.uniform(-1, 1, (4, layers[-1]))
    q = net.get_q_values(xs)
    for x, qq in zip(xs, q):
        out = np.zeros(layers[-1])
        oracle_lib.xqo_nn_forward(la, len(la), w, b, np.ascontiguousarray(x), out)
        assert np.abs(out - qq).max() < TOL
    net.backpropagate(xs, ts, lr=0.01)
    w0, b0 = w.copy(), b.copy()
    for x, t in zip(xs, ts):
        oracle_lib.xqo_nn_backprop(la, len(la), w0, b0, np.ascontiguousarray(x), np.ascontiguousarray(t), 0.01, mode)
    w1, b1 = net.get_params()
    assert np.abs(w1 - w0).max() < TOL and np.abs(b1 - b0).max() < TOL
    assert np.abs(w1 - w).max() > 1e-6


def test_select_action_and_td_step(xq, O, oracle_lib):
    layers = [1260, 128, 8100]
    la = np.array(layers, np.int32)
    rng = np.random.default_rng(3)
    w, b = rand_net(rng, layers)
    net = xq.DQN(layers, lr=0.001, gamma=0.99, mode=xq.AS_WRITTEN)
    net.set_params(w, b)
    envs = O.new_envs(1)
    st = np.zeros(1, O.STATS_DTYPE)
    oracle_lib.xqo_rollout_random(envs.ctypes.data, 1, 0, 1, 37, None, st.ctypes.data)
    s = np.zeros(1260)
    oracle_lib.xqo_state(envs.ctypes.data, s)
    acts = np.zeros(128, np.uint16)
    n = oracle_lib.xqo_all_actions(envs.ctypes.data, int(envs[0]["player"]), acts)
    q = np.zeros(8100)
    oracle_lib.xqo_nn_forward(la, 3, w, b, s, q)
    thr = oracle_lib.xqo_eps_threshold(0.1)
    assert xq.lib().xq_eps_threshold(0.1) == thr
    for coin, idx in ((0, 12345), (thr - 1, 99), (thr, 5), (2 ** 31 - 1, 7)):
        want = oracle_lib.xqo_select_action(q, acts, n, coin, idx, 0.1)
        assert net.select_action(s, 0.1, acts[:n], coin, idx) == want
    with pytest.raises(xq.XQError):
        net.select_action(s, 0.1, acts[:0], 0, 0)
    # TD step, online bootstrap (ChessAI::train) and target-net bootstrap (DQN::train), done and not done
    oracle_lib.xqo_rollout_random(envs.ctypes.data, 1, 0, 1, 1, None, st.ctypes.data)
    s2 = np.zeros(1260)
    oracle_lib.xqo_state(envs.ctypes.data, s2)
    w0, b0 = w.copy(), b.copy()
    tw, tb = w.copy(), b.copy()      # target network = initial parameters
    for a_to, r, done, use_t in ((13, 39.0, False, False), (4, -40.0, True, False), (77, 5.0, False, True)):
        net.train(s, a_to, r, s2, done, use_target_net=use_t, lr=0.001)
        qs = np.zeros(8100); qn = np.zeros(8100); tgt = np.zeros(8100)
        oracle_lib.xqo_nn_forward(la, 3, w0, b0, s, qs)
        oracle_lib.xqo_nn_forward(la, 3, tw if use_t else w0, tb if use_t else b0, s2, qn)
        oracle_lib.xqo_td_target(qs, qn, 8100, a_to, r, int(done), 0.99, tgt)
        oracle_lib.xqo_nn_backprop(la, 3, w0, b0, s, tgt, 0.001, 0)
        w1, b1 = net.get_params()
        assert np.abs(w1 - w0).max() < TOL and np.abs(b1 - b0).max() < TOL
    net.update_target_network()


def test_model_file_format(xq, tmp_path):
    layers = [1260, 128, 8100]
    net = xq.DQN(layers, seed=5)
    w, b = net.get_params()
    assert np.abs(w).max() <= 0.05 and (b == 0).all() and np.unique(w).size > 1000000
    path = tmp_path / "model.bin"
    net.save_model(path)
    raw = open(path, "rb").read()
    assert len(raw) == 9650484                                   # SURVEY section 5: 9,584,640 + 65,824 + 8 + 12
    assert np.frombuffer(raw, np.float64, net.n_weights).tobytes() == w.tobytes()
    assert raw[-20:] == (3).to_bytes(8, "big") + (1260).to_bytes(4, "big") + (128).to_bytes(4, "big") + (8100).to_bytes(4, "big")
    net2 = xq.DQN(layers, seed=6)
    assert not np.array_equal(net2.get_params()[0], w)
    net2.load_model(path)
    w2, b2 = net2.get_params()
    assert np.array_equal(w2, w) and np.array_equal(b2, b)
    bad = xq.DQN([1260, 64, 8100])
    with pytest.raises(xq.XQError):
        bad.load_model(path)
    with pytest.raises(xq.XQError):
        net.load_model(tmp_path / "missing.bin")
    with pytest.raises(xq.XQError):
        xq.DQN([5])
    # same seed => same init on every rank (multi-GPU replicas start identical)
    assert np.array_equal(xq.DQN(layers, seed=5).get_params()[0], w)
