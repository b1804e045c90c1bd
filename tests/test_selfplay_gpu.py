"""GPU tests of the replay buffer, batched epsilon-greedy action selection and the self-play collector
(BASELINE configs 3/4).  Selection parity is checked GIVEN identical Q inputs (SURVEY section 7, last bullet):
the Q-values the GPU used are fed to the oracle's restatement of DQN::selectAction with the same draws."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
LAYERS = [1260, 128, 8100]
LA = np.array(LAYERS, np.int32)


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


def rand_params(seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-0.05, 0.05, 1260 * 128 + 128 * 8100), rng.uniform(-0.05, 0.05, 128 + 8100)


def oracle_lists(L, recs):
    n = len(recs)
    counts = np.zeros(n, np.uint8)
    acts = np.zeros((n, 128), np.uint16)
    L.xqo_batch_all_actions(recs.ctypes.data, n, counts, acts)
    return counts, acts


def test_replay_ring_and_sampling(xq, O):
    rb = xq.ReplayBuffer(1000)
    rng = np.random.default_rng(0)
    def mk(n, tag):
        b = np.zeros(n, xq.TRANSITION_DTYPE)
        b["s"] = rng.integers(0, 2 ** 32, (n, 12), dtype=np.uint64).astype(np.uint32)
        b["reward"] = tag + np.arange(n)
        return b
    a = mk(600, 0); rb.insert(a)
    assert rb.info() == (600, 1000, 600)
    assert rb.get(0, 600).tobytes() == a.tobytes()
    b = mk(700, 10000); rb.insert(b)                         # wraps: slots 600..999 then 0..299
    assert rb.info() == (1000, 1000, 1300)
    ring = rb.get()
    assert ring[600:].tobytes() == b[:400].tobytes() and ring[:300].tobytes() == b[400:].tobytes() and ring[300:600].tobytes() == a[300:600].tobytes()
    out, idx = rb.sample(4096, seed=7, counter=3)
    want = ((O.rng_np(7, np.arange(4096, dtype=np.uint64), np.full(4096, 3, np.uint32)) >> np.uint64(1)) % np.uint64(1000)).astype(np.int64)
    assert (idx == want).all() and out.tobytes() == ring[idx].tobytes()
    assert len(np.unique(idx)) > 900                         # uniform over the ring
    with pytest.raises(xq.XQError):
        xq.ReplayBuffer(10).sample(4, 0, 0)                  # empty
    with pytest.raises(xq.XQError):
        xq.ReplayBuffer(0)


def test_act_stepwise_vs_oracle(xq, O, oracle_lib):
    """config 3 in small: eps-greedy choice per env per ply == oracle selectAction on the same Q and draws"""
    n, plies, seed, eps = 700, 25, 11, 0.1
    w, b = rand_params(4)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    env = xq.BatchedEnv(n, seed=seed, env_id0=50)
    ref = O.new_envs(n)
    thr = oracle_lib.xqo_eps_threshold(eps)
    explored = 0
    for p in range(plies):
        actions, q = xq.act(net, env, eps, want_q=True)
        counts, lists = oracle_lists(oracle_lib, ref)
        x = O.rng_np(seed, np.arange(n, dtype=np.uint64) + np.uint64(50), ref["ctr"])
        coin, idx = (x & np.uint64(0x7FFFFFFF)).astype(np.uint32), (x >> np.uint64(33)).astype(np.uint32)
        explored += int((coin < thr).sum())
        for i in range(n):
            qi = np.zeros(8100); qi[:90] = q[i, :90]
            k = oracle_lib.xqo_select_action(qi, lists[i], int(counts[i]), int(coin[i]), int(idx[i]), eps)
            assert actions[i] == lists[i, k], (p, i)
        if p == 0:   # Q used for acting vs the FP64 oracle: FP32 layer-0 gather + split-precision (BF16 hi+lo, 3 MMAs) layer 1
            st = np.zeros(1260); qq = np.zeros(8100)
            for i in range(0, n, 97):
                oracle_lib.xqo_state(ref[i:i + 1].ctypes.data, st)
                oracle_lib.xqo_nn_forward(LA, 3, w, b, st, qq)
                assert np.abs(q[i, :90] - qq[:90]).max() < 2e-5
        rew, done, win, cap, valid = env.step(actions, auto_reset=True)
        r0 = np.zeros(n, np.int32); d0, w0, c0, v0 = (np.zeros(n, np.uint8) for _ in range(4))
        oracle_lib.xqo_batch_step(ref.ctypes.data, n, actions, r0, d0, w0, c0, v0)
        assert (valid == 1).all() and (rew == r0).all() and (done == d0).all()
        for i in np.nonzero(d0)[0]:
            oracle_lib.xqo_reset(ref[i:i + 1].ctypes.data)
        assert env.get_boards().tobytes() == ref.tobytes()
    assert 0.05 * n * plies < explored < 0.15 * n * plies


@pytest.mark.parametrize("w0_scale", [1.0, 8.0])
def test_acting_q_is_a_pure_function_of_board_and_weights(xq, O, oracle_lib, w0_scale):
    """The acting path carries the layer-0 sum from ply to ply in fixed point and updates it from the squares a ply changed
    (l0_act_kernel).  Integer sums are associative, so the carried sum must equal a gather over all rows BIT FOR BIT: net A is
    used ply after ply (incremental, across captures, resets at the move cap / general captures and an injected position),
    net B is handed its weights again before every call (new weight version => full gather).  Both stay within 2e-5 of the FP64
    oracle at every checked ply (the scale of the fixed-point table follows max |W0|: second parameter set)."""
    n, plies, seed, eps = 600, 215, 23, 0.3
    w, b = rand_params(12)
    w = w.copy(); w[:1260 * 128] *= w0_scale
    netA = xq.DQN(LAYERS); netA.set_params(w, b)
    netB = xq.DQN(LAYERS)
    env = xq.BatchedEnv(n, seed=seed)
    st = np.zeros(1260); qq = np.zeros(8100)
    worst, finished = 0.0, 0
    for p in range(plies):
        if p == 40:      # an injected position (endgame-like: most squares change) in some envs
            recs = env.get_boards()
            recs["sq"][::7] = 0
            recs["sq"][::7, 0] = 0x00010000          # Red General on square 4
            recs["sq"][::7, 10] = 0x00000008 << 20   # Black General on square 85
            recs["sq"][::7, 5] = 0x0000C005          # a Red chariot and a Black chariot mid-board
            env.set_boards(recs)
        aA, qA = xq.act(netA, env, eps, want_q=True)
        netB.set_params(w, b)
        aB, qB = xq.act(netB, env, eps, want_q=True)
        assert np.array_equal(qA.view(np.uint32), qB.view(np.uint32)), p
        assert (aA == aB).all()
        if p in (0, 1, 2, 17, 41, 42, 120, 214):
            recs = env.get_boards()
            for i in range(0, n, 53):
                oracle_lib.xqo_state(recs[i:i + 1].ctypes.data, st)
                oracle_lib.xqo_nn_forward(LA, 3, w, b, st, qq)
                worst = max(worst, float(np.abs(qA[i, :90] - qq[:90]).max()))
        finished += int(env.step(aA, auto_reset=True)[1].sum())
    assert worst < 2e-5, worst
    assert finished > n          # resets happened (move cap at ply 200 + general captures)


def test_carried_sums_follow_every_weight_change(xq, O):
    """The per-env layer-0 sums (and the fixed-point table they are built from) belong to ONE version of W0 / b0.  Every way the online
    weights can change -- a TD update from the replay ring, the pipelined multi-update call, a host batch update, apply_grads after a
    gradient-only update, set_params, load_model, an FP64 reference-semantics step -- must invalidate them: after each, the Q the collector
    would act on equals, bit for bit, the Q of a second network that was just handed the same parameters (full gather, new table)."""
    import tempfile, os
    n = 500
    w, b = rand_params(21)
    net = xq.DQN(LAYERS, lr=1e-3); net.set_params(w, b)
    env = xq.BatchedEnv(n, seed=9)
    rb = xq.ReplayBuffer(1 << 15)
    probe = xq.DQN(LAYERS)

    def check(tag):
        xq.collect(net, env, rb, 3, 0.2)                     # carried plies under the current weights
        _, q1 = xq.act(net, env, 0.0, want_q=True)
        probe.set_params(*net.get_params())
        _, q2 = xq.act(probe, env, 0.0, want_q=True)
        assert np.array_equal(q1.view(np.uint32), q2.view(np.uint32)), tag

    check("initial")
    changes = {
        "td_update_replay": lambda: xq.td_update_replay(net, rb, 512, 3, 0, True, 1e-2, apply=True),
        "td_update_replay_n": lambda: xq.td_update_replay_n(net, rb, 512, 3, 10, 3, True, 1e-2),
        "td_update (host batch)": lambda: net.td_update(rb.get(0, 256), lr=1e-2),
        "gradient only + apply_grads": lambda: (xq.td_update_replay(net, rb, 512, 3, 50, True, 1e-2, apply=False), net.apply_grads(1e-2)),
        "set_params": lambda: net.set_params(*rand_params(22)),
        "fp64 backpropagate": lambda: net.backpropagate(np.eye(1, 1260, 7)[0], np.full(8100, 0.25), 0.05),
    }
    for tag, change in changes.items():
        before = net.get_params()[0][:1260 * 128].copy()
        change()
        assert np.abs(net.get_params()[0][:1260 * 128] - before).max() > 0, tag      # W0 did change
        check(tag)
    with tempfile.TemporaryDirectory() as d:
        other = xq.DQN(LAYERS); other.set_params(*rand_params(23)); other.save_model(os.path.join(d, "m.bin"))
        net.load_model(os.path.join(d, "m.bin"))
        check("load_model")


@pytest.mark.parametrize("train_done", [True, False])
def test_collect_fills_replay_like_the_train_loop(xq, O, oracle_lib, train_done):
    n, plies, seed, eps = 300, 230, 5, 0.1              # > 200 plies: crosses the move cap and the done-one-ply-early quirk
    w, b = rand_params(6)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    envA = xq.BatchedEnv(n, seed=seed)
    rb = xq.ReplayBuffer(n * plies + 17)
    xq.collect(net, envA, rb, plies, eps, train_done=train_done)
    envA.sync()
    stats = envA.stats()
    assert rb.info()[2] == n * plies and stats["steps"] == n * plies
    ring = rb.get(0, n * plies).reshape(plies, n)
    # replay the same policy step by step: GPU act (same Q, same draws) + oracle rules
    envB = xq.BatchedEnv(n, seed=seed)
    ref = O.new_envs(n)
    for p in range(plies):
        actions = xq.act(net, envB, eps)
        before = ref.copy()
        r0 = np.zeros(n, np.int32); d0, w0, c0, v0 = (np.zeros(n, np.uint8) for _ in range(4))
        oracle_lib.xqo_batch_step(ref.ctypes.data, n, actions, r0, d0, w0, c0, v0)
        t = ring[p]
        assert (t["action"] == actions).all() and (t["reward"] == r0).all() and (t["mover"] == before["player"]).all()
        assert t["s"].tobytes() == before["sq"].tobytes() and t["s2"].tobytes() == ref["sq"].tobytes()
        want_done = d0 | ((ref["move_count"] + 1 >= 200).astype(np.uint8) if train_done else 0)
        assert (t["done"] == want_done).all(), p
        for i in np.nonzero(d0)[0]:
            oracle_lib.xqo_reset(ref[i:i + 1].ctypes.data)
        envB.step(actions, auto_reset=True)
    assert envA.get_boards().tobytes() == ref.tobytes()
    assert stats["games"] >= n                              # every env finished at least one game


def test_two_stream_collector_plies(xq, O, oracle_lib):
    """At >= 4,096 envs per stream the collector cuts the env range in parts that run their [contraction -> act] chains on 2..4 streams
    (xq_selfplay_collect).  Same transitions, same finished-game events (with the env index of the whole range) and same final boards as
    the step-by-step path: GPU act (same Q, same draws) + oracle rules."""
    from cn_chess_ai_b200.trainer import drain_game_events, enable_game_events
    n, plies, seed, eps = 16500, 44, 17, 0.6            # not a multiple of 128: the second half ends in partial tiles / CTAs
    w, b = rand_params(31)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    envA = xq.BatchedEnv(n, seed=seed, env_id0=1000)
    rb = xq.ReplayBuffer(n * plies)
    enable_game_events(envA, n * plies)
    xq.collect(net, envA, rb, plies, eps, train_done=True)
    envA.sync()
    events, dropped = drain_game_events(envA)
    ring = rb.get(0, n * plies).reshape(plies, n)
    envB = xq.BatchedEnv(n, seed=seed, env_id0=1000)
    ref = O.new_envs(n)
    finished = []
    for p in range(plies):
        actions = xq.act(net, envB, eps)
        before = ref.copy()
        r0 = np.zeros(n, np.int32); d0, w0, c0, v0 = (np.zeros(n, np.uint8) for _ in range(4))
        oracle_lib.xqo_batch_step(ref.ctypes.data, n, actions, r0, d0, w0, c0, v0)
        t = ring[p]
        assert (t["action"] == actions).all() and (t["reward"] == r0).all(), p
        assert t["s"].tobytes() == before["sq"].tobytes() and t["s2"].tobytes() == ref["sq"].tobytes(), p
        for i in np.nonzero(d0)[0]:
            finished.append((p, int(i), int(ref[i]["red_score"]), int(ref[i]["black_score"])))
            oracle_lib.xqo_reset(ref[i:i + 1].ctypes.data)
        envB.step(actions, auto_reset=True)
    assert envA.get_boards().tobytes() == ref.tobytes()
    assert dropped == 0 and len(finished) > 20
    assert [(int(e["ply"]), int(e["env"]), int(e["red_score"]), int(e["black_score"])) for e in events] == finished


def test_td_update_from_replay_matches_host_batch(xq, O):
    w, b = rand_params(8)
    net1 = xq.DQN(LAYERS); net1.set_params(w, b)
    net2 = xq.DQN(LAYERS); net2.set_params(w, b)
    env = xq.BatchedEnv(512, seed=9)
    rb = xq.ReplayBuffer(4096)
    xq.collect(net1, env, rb, 8, 0.3)
    batch, idx = rb.sample(1000, seed=1, counter=2)
    xq.td_update_replay(net1, rb, 1000, seed=1, counter=2, lr=1e-6)
    net2.td_update(batch, lr=1e-6)
    w1, b1 = net1.get_params(); w2, b2 = net2.get_params()
    scale = np.abs(w2 - w).max()
    assert scale > 0 and np.abs(w1 - w2).max() <= 1e-4 * scale + 1e-9 and np.abs(b1 - b2).max() <= 1e-4 * scale + 1e-9


def test_pipelined_updates_equal_sequential_updates(xq):
    """xq_dqn_td_update_replay_n (bootstrap branch of update i+1 on a second stream under update i) == n single updates, bit for bit"""
    w, b = rand_params(12)
    env = xq.BatchedEnv(2048, seed=4)
    rb = xq.ReplayBuffer(1 << 15)
    nets = [xq.DQN(LAYERS, lr=1e-4) for _ in range(3)]
    for n in nets:
        n.set_params(w, b)
    xq.collect(nets[0], env, rb, 12, 0.3)
    env.sync()
    for u in range(7):
        xq.td_update_replay(nets[0], rb, 1500, 77, 40 + u, True, 1e-4)
    xq.td_update_replay_n(nets[1], rb, 1500, 77, 40, 7, True, 1e-4)
    xq.td_update_replay_n(nets[2], rb, 1500, 77, 40, 3, True, 1e-4)           # split in two calls + a target sync in between
    xq.td_update_replay_n(nets[2], rb, 1500, 77, 43, 4, True, 1e-4)
    p = [n.get_params() for n in nets]
    assert np.abs(p[0][0] - w).max() > 0
    for k in (1, 2):
        assert p[k][0].tobytes() == p[0][0].tobytes() and p[k][1].tobytes() == p[0][1].tobytes()
    # online-net bootstrap: the sequential fallback of the same entry point
    a, c = xq.DQN(LAYERS, lr=1e-4), xq.DQN(LAYERS, lr=1e-4)
    a.set_params(w, b); c.set_params(w, b)
    for u in range(3):
        xq.td_update_replay(a, rb, 1024, 5, u, False, 1e-4)
    xq.td_update_replay_n(c, rb, 1024, 5, 0, 3, False, 1e-4)
    assert a.get_params()[0].tobytes() == c.get_params()[0].tobytes()
