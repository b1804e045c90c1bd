"""Generates tests/golden/*.npz from the reference's OWN sources compiled unmodified
(oracle/_ref/libxq_ref.so; recipe oracle/Makefile).  XQ_REFERENCE_SRC names a checkout of the
reference project:   XQ_REFERENCE_SRC=<checkout> python tests/golden/make_golden.py
The rules fixtures need no GPU.  `--nn-gpu` instead runs the reference's own CUDA network
(src/dqn.cu compiled unmodified into oracle/_ref/libxq_ref_cuda.so, which the first form builds
when nvcc is present) on a B200 and writes tests/golden/nn_refcuda.npz.
"""
import ctypes as C
import hashlib
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import loader as O  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def ref_get(R, h):
    codes = np.zeros(90, np.uint8)
    meta = np.zeros(4, np.int32)
    R.ref_env_get(h, codes, meta)
    return codes, meta


def rules():
    R = O.ref()
    L = O.oracle()
    assert R is not None, "reference build missing"
    h = C.c_void_p(R.ref_env_new())
    buf = np.zeros(256, np.int32)
    # 1. opening KAT
    n = R.ref_env_all_actions(h, 0, buf)
    opening = buf[:2 * n].reshape(n, 2).copy()
    # 2. traced random rollouts: 8 envs x 600 plies, draws = xq_rng(seed, env, ctr) >> 33
    seed, n_envs, plies = 20240607, 8, 600
    traces = np.zeros((n_envs, plies, 6), np.int32)
    finals = np.zeros((n_envs, 94), np.int32)
    pos_codes, pos_meta, pos_counts, pos_lists = [], [], [], []
    for e in range(n_envs):
        R.ref_env_reset(h)
        draws = (O.rng_draws(seed, e, 0, plies) >> np.uint64(33)).astype(np.uint32)
        # replay ply by ply so positions + ordered lists can be harvested on the way
        for p in range(plies):
            codes, meta = ref_get(R, h)
            k = R.ref_env_all_actions(h, int(meta[1]), buf)
            if (p % 9) == e % 9:
                pos_codes.append(codes.copy()); pos_meta.append(meta.copy()); pos_counts.append(k)
                lst = np.full(128, 0xFFFF, np.uint16)
                lst[:k] = (buf[0:2 * k:2] << 7) | buf[1:2 * k:2]
                pos_lists.append(lst)
            t = np.zeros(6, np.int32)
            got = R.ref_env_rollout_random(h, draws[p:p + 1], 1, t.ctypes.data, None)
            assert got == 1
            traces[e, p] = t
        codes, meta = ref_get(R, h)
        finals[e, :90] = codes
        finals[e, 90:] = meta
    # 3. isValidMove / getValidMoves on arbitrary (mostly unreachable) boards
    rng = np.random.default_rng(5)
    m = 256
    arb_codes = np.zeros((m, 90), np.uint8)
    arb_player = rng.integers(0, 2, m).astype(np.uint8)
    arb_q = np.zeros((m, 48, 4), np.int32)
    arb_valid = np.zeros((m, 48), np.uint8)
    arb_counts = np.zeros(m, np.uint8)
    arb_lists = np.full((m, 128), 0xFFFF, np.uint16)
    for i in range(m):
        k = int(rng.integers(2, 36))
        pos = rng.choice(90, k, replace=False)
        arb_codes[i, pos] = rng.integers(1, 15, k)
        meta = np.array([int(rng.integers(0, 199)), int(arb_player[i]), 0, 0], np.int32)
        R.ref_env_set(h, arb_codes[i], meta)
        cnt = R.ref_env_all_actions(h, int(arb_player[i]), buf)
        assert cnt <= 128
        arb_counts[i] = cnt
        arb_lists[i, :cnt] = (buf[0:2 * cnt:2] << 7) | buf[1:2 * cnt:2]
        for j in range(48):
            if j < 40:
                f = int(rng.choice(pos)); t = int(rng.integers(0, 90))
                q = (f // 9, f % 9, t // 9, t % 9)
            else:
                q = tuple(int(v) for v in rng.integers(-1, 11, 4))
            arb_q[i, j] = q
            arb_valid[i, j] = R.ref_env_is_valid_move(h, *q)
    # 4. reward table: evaluateBoard(Red, mc) on boards with assorted material, every mc 0..200
    rew_codes, rew_mc, rew_val = [], [], []
    for i in range(64):
        codes = arb_codes[i]
        R.ref_env_set(h, codes, np.array([0, 0, 0, 0], np.int32))
        for mc in range(0, 201, 1):
            for pl in (0, 1):
                rew_codes.append(i); rew_mc.append((mc, pl)); rew_val.append(R.ref_env_evaluate(h, pl, mc))
    np.savez_compressed(os.path.join(HERE, "rules_ref.npz"), opening=opening, seed=np.uint64(seed), traces=traces, finals=finals,
                        pos_codes=np.array(pos_codes), pos_meta=np.array(pos_meta), pos_counts=np.array(pos_counts, np.uint8),
                        pos_lists=np.array(pos_lists), arb_codes=arb_codes, arb_player=arb_player, arb_q=arb_q,
                        arb_valid=arb_valid, arb_counts=arb_counts, arb_lists=arb_lists,
                        rew_board=np.array(rew_codes, np.int32), rew_mc=np.array(rew_mc, np.int32), rew_val=np.array(rew_val, np.int32))
    print("rules_ref.npz:", len(pos_codes), "positions,", n_envs * plies, "traced plies,", m, "arbitrary boards")


def nn_cases(rng):
    cases = []
    for layers in ([1260, 128, 8100], [12, 8, 30]):
        nw = sum(layers[i] * layers[i + 1] for i in range(len(layers) - 1))
        nb = sum(layers[1:])
        w = rng.uniform(-0.05, 0.05, nw)
        b = rng.uniform(-0.02, 0.02, nb)
        xs = (rng.random((3, layers[0])) < (32.0 / 1260 if layers[0] == 1260 else 0.3)).astype(np.float64)
        ts = rng.uniform(-1, 1, (3, layers[-1]))
        cases.append((np.array(layers, np.int32), w, b, xs, ts))
    return cases


NN_SEED = 11
NN_SAMPLED_Q = 4096
NN_SAMPLED_WEIGHTS = 6144


def nn_inputs_digest(w, b, xs, ts):
    """sha256 of the inputs of a case, so that a test regenerating them from NN_SEED knows they are the ones the reference saw"""
    return hashlib.sha256(b"".join(np.ascontiguousarray(a, np.float64).tobytes() for a in (w, b, xs, ts))).hexdigest()


def compact_nn(out):
    """what tests/golden/nn_refcuda.npz keeps of case 0, the {1260,128,8100} network (its 1.2M weights before and after would take
    19 MB): the inputs as their digest (the test regenerates them from NN_SEED), the biases after the update in full, and fixed,
    seeded samples: NN_SAMPLED_Q entries of Q, and the weights after the update at every layer-0 entry the reference changed (the
    others kept w0) plus NN_SAMPLED_WEIGHTS further entries."""
    rng = np.random.default_rng(0)
    w, w_after, q = out["w0"], out["w_after0"], out["q0"].ravel()
    n0 = int(out["layers0"][0]) * int(out["layers0"][1])
    changed = np.nonzero(w_after[:n0] != w[:n0])[0]
    rest = np.setdiff1d(np.arange(w.size), changed)
    idx = np.sort(np.concatenate([changed, rng.choice(rest, NN_SAMPLED_WEIGHTS, replace=False)]))
    q_idx = np.sort(rng.choice(q.size, NN_SAMPLED_Q, replace=False))
    return {"layers0": out["layers0"], "inputs_sha256": np.array(nn_inputs_digest(w, out["b0"], out["x0"], out["t0"])),
            "q0_idx": q_idx.astype(np.int32), "q0_at": q[q_idx], "b_after0": out["b_after0"],
            "w_after0_idx": idx.astype(np.int32), "w_after0_at": w_after[idx]}


def nn(lib_name, out_path):
    """forward / backpropagate through the reference DQN class; with libxq_ref_cuda.so this is the
    reference's own CUDA code (src/dqn.cu) and needs a GPU."""
    R = C.CDLL(os.path.join(ROOT, "oracle", "_ref", lib_name))
    R.ref_dqn_new.restype = C.c_void_p
    R.ref_last_error.restype = C.c_char_p
    P = C.c_void_p
    rng = np.random.default_rng(NN_SEED)
    out = {}
    for ci, (layers, w, b, xs, ts) in enumerate(nn_cases(rng)):
        h = R.ref_dqn_new(layers.ctypes.data_as(P), len(layers))
        assert h, R.ref_last_error()
        h = P(h)
        R.ref_dqn_set_params(h, w.ctypes.data_as(P), b.ctypes.data_as(P))
        qs = np.zeros((len(xs), layers[-1]))
        for i, x in enumerate(xs):
            q = np.zeros(layers[-1])
            assert R.ref_dqn_forward(h, x.ctypes.data_as(P), len(x), q.ctypes.data_as(P), len(q)) == len(q)
            qs[i] = q
        for x, t in zip(xs, ts):
            assert R.ref_dqn_backprop(h, x.ctypes.data_as(P), len(x), t.ctypes.data_as(P), len(t), C.c_double(0.001)) == 0
        w2 = np.zeros_like(w); b2 = np.zeros_like(b)
        R.ref_dqn_get_params(h, w2.ctypes.data_as(P), b2.ctypes.data_as(P))
        out.update({f"layers{ci}": layers, f"w{ci}": w, f"b{ci}": b, f"x{ci}": xs, f"t{ci}": ts, f"q{ci}": qs,
                    f"w_after{ci}": w2, f"b_after{ci}": b2})
        R.ref_dqn_free(h)
    np.savez_compressed(out_path, **compact_nn(out))
    print(out_path, "written")


LA = np.array([1260, 128, 8100], np.int32)


def train_loop_inputs():
    """weights, biases and injected rand() stream of tests/test_oracle.py::test_train_loop_vs_reference"""
    rng = np.random.default_rng(5)
    w = rng.uniform(-0.05, 0.05, 1260 * 128 + 128 * 8100)
    b = rng.uniform(-0.05, 0.05, 128 + 8100)
    return w, b, rng.integers(0, 2 ** 31 - 1, 2000, dtype=np.int64).astype(np.int32)


def adapter_inputs():
    """the same for tests/test_adapter_gpu.py: the adapter's DQN::selectAction draws (coin31, idx31) from xq_rng(0xD09A, 0, call);
    the reference consumes rand() once, and once more when exploring"""
    rng = np.random.default_rng(77)
    w = rng.uniform(-0.05, 0.05, 1260 * 128 + 128 * 8100)
    b = rng.uniform(-0.05, 0.05, 128 + 8100)
    stream = []
    for v in O.rng_np(0xD09A, np.zeros(600, np.uint64), np.arange(600, dtype=np.uint32)):
        coin, idx = int(v) & 0x7FFFFFFF, int(v) >> 33
        stream.append(coin)
        if coin / 2147483647.0 < 0.1:
            stream.append(idx)
    return w, b, np.array(stream, np.int32)


def oracle_train_loop(L, w, b, draws, episodes, self_play):
    """ChessAI::train / startSelfPlay (src/chessai.cpp:85-170, :191-266) composed from the oracle's restatements: selectAction fed the
    rand() stream `draws`, movePiece, evaluateBoard, done one ply early, TD target from the ONLINE network over all 8100 outputs,
    backpropagate as written, gameCompleted.  Returns (events, draws consumed, plies, weights, biases)."""
    w2, b2 = w.copy(), b.copy()
    pos, events, plies = 0, [], 0
    acts = np.zeros(128, np.uint16)
    state, nxt, q, qs, qn, tgt = np.zeros(1260), np.zeros(1260), np.zeros(8100), np.zeros(8100), np.zeros(8100), np.zeros(8100)
    for ep in range(episodes):
        e = O.new_envs(1)
        player, move_count = 0, 0                                             # chessai.cpp:90-94
        L.xqo_state(e.ctypes.data, state)
        while not L.xqo_game_over(e.ctypes.data) and (self_play or move_count < 200):
            if self_play:
                player = int(e[0]["player"])                                  # :198 board->getCurrentPlayer()
            n = L.xqo_all_actions(e.ctypes.data, player, acts)
            if n == 0:
                break
            coin = int(draws[pos]); pos += 1
            idx = 0
            if coin / 2147483647.0 < 0.1:                                     # dqn.cpp:30-33: the second rand() only when exploring
                idx = int(draws[pos]); pos += 1
            else:
                L.xqo_nn_forward(LA, 3, w2, b2, state, q)
            a = int(acts[L.xqo_select_action(q, acts, n, coin, idx, 0.1)])
            f, t = a >> 7, a & 127
            L.xqo_move(e.ctypes.data, f // 9, f % 9, t // 9, t % 9)
            move_count = int(e[0]["move_count"])
            reward = L.xqo_evaluate(e.ctypes.data, player, move_count)
            L.xqo_state(e.ctypes.data, nxt)
            done = bool(L.xqo_game_over(e.ctypes.data)) or (not self_play and move_count + 1 >= 200)      # :119 vs :227
            L.xqo_nn_forward(LA, 3, w2, b2, state, qs)
            if not done:
                L.xqo_nn_forward(LA, 3, w2, b2, nxt, qn)
            L.xqo_td_target(qs, qn, 8100, t, float(reward), int(done), 0.99, tgt)
            L.xqo_nn_backprop(LA, 3, w2, b2, state, tgt, 0.001, 0)
            state[:] = nxt
            player ^= 1
            plies += 1
        events += [ep + 1, int(e[0]["red_score"]), int(e[0]["black_score"])]
    return events, pos, plies, w2, b2


LOOP_SAMPLED_WEIGHTS = 4096


def compact_loop(key, w, b, draws, events, consumed, w_after, b_after):
    """a training loop's result in little space: its events and rand() draws consumed, the digest of its inputs, which weights and
    biases it changed (bit masks), the changed biases in full and the changed weights at a fixed, seeded sample of LOOP_SAMPLED_WEIGHTS"""
    changed = np.nonzero(w_after != w)[0]
    idx = np.sort(np.random.default_rng(0).choice(changed, min(LOOP_SAMPLED_WEIGHTS, changed.size), replace=False))
    bch = np.nonzero(b_after != b)[0]
    return {key + "_inputs_sha256": np.array(nn_inputs_digest(w, b, draws, np.zeros(0))), key + "_events": np.array(events, np.int32),
            key + "_consumed": np.array(consumed), key + "_w_changed": np.packbits(w_after != w), key + "_w_idx": idx.astype(np.int32),
            key + "_w_at": w_after[idx], key + "_b_changed": np.packbits(b_after != b), key + "_b_at": b_after[bch]}


def check_loop(g, key, w, b, draws, w_out, b_out, tol):
    """w_out / b_out (a loop started from w, b with the rand() stream draws) against the stored result of the same loop"""
    assert nn_inputs_digest(w, b, draws, np.zeros(0)) == str(g[key + "_inputs_sha256"]), "inputs differ from the stored run's"
    for v0, v, mask, idx, at in ((w, w_out, g[key + "_w_changed"], g[key + "_w_idx"], None), (b, b_out, g[key + "_b_changed"], None, None)):
        changed = np.unpackbits(mask, count=v0.size).astype(bool)
        kept = ~changed
        idx, at = (idx, g[key + "_w_at"]) if idx is not None else (np.nonzero(changed)[0], g[key + "_b_at"])
        assert np.abs(v[kept] - v0[kept]).max() < tol and np.abs(v[idx] - at).max() < tol


def strict_positions():
    """the positions of tests/test_strict.py::test_oracle_equals_reference_composition"""
    sys.path.insert(0, os.path.dirname(HERE))
    from conftest import harvest_positions, random_boards
    return np.concatenate([harvest_positions(O, 40, 5, 31, seed=2), random_boards(O, 150, seed=5, max_pieces=24)])


def lockstep_answers(L, steps=6000):
    """what tests/test_oracle.py::test_lockstep_vs_reference asks along its random games (moves picked by default_rng(0) from the
    ordered list, reset on game over): per ply the record (crc32 of the squares + move count, player, scores), the list size and the
    crc32 of the ordered list, movePiece's return, evaluateBoard for both sides, game over, winner; every 50 plies the crc32 of the
    state vector and isValidMove on 200 random queries, off-board included"""
    rng = np.random.default_rng(0)
    e = O.new_envs(1)
    acts = np.zeros(128, np.uint16)
    st = np.zeros(1260)
    out = {k: [] for k in ("record", "count", "list", "move", "eval", "over", "winner", "state", "valid")}
    for step in range(steps):
        r = e[0]
        out["record"].append([zlib.crc32(r["sq"].tobytes()), r["move_count"], r["player"], r["red_score"], r["black_score"]])
        pl = int(r["player"])
        n = L.xqo_all_actions(e.ctypes.data, pl, acts)
        out["count"].append(n)
        out["list"].append(zlib.crc32(acts[:n].tobytes()))
        if step % 50 == 0:
            L.xqo_state(e.ctypes.data, st)
            out["state"].append(zlib.crc32(st.tobytes()))
            for _ in range(200):
                q = [int(v) for v in rng.integers(-1, 11, 4)]
                out["valid"].append(L.xqo_is_valid_move(e.ctypes.data, *q))
        k = int(rng.integers(n))
        f, t = int(acts[k]) >> 7, int(acts[k]) & 127
        out["move"].append(L.xqo_move(e.ctypes.data, f // 9, f % 9, t // 9, t % 9))
        mc = int(e[0]["move_count"])
        out["eval"].append([L.xqo_evaluate(e.ctypes.data, side, mc) for side in (0, 1)])
        over = L.xqo_game_over(e.ctypes.data)
        out["over"].append(over)
        out["winner"].append(L.xqo_winner(e.ctypes.data))
        if over:
            L.xqo_reset(e.ctypes.data)
    types = {"record": np.int64, "list": np.uint32, "state": np.uint32, "move": np.int32, "eval": np.int32, "count": np.uint8,
             "over": np.int8, "winner": np.int8, "valid": np.int8}
    return {k: np.array(v, types[k]) for k, v in out.items()}


def arbitrary_answers(L, boards=300):
    """what tests/test_oracle.py::test_arbitrary_boards_vs_reference asks on its unreachable positions (default_rng(9)): the ordered
    list, isValidMove from the first six occupied squares to every square, game over and winner"""
    sys.path.insert(0, os.path.dirname(HERE))
    from conftest import recs_from_codes
    rng = np.random.default_rng(9)
    acts = np.zeros(128, np.uint16)
    out = {"count": [], "list": [], "valid": [], "over": [], "winner": []}
    for _ in range(boards):
        codes = np.zeros(90, np.uint8)
        k = int(rng.integers(2, 34))
        pos = rng.choice(90, k, replace=False)
        codes[pos] = rng.integers(1, 15, k)
        pl = int(rng.integers(0, 2))
        meta = np.array([[int(rng.integers(0, 200)), pl, 0, 0]], np.int32)
        rec = recs_from_codes(O, codes[None], meta)
        n = L.xqo_all_actions(rec.ctypes.data, pl, acts)
        lst = np.full(128, 0xFFFF, np.uint16)
        lst[:n] = acts[:n]
        out["count"].append(n)
        out["list"].append(lst)
        valid = np.full(6 * 90, 255, np.uint8)                              # 255: fewer than six pieces on the board
        valid[:len(pos[:6]) * 90] = [L.xqo_is_valid_move(rec.ctypes.data, int(f) // 9, int(f) % 9, t // 9, t % 9) for f in pos[:6] for t in range(90)]
        out["valid"].append(valid)
        out["over"].append(L.xqo_game_over(rec.ctypes.data))
        out["winner"].append(L.xqo_winner(rec.ctypes.data))
    return {k: np.array(v, np.uint16 if k == "list" else np.int8) for k, v in out.items()}


def rollout_answers(L, seed=99, env_id=5, plies=1500):
    """the trace of tests/test_oracle.py::test_rollout_vs_reference_driver: the reference's random-policy driver fed
    xq_rng(seed, env_id, ply) >> 33, auto-reset included; (n_legal, from, to, reward, done, winner) per ply and the games finished"""
    envs = O.new_envs(1)
    tr = np.zeros((plies, 1), O.TRACE_DTYPE)
    st = np.zeros(1, O.STATS_DTYPE)
    L.xqo_rollout_random(envs.ctypes.data, 1, env_id, seed, plies, tr.ctypes.data, st.ctypes.data)
    tr = tr[:, 0]
    trace = np.stack([tr["n_legal"], tr["action"] >> 7, tr["action"] & 127, tr["reward"], tr["flags"] & 1, (tr["flags"] >> 1) & 3], 1)
    return {"trace": trace.astype(np.int32), "games": np.array(int(st[0]["games"]))}


def answers():
    """tests/golden/reference_answers.npz: the reference's answers where the tests above once compared the oracle with it live,
    reproduced by the oracle: training loops (events, draws consumed, changed weights), strict action lists, the lockstep games,
    the arbitrary boards and the random-policy rollout trace.  The live tests
    pinned the oracle to the reference on exactly these inputs (events and lists equal, weights to 1e-12), so regenerating this
    file is only sound while they still pass against oracle/_ref."""
    L = O.oracle()
    out = {}
    for key, (w, b, draws), self_play in (("train", train_loop_inputs(), False), ("selfplay", train_loop_inputs(), True),
                                          ("adapter_train", adapter_inputs(), False), ("adapter_selfplay", adapter_inputs(), True)):
        events, consumed, _, w2, b2 = oracle_train_loop(L, w, b, draws, 2, self_play)
        out.update(compact_loop(key, w, b, draws, events, consumed, w2, b2))
    recs = strict_positions()
    n = len(recs)
    counts, acts = np.zeros(n, np.uint8), np.zeros((n, 128), np.uint16)
    loose = np.zeros(n, np.uint8)
    L.xqo_batch_all_actions_strict(recs.ctypes.data, n, counts, acts)
    L.xqo_batch_all_actions(recs.ctypes.data, n, loose, np.zeros((n, 128), np.uint16))
    acts[np.arange(128)[None, :] >= counts[:, None]] = 0xFFFF
    out.update(strict_counts=counts, strict_lists=acts, strict_rejected=np.array(int(loose.sum()) - int(counts.sum())))
    for prefix, got in (("lockstep_", lockstep_answers(L)), ("arbitrary_", arbitrary_answers(L)), ("rollout_", rollout_answers(L))):
        out.update({prefix + k: v for k, v in got.items()})
    np.savez_compressed(os.path.join(HERE, "reference_answers.npz"), **out)
    print("reference_answers.npz written")


if __name__ == "__main__":
    if "--answers" in sys.argv:
        answers()
    elif "--nn-gpu" in sys.argv:
        nn("libxq_ref_cuda.so", os.path.join(HERE, "nn_refcuda.npz"))
    else:
        O.build()
        rules()
