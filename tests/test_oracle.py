"""CPU suite, part 1: pins the plain-C oracle (oracle/xq_oracle.c) to the reference.

* against tests/golden/rules_ref.npz, generated from the reference's own sources compiled
  unmodified (tests/golden/make_golden.py) -- runs anywhere, also on the GPU box;
* against tests/golden/reference_answers.npz, the reference's answers where it was once compared live (see
  make_golden.answers);
* live, in lock step, against oracle/_ref/libxq_ref.so when that library is present.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import recs_from_codes


def test_opening_kat(O, oracle_lib, golden):
    # SURVEY Appendix A.4: Red has 44 ordered actions at the opening
    e = O.new_envs(1)
    acts = np.zeros(128, np.uint16)
    n = oracle_lib.xqo_all_actions(e.ctypes.data, 0, acts)
    assert n == 44
    want = golden["opening"]
    assert [(a >> 7, a & 127) for a in acts[:n]] == [tuple(r) for r in want]
    assert (int(acts[0]) >> 7, int(acts[0]) & 127) == (0, 9)
    # reward KATs of SURVEY section 4
    assert oracle_lib.xqo_evaluate(e.ctypes.data, 0, 0) == 0 and oracle_lib.xqo_evaluate(e.ctypes.data, 0, 7) == 0
    assert oracle_lib.xqo_move(e.ctypes.data, 2, 1, 9, 1) == 11      # Red cannon takes the Black horse
    assert e[0]["red_score"] == 40
    assert oracle_lib.xqo_evaluate(e.ctypes.data, 0, 1) == 39
    assert oracle_lib.xqo_evaluate(e.ctypes.data, 1, 1) == -40
    assert oracle_lib.xqo_evaluate(e.ctypes.data, 0, 30) == 37
    st = np.zeros(1260)
    oracle_lib.xqo_state(e.ctypes.data, st)
    assert st.sum() == 31 and set(np.unique(st)) == {0.0, 1.0}


def test_golden_positions(O, oracle_lib, golden):
    recs = recs_from_codes(O, golden["pos_codes"], golden["pos_meta"])
    n = len(recs)
    counts = np.zeros(n, np.uint8)
    acts = np.zeros((n, 128), np.uint16)
    oracle_lib.xqo_batch_all_actions(recs.ctypes.data, n, counts, acts)
    assert (counts == golden["pos_counts"]).all()
    want = golden["pos_lists"]
    for i in range(n):
        assert (acts[i, :counts[i]] == want[i, :counts[i]]).all()


def test_golden_arbitrary_boards(O, oracle_lib, golden):
    codes = golden["arb_codes"]
    m = len(codes)
    meta = np.zeros((m, 4), np.int32)
    meta[:, 1] = golden["arb_player"]
    recs = recs_from_codes(O, codes, meta)
    counts = np.zeros(m, np.uint8)
    acts = np.zeros((m, 128), np.uint16)
    oracle_lib.xqo_batch_all_actions(recs.ctypes.data, m, counts, acts)
    assert (counts == golden["arb_counts"]).all()
    for i in range(m):
        assert (acts[i, :counts[i]] == golden["arb_lists"][i, :counts[i]]).all()
        for q, v in zip(golden["arb_q"][i], golden["arb_valid"][i]):
            assert oracle_lib.xqo_is_valid_move(recs[i:i + 1].ctypes.data, *[int(x) for x in q]) == v


def test_golden_traces(O, oracle_lib, golden):
    tr = golden["traces"]          # [env, ply, (n_legal, from, to, reward, done, winner)]
    n_envs, plies, _ = tr.shape
    seed = int(golden["seed"])
    envs = O.new_envs(n_envs)
    out = np.zeros((plies, n_envs), O.TRACE_DTYPE)
    st = np.zeros(1, O.STATS_DTYPE)
    oracle_lib.xqo_rollout_random(envs.ctypes.data, n_envs, 0, seed, plies, out.ctypes.data, st.ctypes.data)
    for e in range(n_envs):
        assert (out["n_legal"][:, e] == tr[e, :, 0]).all()
        assert ((out["action"][:, e] >> 7) == tr[e, :, 1]).all() and ((out["action"][:, e] & 127) == tr[e, :, 2]).all()
        assert (out["reward"][:, e] == tr[e, :, 3]).all()
        assert ((out["flags"][:, e] & 1) == tr[e, :, 4]).all()
        assert (((out["flags"][:, e] >> 1) & 3) == tr[e, :, 5]).all()
        fin = golden["finals"][e]
        assert (O.codes_of(envs[e]) == fin[:90]).all()
        assert (envs[e]["move_count"], envs[e]["player"], envs[e]["red_score"], envs[e]["black_score"]) == tuple(fin[90:])
    assert st[0]["steps"] == n_envs * plies and st[0]["games"] == tr[:, :, 4].sum()


def test_golden_rewards(O, oracle_lib, golden):
    codes = golden["arb_codes"]
    recs = recs_from_codes(O, codes[:64], np.zeros((64, 4), np.int32))
    for bi, (mc, pl), val in zip(golden["rew_board"], golden["rew_mc"], golden["rew_val"]):
        p = recs[bi:bi + 1].ctypes.data
        assert oracle_lib.xqo_evaluate(p, int(pl), int(mc)) == val
        assert oracle_lib.xqo_evaluate_int(p, int(pl), int(mc)) == val


def test_reward_integer_form_exhaustive():
    # SURVEY F5: (int)((double)s - (double)mc*0.1) == (10*s - mc)/10 (C truncation) on the whole
    # reachable domain; material differences are multiples of 5 in [-1480, 1480] (we test every int)
    s = np.arange(-3000, 3001, dtype=np.int64)[:, None]
    mc = np.arange(0, 201, dtype=np.int64)[None, :]
    fp = np.trunc(s.astype(np.float64) - mc.astype(np.float64) * 0.1).astype(np.int64)
    num = 10 * s - mc
    integer = np.sign(num) * (np.abs(num) // 10)
    assert (fp == integer).all()


def test_eps_threshold(oracle_lib):
    for eps in (0.0, 0.1, 0.5, 1.0, 1e-9, 0.999999999):
        t = oracle_lib.xqo_eps_threshold(eps)
        for c in (max(t, 1) - 1, t):
            if 0 <= c <= 2147483647:
                assert ((c / 2147483647.0) < eps) == (c < t)


def test_lockstep_vs_reference(O, oracle_lib, make_golden, answers):
    """oracle and the unmodified reference classes play the same random games move by move: against the reference's answers
    stored in tests/golden/reference_answers.npz, and live against oracle/_ref when it is built"""
    got = make_golden.lockstep_answers(oracle_lib)
    for k, v in got.items():
        assert np.array_equal(v, answers["lockstep_" + k]), k
    assert int(got["over"].sum()) >= 20
    ref_lib = O.ref()
    if ref_lib is None:
        return
    h = C.c_void_p(ref_lib.ref_env_new())
    rng = np.random.default_rng(0)
    e = O.new_envs(1)
    codes = np.zeros(90, np.uint8)
    meta = np.zeros(4, np.int32)
    buf = np.zeros(256, np.int32)
    acts = np.zeros(128, np.uint16)
    st1 = np.zeros(1260)
    st2 = np.zeros(1260)
    games = 0
    for step in range(6000):
        ref_lib.ref_env_get(h, codes, meta)
        assert (codes == O.codes_of(e[0])).all()
        assert tuple(meta) == (e[0]["move_count"], e[0]["player"], e[0]["red_score"], e[0]["black_score"])
        pl = int(e[0]["player"])
        n1 = ref_lib.ref_env_all_actions(h, pl, buf)
        n2 = oracle_lib.xqo_all_actions(e.ctypes.data, pl, acts)
        assert n1 == n2 and ((buf[0:2 * n1:2] << 7 | buf[1:2 * n1:2]) == acts[:n1]).all()
        if step % 50 == 0:
            ref_lib.ref_env_state(h, st1)
            oracle_lib.xqo_state(e.ctypes.data, st2)
            assert (st1 == st2).all()
            for _ in range(200):  # predicate on random queries, off-board included
                q = [int(v) for v in rng.integers(-1, 11, 4)]
                assert ref_lib.ref_env_is_valid_move(h, *q) == oracle_lib.xqo_is_valid_move(e.ctypes.data, *q)
        k = int(rng.integers(n1))
        f, t = int(acts[k]) >> 7, int(acts[k]) & 127
        assert ref_lib.ref_env_move(h, f, t) == oracle_lib.xqo_move(e.ctypes.data, f // 9, f % 9, t // 9, t % 9)
        mc = int(e[0]["move_count"])
        for side in (0, 1):
            assert ref_lib.ref_env_evaluate(h, side, mc) == oracle_lib.xqo_evaluate(e.ctypes.data, side, mc)
        over = ref_lib.ref_env_game_over(h)
        assert over == oracle_lib.xqo_game_over(e.ctypes.data)
        assert ref_lib.ref_env_winner(h) == oracle_lib.xqo_winner(e.ctypes.data)
        if over:
            games += 1
            ref_lib.ref_env_reset(h)
            oracle_lib.xqo_reset(e.ctypes.data)
    ref_lib.ref_env_free(h)
    assert games >= 20


def test_arbitrary_boards_vs_reference(O, oracle_lib, make_golden, answers):
    """unreachable positions: generator lists and the stand-alone predicate (SURVEY A.3 caveat); against the reference's answers
    stored in tests/golden/reference_answers.npz, and live against oracle/_ref when it is built"""
    got = make_golden.arbitrary_answers(oracle_lib)
    for k, v in got.items():
        assert np.array_equal(v, answers["arbitrary_" + k]), k
    ref_lib = O.ref()
    if ref_lib is None:
        return
    h = C.c_void_p(ref_lib.ref_env_new())
    rng = np.random.default_rng(9)
    buf = np.zeros(512, np.int32)
    acts = np.zeros(128, np.uint16)
    for i in range(300):
        codes = np.zeros(90, np.uint8)
        k = int(rng.integers(2, 34))
        pos = rng.choice(90, k, replace=False)
        codes[pos] = rng.integers(1, 15, k)
        pl = int(rng.integers(0, 2))
        meta = np.array([[int(rng.integers(0, 200)), pl, 0, 0]], np.int32)
        ref_lib.ref_env_set(h, codes, meta[0])
        rec = recs_from_codes(O, codes[None], meta)
        n1 = ref_lib.ref_env_all_actions(h, pl, buf)
        n2 = oracle_lib.xqo_all_actions(rec.ctypes.data, pl, acts)
        assert n1 == n2 and ((buf[0:2 * n1:2] << 7 | buf[1:2 * n1:2]) == acts[:n1]).all()
        for f in pos[:6]:
            for t in range(90):
                q = (int(f) // 9, int(f) % 9, t // 9, t % 9)
                assert ref_lib.ref_env_is_valid_move(h, *q) == oracle_lib.xqo_is_valid_move(rec.ctypes.data, *q)
        assert ref_lib.ref_env_game_over(h) == oracle_lib.xqo_game_over(rec.ctypes.data)
        assert ref_lib.ref_env_winner(h) == oracle_lib.xqo_winner(rec.ctypes.data)
    ref_lib.ref_env_free(h)


def test_rollout_vs_reference_driver(O, oracle_lib, make_golden, answers):
    """whole trajectories: same draws => identical traces for 1500 plies (auto-reset included); against the reference's trace
    stored in tests/golden/reference_answers.npz, and live against oracle/_ref when it is built"""
    got = make_golden.rollout_answers(oracle_lib)
    for k, v in got.items():
        assert np.array_equal(v, answers["rollout_" + k]), k
    ref_lib = O.ref()
    if ref_lib is None:
        return
    seed, env_id, plies = 99, 5, 1500
    draws = (O.rng_draws(seed, env_id, 0, plies) >> np.uint64(33)).astype(np.uint32)
    h = C.c_void_p(ref_lib.ref_env_new())
    tr = np.zeros((plies, 6), np.int32)
    games = C.c_long()
    assert ref_lib.ref_env_rollout_random(h, draws, plies, tr.ctypes.data, C.addressof(games)) == plies
    envs = O.new_envs(1)
    out = np.zeros((plies, 1), O.TRACE_DTYPE)
    st = np.zeros(1, O.STATS_DTYPE)
    oracle_lib.xqo_rollout_random(envs.ctypes.data, 1, env_id, seed, plies, out.ctypes.data, st.ctypes.data)
    assert (out["n_legal"][:, 0] == tr[:, 0]).all() and (out["reward"][:, 0] == tr[:, 3]).all()
    assert ((out["action"][:, 0] >> 7) == tr[:, 1]).all() and ((out["action"][:, 0] & 127) == tr[:, 2]).all()
    assert ((out["flags"][:, 0] & 1) == tr[:, 4]).all() and (((out["flags"][:, 0] >> 1) & 3) == tr[:, 5]).all()
    assert st[0]["games"] == games.value
    ref_lib.ref_env_free(h)


@pytest.mark.parametrize("self_play", [False, True])
def test_train_loop_vs_reference(O, oracle_lib, make_golden, answers, self_play, tmp_path, monkeypatch):
    """SURVEY 8(a) rows a12-a18 end to end: the reference's OWN ChessAI::train / startSelfPlay (src/chessai.cpp:85-170, :191-266: selectAction with its rand()
    stream injected, movePiece, evaluateBoard, done one ply early, TD target from the ONLINE network over all 8100 outputs,
    backpropagate as written, gameCompleted) against the same loop composed from the oracle's restatements (make_golden.oracle_train_loop).
    Same events, same draws consumed, final weights equal to rounding: against the reference's result stored in
    tests/golden/reference_answers.npz, and live against oracle/_ref when it is built (its network is oracle/nn_cpu.cpp's CPU definition)."""
    w, b, draws = make_golden.train_loop_inputs()
    episodes = 2
    events, pos, plies, w2, b2 = make_golden.oracle_train_loop(oracle_lib, w, b, draws, episodes, self_play)
    key = "selfplay" if self_play else "train"
    assert plies > 20 and events == list(answers[key + "_events"]) and pos == int(answers[key + "_consumed"])
    make_golden.check_loop(answers, key, w, b, draws, w2, b2, 1e-12)
    assert np.abs(w2 - w).max() > 1e-6                                        # the weights did move
    ref_lib = O.ref()
    if ref_lib is None:
        return
    h = C.c_void_p(ref_lib.ref_env_new())
    ref_lib.ref_rand_load(draws, len(draws))
    w_ref, b_ref = np.zeros_like(w), np.zeros_like(b)
    P = C.c_void_p
    monkeypatch.chdir(tmp_path)              # the reference appends to game_log.txt in the working directory
    assert (ref_lib.ref_ai_selfplay if self_play else ref_lib.ref_ai_train)(h, episodes, w.ctypes.data_as(P), b.ctypes.data_as(P), w_ref.ctypes.data_as(P), b_ref.ctypes.data_as(P)) == 0
    n_ev = ref_lib.ref_events_count()
    ev_ref = np.zeros(3 * n_ev, np.int32)
    ref_lib.ref_events_get(ev_ref)
    consumed = ref_lib.ref_rand_consumed()
    ref_lib.ref_env_free(h)
    assert pos == consumed
    assert list(ev_ref) == events
    assert np.abs(w2 - w_ref).max() < 1e-12 and np.abs(b2 - b_ref).max() < 1e-12


def test_reference_train_bench_leg(ref_lib):
    """bench.py's `reference_train` leg: the reference's own ChessAI::train timed for one game (CPU definition of its network without a GPU)"""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "oracle.ref_train_bench", "1"], cwd=root, capture_output=True, text=True, timeout=600)
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert r.returncode == 0 and out.get("plies", 0) > 0 and out["transitions_per_s"] > 0 and out["batch"] == 1, (out, r.stderr[-500:])
