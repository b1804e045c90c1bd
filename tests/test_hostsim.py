"""CPU suite, part 2: the DEVICE rules source (cn_chess_ai_b200/csrc/xq_rules.cuh), compiled for
the host by tests/hostsim (test-only, never shipped), diffed against the oracle and the golden
fixtures.  This is how the kernel logic is proven before any GPU time is spent."""
import numpy as np

from conftest import harvest_positions, random_boards, recs_from_codes


def _lists(H, recs, bitboard=False):
    n = len(recs)
    counts = np.zeros(n, np.uint8)
    acts = np.zeros((n, 128), np.uint16)
    (H.hs_bb_all_actions if bitboard else H.hs_all_actions)(recs.ctypes.data, n, counts.ctypes.data, acts.ctypes.data)
    return counts, acts


def _oracle_lists(L, recs):
    n = len(recs)
    counts = np.zeros(n, np.uint8)
    acts = np.zeros((n, 128), np.uint16)
    L.xqo_batch_all_actions(recs.ctypes.data, n, counts, acts)
    acts[np.arange(128)[None, :] >= counts[:, None]] = 0xFFFF
    return counts, acts


def test_device_rules_reachable_positions(O, oracle_lib, hostsim):
    recs = harvest_positions(O, 1500, 45, 5)      # 67,500 positions over whole games
    c1, a1 = _oracle_lists(oracle_lib, recs)
    c2, a2 = _lists(hostsim, recs)
    assert (c1 == c2).all() and (a1 == a2).all()
    assert c1.max() <= 119 and c1.min() >= 1


def test_device_rules_arbitrary_boards(O, oracle_lib, hostsim):
    recs = random_boards(O, 4000, seed=21)
    c1, a1 = _oracle_lists(oracle_lib, recs)
    c2, a2 = _lists(hostsim, recs)
    assert (c1 == c2).all() and (a1 == a2).all()
    rng = np.random.default_rng(4)
    for i in range(400):
        p = recs[i:i + 1].ctypes.data
        for _ in range(120):
            q = [int(v) for v in rng.integers(-1, 11, 4)]
            assert oracle_lib.xqo_is_valid_move(p, *q) == hostsim.hs_is_valid_move(p, *q)
        for s in range(0, 90, 7):
            t1 = np.zeros(32, np.uint8)
            t2 = np.zeros(32, np.uint8)
            n1 = oracle_lib.xqo_valid_moves(p, s // 9, s % 9, t1)
            n2 = hostsim.hs_valid_moves(p, s // 9, s % 9, t2.ctypes.data)
            assert n1 == n2 and (t1[:n1] == t2[:n1]).all()


def test_device_rules_golden(O, hostsim, golden):
    recs = recs_from_codes(O, golden["pos_codes"], golden["pos_meta"])
    c, a = _lists(hostsim, recs)
    assert (c == golden["pos_counts"]).all() and (a == golden["pos_lists"]).all()
    meta = np.zeros((len(golden["arb_codes"]), 4), np.int32)
    meta[:, 1] = golden["arb_player"]
    recs = recs_from_codes(O, golden["arb_codes"], meta)
    c, a = _lists(hostsim, recs)
    assert (c == golden["arb_counts"]).all() and (a == golden["arb_lists"]).all()
    for i in range(len(recs)):
        for q, v in zip(golden["arb_q"][i], golden["arb_valid"][i]):
            assert hostsim.hs_is_valid_move(recs[i:i + 1].ctypes.data, *[int(x) for x in q]) == v


def test_device_scalar_helpers(oracle_lib, hostsim):
    assert all(hostsim.hs_piece_score(t) == oracle_lib.xqo_piece_score(t) for t in range(8))
    for s in (0, 1, 2 ** 63 + 5):
        for e in (0, 1, 99999, 2 ** 40):
            for c in (0, 1, 2 ** 32 - 1):
                assert hostsim.hs_rng(s, e, c) == oracle_lib.xqo_rng(s, e, c)
    for d in range(-2960, 2961, 5):
        for mc in range(0, 201):
            num = 10 * d - mc
            want = int(np.trunc(float(d) - float(mc) * 0.1))
            assert hostsim.hs_reward(d, mc) == want


def test_bitboard_count_and_decode(O, oracle_lib, hostsim, golden):
    """xq_bitboard.cuh (slot-parallel rollout kernel): per-piece count + k-th decode == oracle lists"""
    for recs in (harvest_positions(O, 1500, 45, 5, seed=8), random_boards(O, 6000, seed=33, max_pieces=50)):
        c1, a1 = _oracle_lists(oracle_lib, recs)
        c2, a2 = _lists(hostsim, recs, bitboard=True)
        bad = np.nonzero((c1 != c2) | (a1 != a2).any(1))[0]
        assert len(bad) == 0, f"{len(bad)} boards differ, first {bad[:4]}"
    recs = recs_from_codes(O, golden["pos_codes"], golden["pos_meta"])
    c, a = _lists(hostsim, recs, bitboard=True)
    assert (c == golden["pos_counts"]).all() and (a == golden["pos_lists"]).all()


def _team_vs_oracle(O, L, H, team, recs, seed, id0, plies):
    n = len(recs)
    a, b = recs.copy(), recs.copy()
    tr0 = np.zeros((plies, n), O.TRACE_DTYPE)
    st0 = np.zeros(1, O.STATS_DTYPE)
    L.xqo_rollout_random(a.ctypes.data, n, id0, seed, plies, tr0.ctypes.data, st0.ctypes.data)
    tr1 = np.zeros((plies, n), O.TRACE_DTYPE)
    st1 = np.zeros(1, O.STATS_DTYPE)
    if team == 1:      # the board-per-thread kernel
        assert H.hs_lane_rollout(b.ctypes.data, n, id0, seed, plies, tr1.ctypes.data, st1.ctypes.data) == 0
    else:
        assert H.hs_team_rollout(team, b.ctypes.data, n, id0, seed, plies, tr1.ctypes.data, st1.ctypes.data) == 0
    bad = np.nonzero((tr0.view(np.uint64) != tr1.view(np.uint64)).any(0))[0]
    assert len(bad) == 0, f"team {team}: {len(bad)} envs differ, first env {bad[:3]}, first ply {np.nonzero(tr0.view(np.uint64)[:, bad[0]] != tr1.view(np.uint64)[:, bad[0]])[0][:3]}"
    assert a.tobytes() == b.tobytes()
    assert st0.tobytes() == st1.tobytes()


def test_team_rollout_phases(O, oracle_lib, hostsim):
    """xq_rollout_team.cuh (rollout_team_kernel, teams of 4): the three phases of a ply, run thread by thread on the host, reproduce the
    oracle's fused rollout record for record -- from the opening over several games, resumed in the middle of games (Black to
    move, captured pieces, non-zero scores and counters) and from finished boards"""
    mid = harvest_positions(O, 600, 6, 37, seed=5)       # snapshots after 37, 74, ... plies: both colours to move
    fin = O.new_envs(8)
    fin["move_count"][:4] = 200
    fin["sq"][4:, 0] &= np.uint32(0xFFF0FFFF)           # Red general gone: never stepped, restarted (chessai.cpp:90,96)
    _team_vs_oracle(O, oracle_lib, hostsim, 4, O.new_envs(1500), 11, 5000, 450)
    _team_vs_oracle(O, oracle_lib, hostsim, 4, mid, 77, 0, 230)
    _team_vs_oracle(O, oracle_lib, hostsim, 4, mid, 78, 123456789012, 1)
    _team_vs_oracle(O, oracle_lib, hostsim, 4, fin, 3, 9, 40)


def test_lane_list_emission(O, oracle_lib, hostsim, golden):
    """xq_rollout_lane.cuh (legal_moves_lane_kernel): register-resident generator + reference-order emission == the oracle's ordered
    lists on reachable positions over whole games (both colours, captured pieces, finished boards keep their lists), on arbitrary
    boards with a standard piece set (the others are flagged for the generic kernel) and on the golden positions"""
    for recs in (harvest_positions(O, 800, 45, 5), random_boards(O, 4000, seed=21), recs_from_codes(O, golden["pos_codes"], golden["pos_meta"])):
        n = len(recs)
        c1, a1 = _oracle_lists(oracle_lib, recs)
        c2 = np.zeros(n, np.uint8)
        a2 = np.zeros((n, 128), np.uint16)
        nonstd = hostsim.hs_lane_all_actions(recs.ctypes.data, n, c2.ctypes.data, a2.ctypes.data)
        std = c2 != 0xFF
        assert nonstd == int((~std).sum()) and std.sum() > 500
        bad = np.nonzero(std & ((c1 != c2) | (a1 != a2).any(1)))[0]
        assert len(bad) == 0, f"{len(bad)} boards differ, first {bad[:4]}"


def test_team_list_emission(O, oracle_lib, hostsim, golden):
    """xq_act_team.cuh (legal_moves_team_kernel): the team's generator (team_unpack_side per colour, team_phase_a) + team_emit_actions ==
    the oracle's ordered lists -- same cases as the board-per-thread list kernel"""
    for recs in (harvest_positions(O, 800, 45, 5), random_boards(O, 4000, seed=21), recs_from_codes(O, golden["pos_codes"], golden["pos_meta"])):
        n = len(recs)
        c1, a1 = _oracle_lists(oracle_lib, recs)
        c2 = np.zeros(n, np.uint8)
        a2 = np.zeros((n, 128), np.uint16)
        nonstd = hostsim.hs_team_all_actions(recs.ctypes.data, n, c2.ctypes.data, a2.ctypes.data)
        std = c2 != 0xFF
        assert nonstd == int((~std).sum()) and std.sum() > 500
        bad = np.nonzero(std & ((c1 != c2) | (a1 != a2).any(1)))[0]
        assert len(bad) == 0, f"{len(bad)} boards differ, first {bad[:4]}"


def test_summarize_words(O, hostsim):
    """xq_bitboard.cuh: summarize_words (step_kernel's material / General search on the packed nibble words, bit-plane SIMD) == a plain
    per-square scan -- reachable positions, arbitrary piece sets (several Generals, none), full and empty boards, padding nibbles ignored"""
    recs = np.concatenate([harvest_positions(O, 500, 6, 37, seed=8), random_boards(O, 5000, seed=33, max_pieces=60), O.new_envs(3)])
    recs["sq"][-1] = 0                                        # empty board
    recs["sq"][-2] = np.uint32(0x88888888)                    # a Black General on every square; the padding nibbles of word 11 must not count ...
    recs["sq"][-2, 11] = np.uint32(0x00000088)                # ... so they are kept zero, as every record has them
    n = len(recs)
    out = np.zeros((n, 4), np.int32)
    hostsim.hs_summarize_words(recs.ctypes.data, n, out.ctypes.data)
    score = np.array([0, 1000, 20, 20, 40, 90, 45, 10, 1000, 20, 20, 40, 90, 45, 10, 0])
    sq = recs["sq"]
    codes = np.stack([(sq[:, s >> 3] >> (4 * (s & 7))) & 15 for s in range(90)], 1).astype(np.int64)
    mat_red = (score[codes] * ((codes >= 1) & (codes <= 7))).sum(1)
    mat_black = (score[codes] * (codes >= 8)).sum(1)
    first = lambda c: np.where((codes == c).any(1), (codes == c).argmax(1), 127)
    assert (out[:, 0] == mat_red).all() and (out[:, 1] == mat_black).all()
    assert (out[:, 2] == first(1)).all() and (out[:, 3] == first(8)).all()
    assert out[-2, 1] == 90 * 1000 and out[-2, 3] == 0 and out[-1].tolist() == [0, 0, 127, 127]


def test_lane_rollout_ply(O, oracle_lib, hostsim):
    """xq_rollout_lane.cuh (rollout_lane_kernel): the board-per-thread ply run on the host reproduces the oracle's fused rollout record
    for record -- same cases as the team kernel (from the opening over several games, resumed mid-game, finished boards)"""
    mid = harvest_positions(O, 600, 6, 37, seed=5)
    fin = O.new_envs(8)
    fin["move_count"][:4] = 200
    fin["sq"][4:, 0] &= np.uint32(0xFFF0FFFF)
    _team_vs_oracle(O, oracle_lib, hostsim, 1, O.new_envs(1500), 11, 5000, 450)
    _team_vs_oracle(O, oracle_lib, hostsim, 1, mid, 77, 0, 230)
    _team_vs_oracle(O, oracle_lib, hostsim, 1, mid, 78, 123456789012, 1)
    _team_vs_oracle(O, oracle_lib, hostsim, 1, fin, 3, 9, 40)


def test_team_act_selection(O, oracle_lib, hostsim):
    """xq_act_team.cuh (act_team_kernel): eps-greedy choice of the team phases == the oracle's selectAction restatement on the same
    Q values and draws -- random Q, heavily tied Q (first maximum in list order must win), reachable and arbitrary standard boards"""
    recs = harvest_positions(O, 500, 8, 23, seed=12)
    n = len(recs)
    counts, lists = _oracle_lists(oracle_lib, recs)
    rng = np.random.default_rng(9)
    ids = np.arange(n, dtype=np.uint64) + np.uint64(31)
    for case, eps in (("random", 0.1), ("ties", 0.0), ("coarse", 0.3), ("signed zero", 0.0), ("explore", 1.0)):
        q = rng.uniform(-0.3, 0.3, (n, 96)).astype(np.float32)
        if case == "ties":
            q[:] = 0.125
        elif case == "coarse":
            q = np.round(q * 8).astype(np.float32) / 8
        elif case == "signed zero":
            q = np.where(rng.integers(0, 2, (n, 96)) == 1, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
        thr = oracle_lib.xqo_eps_threshold(eps)
        x = O.rng_np(77, ids, recs["ctr"])
        coin, idx = (x & np.uint64(0x7FFFFFFF)).astype(np.uint32), (x >> np.uint64(33)).astype(np.uint32)
        want = np.zeros(n, np.uint16)
        for i in range(n):
            qi = np.zeros(8100); qi[:96] = q[i]
            want[i] = lists[i, oracle_lib.xqo_select_action(qi, lists[i], int(counts[i]), int(coin[i]), int(idx[i]), eps)]
        for name, fn in (("team", hostsim.hs_act_team), ("lane", hostsim.hs_act_lane)):      # act_team_kernel's phases; the board-per-thread functions of xq_rollout_lane.cuh
            got = np.zeros(n, np.uint16)
            assert fn(recs.ctypes.data, n, 31, 77, q.ctypes.data, thr, got.ctypes.data) == 0
            bad = np.nonzero(got != want)[0]
            assert len(bad) == 0, (name, case, len(bad), int(bad[0]), int(got[bad[0]]) >> 7, int(got[bad[0]]) & 127, int(want[bad[0]]) >> 7, int(want[bad[0]]) & 127)


def test_team_phases_under_sanitizers(tmp_path):
    """the device source of the team kernels, compiled for the host with -fsanitize=address,undefined, runs clean"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = str(tmp_path / "libxq_hostsim_asan.so")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fPIC", "-shared",
                    "-Wno-unknown-pragmas", "-o", so, os.path.join(root, "tests", "hostsim", "hostsim.cpp")], check=True)
    pre = ":".join(subprocess.run(["g++", f"-print-file-name={n}"], capture_output=True, text=True, check=True).stdout.strip() for n in ("libasan.so", "libubsan.so"))
    env = dict(os.environ, LD_PRELOAD=pre, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "hostsim", "asan_run.py"), so], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "asan/ubsan clean" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_fixed_point_layer0_table(hostsim):
    """The acting path carries the layer-0 sum in int32 fixed point (xq_act_quant.cuh: the device functions, compiled for the host).  For weight
    scales from 1e-30 to 1e30 a sum over up to 90 rows + bias (a) never leaves the int32 range -- checked against an int64 sum of the same
    entries -- and (b) equals the FP64 sum to the quantum: |sum * 2^-k - exact| <= one half-quantum per term, a quantum being < 1.8e-7 of the largest weight.
    Non-finite and all-zero weights give a defined scale and defined (saturated / zero) entries."""
    rng = np.random.default_rng(4)
    n_rows, hid = 1260, 128
    for scale in (1e-30, 1e-12, 1e-3, 0.05, 1.0, 37.0, 1e6, 1e30):
        w = (rng.uniform(-scale, scale, (n_rows + 1, hid))).astype(np.float32)          # last row = the bias
        q = np.zeros_like(w, dtype=np.int32)
        k = hostsim.hs_act_quant(w.ctypes.data, w.size, q.ctypes.data)
        assert -100 <= k <= 124
        wmax = float(np.abs(w).max())
        assert 92.0 * wmax * 2.0 ** k < 2.0 ** 30 and (k == 124 or 92.0 * wmax * 2.0 ** k >= 2.0 ** 29), (scale, k)      # the largest scale that fits
        assert np.abs(q.astype(np.float64) - w.astype(np.float64) * 2.0 ** k).max() <= 0.5                              # rint
        for pieces in (1, 32, 90):
            rows = np.concatenate([rng.choice(n_rows, pieces, replace=False), [n_rows]])
            s64 = q[rows].astype(np.int64).sum(axis=0)
            s32 = q[rows].sum(axis=0, dtype=np.int32)                                    # wrap-around arithmetic, as on the device
            assert (s64 == s32).all() and np.abs(s64).max() < 2 ** 30, (scale, pieces)
            exact = w[rows].astype(np.float64).sum(axis=0)
            assert np.abs(s64 * 2.0 ** -k - exact).max() <= (pieces + 1) * 0.5 * 2.0 ** -k
            assert np.abs(s64 * 2.0 ** -k - exact).max() <= (pieces + 1) * 1e-7 * wmax          # a quantum is < 1.8e-7 of the largest weight
        # carried == gathered: remove a row, add another one, in any order (integer sums are associative)
        rows = list(rng.choice(n_rows, 30, replace=False))
        z = q[rows].sum(axis=0, dtype=np.int32)
        z2 = z - q[rows[3]] + q[7] - q[rows[11]]
        rows2 = [r for i, r in enumerate(rows) if i not in (3, 11)] + [7]
        assert (z2 == q[rows2].sum(axis=0, dtype=np.int32)).all()
    for special in (np.zeros(8, np.float32), np.array([np.inf, 1, -2], np.float32), np.array([np.nan, 0.5], np.float32),
                    np.array([3.4e38, -3.4e38, 1.0], np.float32)):
        q = np.zeros(len(special), np.int32)
        k = hostsim.hs_act_quant(special.ctypes.data, len(special), q.ctypes.data)
        assert -100 <= k <= 124
