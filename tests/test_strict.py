"""Opt-in strict legality (xq_env_legal_moves_strict: self-check and flying-general rejection -- not a rule of the reference).
CPU: the plain-C statement (oracle) == the same statement composed from the reference's OWN classes (ref_wrap) == the device source
compiled for the host, on reachable and arbitrary positions and on hand-made known answers.  GPU: the kernel == the oracle."""
import numpy as np
import pytest

from conftest import harvest_positions, random_boards, recs_from_codes

G, A, E, H, R, C, S = 1, 2, 3, 4, 5, 6, 7      # Red codes; Black = +7


def _oracle(L, recs, strict=True):
    n = len(recs)
    counts = np.zeros(n, np.uint8)
    acts = np.zeros((n, 128), np.uint16)
    (L.xqo_batch_all_actions_strict if strict else L.xqo_batch_all_actions)(recs.ctypes.data, n, counts, acts)
    acts[np.arange(128)[None, :] >= counts[:, None]] = 0xFFFF
    return counts, acts


def _board(O, pieces, player=0):
    codes = np.zeros((1, 90), np.uint8)
    for (r, c), code in pieces.items():
        codes[0, r * 9 + c] = code
    return recs_from_codes(O, codes, np.array([[0, player, 0, 0]], np.int32))


def _pairs(counts, acts, i=0):
    return [(int(a) >> 7, int(a) & 127) for a in acts[i, :counts[i]]]


def test_known_answers(O, oracle_lib):
    # flying general: Red General (0,4) and Black General (9,4) on one file, a Red Chariot between them on (4,4)
    rec = _board(O, {(0, 4): G, (9, 4): G + 7, (4, 4): R})
    c0, a0 = _oracle(oracle_lib, rec, strict=False)
    c1, a1 = _oracle(oracle_lib, rec)
    loose, strict = _pairs(c0, a0), _pairs(c1, a1)
    off_file = [(f, t) for f, t in loose if f == 40 and t % 9 != 4]
    assert len(off_file) == 8 and all(m not in strict for m in off_file)            # the Chariot may not leave the file ...
    assert all((40, t) in strict for t in range(13, 82, 9) if t != 40)              # ... but may slide along it (and take the General)
    assert (4, 3) in strict and (4, 5) in strict and (4, 13) in strict              # the Red General steps aside or forward freely
    # self-check: a Black Chariot on (5,3) attacks the file the Red General would step onto
    rec = _board(O, {(0, 4): G, (9, 5): G + 7, (5, 3): R + 7})
    strict = _pairs(*_oracle(oracle_lib, rec))
    assert (4, 3) not in strict and (4, 5) not in strict and (4, 13) in strict      # (0,5) faces the Black General on file 5
    # a pinned Horse: it is one of two pieces between a Black Cannon and the Red General; moving it leaves exactly one screen
    rec = _board(O, {(0, 4): G, (9, 3): G + 7, (1, 4): H, (3, 4): S + 7, (5, 4): C + 7})
    c0, a0 = _oracle(oracle_lib, rec, strict=False)
    loose, strict = _pairs(c0, a0), _pairs(*_oracle(oracle_lib, rec))
    assert sum(f == 13 for f, _ in loose) == 6 and all(f != 13 for f, _ in strict)
    # a side without a General keeps every pseudo-legal action
    rec = _board(O, {(9, 4): G + 7, (4, 4): R, (2, 2): H})
    assert _pairs(*_oracle(oracle_lib, rec)) == _pairs(*_oracle(oracle_lib, rec, strict=False))
    # the opening: nothing is rejected (44 actions)
    rec = O.new_envs(1)
    assert _oracle(oracle_lib, rec)[0][0] == 44


def test_oracle_equals_reference_composition(O, oracle_lib, make_golden, answers):
    """the pin: xqo_all_actions_strict == the reference's own getAllValidActions / movePiece / getPieceAt composed the same way:
    its lists stored in tests/golden/reference_answers.npz, and live against oracle/_ref when it is built"""
    recs = make_golden.strict_positions()
    c1, a1 = _oracle(oracle_lib, recs)
    c0, _ = _oracle(oracle_lib, recs, strict=False)
    assert (c1 == answers["strict_counts"]).all() and (a1 == answers["strict_lists"]).all()
    assert int(c0.sum()) - int(c1.sum()) == int(answers["strict_rejected"]) > 50          # the filter is exercised
    ref_lib = O.ref()
    if ref_lib is None:
        return
    h = ref_lib.ref_env_new()
    buf = np.zeros(256, np.int32)
    rejected = 0
    for i in range(len(recs)):
        codes = O.codes_of(recs[i]).astype(np.uint8)
        meta = np.array([recs[i]["move_count"], recs[i]["player"], recs[i]["red_score"], recs[i]["black_score"]], np.int32)
        ref_lib.ref_env_set(h, codes, meta)
        n = ref_lib.ref_env_all_actions_strict(h, int(recs[i]["player"]), buf)
        assert n == c1[i] and ((buf[0:2 * n:2] << 7 | buf[1:2 * n:2]) == a1[i, :n]).all(), i
        rejected += ref_lib.ref_env_all_actions(h, int(recs[i]["player"]), buf) - n
    ref_lib.ref_env_free(h)
    assert rejected > 50          # the filter is exercised


def test_device_source_on_host(O, oracle_lib, hostsim):
    recs = np.concatenate([harvest_positions(O, 400, 8, 29, seed=4), random_boards(O, 3000, seed=8, max_pieces=30)])
    c1, a1 = _oracle(oracle_lib, recs)
    n = len(recs)
    c2 = np.zeros(n, np.uint8)
    a2 = np.zeros((n, 128), np.uint16)
    hostsim.hs_all_actions_strict(recs.ctypes.data, n, c2.ctypes.data, a2.ctypes.data)
    assert (c1 == c2).all() and (a1 == a2).all()
    c0, _ = _oracle(oracle_lib, recs, strict=False)
    assert (c1 <= c0).all() and (c1 < c0).sum() > 500


@pytest.mark.gpu
def test_kernel_equals_oracle(O, oracle_lib):
    import cn_chess_ai_b200 as xq
    recs = np.concatenate([harvest_positions(O, 700, 8, 27, seed=9), random_boards(O, 2500, seed=10, max_pieces=32), O.new_envs(3)])
    env = xq.BatchedEnv(len(recs))
    env.set_boards(recs)
    c, a = env.legal_moves(strict=True)
    c1, a1 = _oracle(oracle_lib, recs)
    assert (c == c1).all() and (a == a1).all()
    assert env.get_boards().tobytes() == recs.tobytes()           # the try-and-undo leaves the boards untouched
    c0, a0 = env.legal_moves()
    cl, al = _oracle(oracle_lib, recs, strict=False)
    assert (c0 == cl).all() and (a0 == al).all()
