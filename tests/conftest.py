import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


@pytest.fixture(scope="session")
def O():
    from oracle import loader
    return loader


@pytest.fixture(scope="session")
def oracle_lib(O):
    return O.oracle()


@pytest.fixture(scope="session")
def ref_lib(O):
    R = O.ref()
    if R is None:
        pytest.skip("oracle/_ref/libxq_ref.so not built (set XQ_REFERENCE_SRC to a checkout of the reference project)")
    return R


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "rules_ref.npz"))


@pytest.fixture(scope="session")
def make_golden():
    """tests/golden/make_golden.py as a module: the inputs, loops and checks the stored reference answers were made with"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg


@pytest.fixture(scope="session")
def answers():
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_answers.npz"))


@pytest.fixture(scope="session")
def hostsim():
    """tests/hostsim: the device rules header compiled for the host (test-only)."""
    import ctypes as C
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "libxq_hostsim.so")
    hdrs = [os.path.join(ROOT, "cn_chess_ai_b200", "csrc", h) for h in ("xq_rules.cuh", "xq_bitboard.cuh", "xq_rollout_team.cuh", "xq_rollout_lane.cuh", "xq_act_team.cuh", "xq_act_quant.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max([os.path.getmtime(src)] + [os.path.getmtime(h) for h in hdrs]):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so, src], check=True)
    H = C.CDLL(so)
    P = C.c_void_p
    H.hs_rng.restype = C.c_uint64
    H.hs_rng.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
    H.hs_all_actions.argtypes = [P, C.c_long, P, P]
    H.hs_all_actions_strict.argtypes = [P, C.c_long, P, P]
    H.hs_bb_all_actions.argtypes = [P, C.c_long, P, P]
    H.hs_valid_moves.argtypes = [P, C.c_int, C.c_int, P]
    H.hs_is_valid_move.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int]
    H.hs_act_team.argtypes = [P, C.c_long, C.c_uint64, C.c_uint64, P, C.c_uint32, P]
    H.hs_act_lane.argtypes = [P, C.c_long, C.c_uint64, C.c_uint64, P, C.c_uint32, P]
    H.hs_team_rollout.argtypes = [C.c_int, P, C.c_long, C.c_uint64, C.c_uint64, C.c_int, P, P]
    H.hs_lane_rollout.argtypes = [P, C.c_long, C.c_uint64, C.c_uint64, C.c_int, P, P]
    H.hs_lane_all_actions.argtypes = [P, C.c_long, P, P]
    H.hs_team_all_actions.argtypes = [P, C.c_long, P, P]
    H.hs_summarize_words.argtypes = [P, C.c_long, P]
    H.hs_act_quant.argtypes = [P, C.c_long, P]
    return H


def recs_from_codes(O, codes, meta):
    """codes [m,90] u8, meta [m,4] (moveCount, player, red, black) -> packed records"""
    m = len(codes)
    recs = np.zeros(m, O.ENV_DTYPE)
    for i in range(m):
        recs[i]["sq"] = O.pack_codes(codes[i])
    recs["move_count"] = meta[:, 0]
    recs["player"] = meta[:, 1]
    recs["red_score"] = meta[:, 2]
    recs["black_score"] = meta[:, 3]
    return recs


def random_boards(O, m, seed, max_pieces=36):
    """arbitrary (mostly unreachable) boards: random codes on random squares"""
    rng = np.random.default_rng(seed)
    codes = np.zeros((m, 90), np.uint8)
    meta = np.zeros((m, 4), np.int32)
    for i in range(m):
        k = int(rng.integers(2, max_pieces))
        pos = rng.choice(90, k, replace=False)
        codes[i, pos] = rng.integers(1, 15, k)
    meta[:, 0] = rng.integers(0, 199, m)
    meta[:, 1] = rng.integers(0, 2, m)
    meta[:, 2] = rng.integers(0, 500, m)
    meta[:, 3] = rng.integers(0, 500, m)
    return recs_from_codes(O, codes, meta)


def harvest_positions(O, n_envs, rounds, plies_per_round, seed=3):
    """positions reached by random play (oracle-driven), one snapshot per round"""
    L = O.oracle()
    envs = O.new_envs(n_envs)
    snaps = []
    for _ in range(rounds):
        st = np.zeros(1, O.STATS_DTYPE)
        L.xqo_rollout_random(envs.ctypes.data, n_envs, 0, seed, plies_per_round, None, st.ctypes.data)
        snaps.append(envs.copy())
    return np.concatenate(snaps)
