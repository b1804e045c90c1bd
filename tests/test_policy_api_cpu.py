"""CPU suite for the external-policy interface: the device helpers of xq_policy.cuh, compiled for the host through
tests/hostsim/policy_shim.cpp, against the oracle's lists and a float64 numpy restatement (policy_oracle.py) -- mask emission in both
views, greedy selection with forced ties, the softmax walk and its log-probability, on both the register-resident generator's path
and the generic path."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import policy_oracle as P
from conftest import ROOT, harvest_positions, random_boards


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("policy_shim") / "libxq_policy_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "policy_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.ps_mask.argtypes = [V, C.c_long, C.c_int, V, V]
    H.ps_choose.argtypes = [V, C.c_long, V, C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_uint64, V, C.c_int, V, V, V]
    return H


@pytest.fixture(scope="module")
def boards(O):
    """~20k reachable positions (both colours to move), arbitrary boards (many leave the generator: non-standard piece sets) and
    player bytes 2 / 255 (no legal action, generic path)"""
    reach = harvest_positions(O, 1000, 20, 5, seed=17)      # odd plies per snapshot: both colours to move
    arb = random_boards(O, 3000, seed=5)
    odd = harvest_positions(O, 200, 1, 9, seed=2)
    odd["player"][:100] = 2
    odd["player"][100:] = 255
    recs = np.concatenate([reach, arb, odd])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 7
    return recs


def _choose(H, recs, scores, view, pick, t, seed=9, id0=0, given=None, generic=False):
    n = len(recs)
    idx = np.zeros(n, np.int64)
    logp = np.zeros(n, np.float32)
    path = np.zeros(n, np.uint8)
    H.ps_choose(recs.ctypes.data, n, None if scores is None else scores.ctypes.data, view, pick, t, seed, id0,
                None if given is None else given.ctypes.data, 1 if generic else 0, idx.ctypes.data, logp.ctypes.data, path.ctypes.data)
    return idx, logp, path


def test_mask_emission_both_views(O, oracle_lib, shim, boards):
    counts, acts = P.oracle_lists(oracle_lib, boards)
    keep = counts < 128                               # the oracle stops its lists at 128 entries
    assert keep.mean() > 0.99
    for view in (0, 1):
        idx = P.policy_indices(boards, counts, acts, view)
        want = P.pack_mask(P.dense_mask(idx))
        got = np.zeros((len(boards), 254), np.uint32)
        path = np.zeros(len(boards), np.uint8)
        shim.ps_mask(boards.ctypes.data, len(boards), view, got.ctypes.data, path.ctypes.data)
        bad = np.nonzero(keep & (got != want).any(1))[0]
        assert len(bad) == 0, (view, bad[:5])
        assert (path[-200:] == 1).all() and 0.05 < path.mean() < 0.5      # both paths ran
        assert (got[:, -1] >> 4 == 0).all()                                # bits >= 8100 stay zero
    # the side-to-move view of a Black-to-move board is the absolute one rotated
    blk = boards["player"] == 1
    assert blk.sum() > 5000


def test_greedy_first_max_with_ties(O, oracle_lib, shim, boards):
    counts, acts = P.oracle_lists(oracle_lib, boards)
    keep = counts < 128
    rng = np.random.default_rng(3)
    for view in (0, 1):
        idx = P.policy_indices(boards, counts, acts, view)
        for chunk in np.array_split(np.arange(len(boards)), 6):
            recs = boards[chunk]
            scores = rng.integers(0, 4, (len(chunk), 8100)).astype(np.float32) / 4      # quantised: ties everywhere
            scores[rng.random(scores.shape) < 0.02] = np.nan
            scores[rng.random(scores.shape) < 0.02] = -np.inf
            scores[rng.random(scores.shape) < 0.005] = np.inf
            l = P.listed_scores(scores, idx[chunk])
            k = P.greedy(l, counts[chunk])
            want = np.where(k >= 0, idx[chunk][np.arange(len(chunk)), np.maximum(k, 0)], -1)
            for generic in (False, True):
                got, _, _ = _choose(shim, recs, scores, view, 0, 1.0, generic=generic)
                bad = np.nonzero(keep[chunk] & (got != want))[0]
                assert len(bad) == 0, (view, generic, bad[:5], got[bad[:5]], want[bad[:5]])
    # every legal score -inf or NaN: the first action in list order
    recs = boards[:300]
    c, a = P.oracle_lists(oracle_lib, recs)
    scores = np.full((300, 8100), -np.inf, np.float32)
    scores[:, ::3] = np.nan
    for pick in (0, 1):
        got, logp, _ = _choose(shim, recs, scores, 1, pick, 1.0)
        assert (got == P.policy_indices(recs, c, a, 1)[:, 0]).all() and np.isnan(logp).all()


def test_sample_walk_and_logp(O, oracle_lib, shim, boards):
    counts, acts = P.oracle_lists(oracle_lib, boards)
    keep = counts < 128
    rng = np.random.default_rng(11)
    seed, id0 = 1234, 77
    u = P.uniform(O.rng_np, seed, np.arange(len(boards)) + id0, boards["ctr"])
    n_amb = n_all = 0
    for view, t in ((0, 1.0), (1, 0.37), (1, 3.0)):
        idx = P.policy_indices(boards, counts, acts, view)
        for chunk in np.array_split(np.arange(len(boards)), 6):
            recs = boards[chunk]
            scores = (rng.standard_normal((len(chunk), 8100)) * 2).astype(np.float32)
            l = P.listed_scores(scores, idx[chunk])
            k, lp, amb = P.sample(l, counts[chunk], t, u[chunk])
            want = np.where(k >= 0, idx[chunk][np.arange(len(chunk)), np.maximum(k, 0)], -1)
            for generic in (False, True):
                got, logp, _ = _choose(shim, recs, scores, view, 1, t, seed, id0 + int(chunk[0]), generic=generic)
                ok = keep[chunk]
                bad = np.nonzero(ok & ~amb & (got != want))[0]
                assert len(bad) == 0, (view, t, generic, bad[:5])
                # ambiguous draws: a neighbour of the float64 choice in list order
                for i in np.nonzero(ok & amb & (got != want))[0]:
                    assert got[i] in idx[chunk][i, max(k[i] - 1, 0):k[i] + 2]
                # logp of the played action (float64 restatement at the action the host code played)
                kk = np.array([list(idx[chunk][i]).index(g) if g >= 0 else -1 for i, g in enumerate(got)])
                want_lp = P.logp_of(l, kk, t)
                fin = ok & (counts[chunk] > 0)
                assert np.abs(logp[fin] - want_lp[fin]).max() < 1e-5
                assert np.isnan(logp[counts[chunk] == 0]).all()
                n_amb += int((ok & amb).sum())
                n_all += int(ok.sum())
    assert n_amb < 1e-3 * n_all       # draws within 1e-5 S of a boundary are rare


def test_given_logp_and_rejection(O, oracle_lib, shim, boards):
    counts, acts = P.oracle_lists(oracle_lib, boards)
    rng = np.random.default_rng(5)
    recs = boards[:4000]
    c = counts[:4000]
    idx = P.policy_indices(recs, c, acts[:4000], 1)
    scores = (rng.standard_normal((4000, 8100)) * 2).astype(np.float32)
    played, logp_s, _ = _choose(shim, recs, scores, 1, 1, 0.8, 3, 0)
    got, logp_g, _ = _choose(shim, recs, scores, 1, 2, 0.8, given=played.copy())
    assert (got == played).all()
    fin = c > 0
    assert np.array_equal(logp_g[fin], logp_s[fin])
    # rejected: -1, 8100 and a legal index of the other view's frame that is not legal here
    bad_given = np.where(np.arange(4000) % 2 == 0, -1, 8100).astype(np.int64)
    got, logp, _ = _choose(shim, recs, scores, 1, 2, 0.8, given=bad_given)
    assert (got == -1).all() and np.isnan(logp).all()
    # without scores: the action is still checked, logp is not defined
    got, logp, _ = _choose(shim, recs, None, 1, 2, 1.0, given=played.copy())
    assert (got == played).all() and np.isnan(logp).all()
    dense = P.dense_mask(idx)
    illegal = np.array([int(np.nonzero(~dense[i])[0][i % 50]) for i in range(4000)], np.int64)
    got, _, _ = _choose(shim, recs, scores, 1, 2, 0.8, given=illegal)
    assert (got == -1).all()
