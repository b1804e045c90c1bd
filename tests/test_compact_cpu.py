"""CPU suite for the compact action lists: the list emission of the compact kernels (tests/hostsim/compact_shim.cpp, built from the
helpers of xq_policy.cuh) against the oracle's reference-ordered lists mapped to the view (compact.py), on positions of random games with
both colours to move, arbitrary boards (the generic path) and player bytes 2 / 255."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import compact as CP
import policy_oracle as P
from conftest import ROOT, harvest_positions, random_boards


@pytest.fixture(scope="module")
def shims(tmp_path_factory):
    d = tmp_path_factory.mktemp("compact_shim")
    out = []
    for name in ("compact_shim", "policy_shim"):
        so = str(d / f"lib{name}.so")
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                        os.path.join(ROOT, "tests", "hostsim", f"{name}.cpp")], check=True)
        out.append(C.CDLL(so))
    V = C.c_void_p
    out[0].cs_actions.argtypes = [V, C.c_long, C.c_int, V, V, V]
    out[1].ps_mask.argtypes = [V, C.c_long, C.c_int, V, V]
    return out


@pytest.fixture(scope="module")
def boards(O):
    """positions of 400 random games snapshot at odd and even plies (both colours to move), arbitrary boards, player bytes 2 / 255"""
    reach = np.concatenate([harvest_positions(O, 400, 6, 7, seed=71), harvest_positions(O, 400, 6, 4, seed=72)])
    arb = random_boards(O, 1500, seed=73)
    odd = harvest_positions(O, 100, 1, 9, seed=74)
    odd["player"][:50] = 2
    odd["player"][50:] = 255
    return np.concatenate([reach, arb, odd])


def _emit(H, recs, view):
    n = len(recs)
    acts = np.zeros((n, 128), np.int32)
    counts = np.zeros(n, np.uint8)
    path = np.zeros(n, np.uint8)
    H.cs_actions(recs.ctypes.data, n, view, acts.ctypes.data, counts.ctypes.data, path.ctypes.data)
    return acts, counts, path


def test_lists_equal_oracle_both_views(oracle_lib, shims, boards):
    H, _ = shims
    for view in (0, 1):
        want, wc = CP.compact_lists(oracle_lib, boards, view)
        got, gc, path = _emit(H, boards, view)
        assert (gc == wc).all(), view
        assert (got == want).all(), (view, np.nonzero((got != want).any(1))[0][:5])
        assert (path[-100:] == 1).all() and 0.02 < path.mean() < 0.5      # both paths ran
        assert (got[-100:] == -1).all() and (gc[-100:] == 0).all()        # a player byte > 1 owns no piece


def test_list_set_is_the_legal_mask_and_padding(oracle_lib, shims, boards):
    H, Pm = shims
    counts, _ = P.oracle_lists(oracle_lib, boards)
    keep = counts < 128                                                     # lists of 128 are cut; masks are not
    for view in (0, 1):
        got, gc, _ = _emit(H, boards, view)
        mask = np.zeros((len(boards), 254), np.uint32)
        path = np.zeros(len(boards), np.uint8)
        Pm.ps_mask(boards.ctypes.data, len(boards), view, mask.ctypes.data, path.ctypes.data)
        assert (P.pack_mask(P.dense_mask(got.astype(np.int64)))[keep] == mask[keep]).all(), view
        k = np.arange(128)[None, :]
        assert ((got >= 0) == (k < gc[:, None])).all() and (got[k >= gc[:, None]] == -1).all()
        assert (np.sort(got, axis=1)[:, 1:] != np.sort(got, axis=1)[:, :-1])[np.sort(got, axis=1)[:, 1:] >= 0].all()   # no repeats


def test_side_view_rotates_black_to_move(oracle_lib, shims, boards):
    H, _ = shims
    a0, c0, _ = _emit(H, boards, 0)
    a1, c1, _ = _emit(H, boards, 1)
    assert (c0 == c1).all()
    blk = boards["player"] == 1
    assert blk.sum() > 1500 and (~blk).sum() > 1500
    live = a0 >= 0
    frm, to = a0 // 90, a0 % 90
    rot = np.where(live, (89 - frm) * 90 + (89 - to), -1)
    assert (a1[blk] == rot[blk]).all()
    assert (a1[~blk] == a0[~blk]).all()
