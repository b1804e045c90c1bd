"""CPU suite for reanalyse (xq_examples_load_device / xq_examples_refresh_device): the status rule of xq_examples.cuh compiled for the host
(tests/hostsim/reanalyse_shim.cpp) -- the claim phase (the smallest row per slot) and each row's status -- against a numpy statement of
the rule on random index vectors with -1, indices >= size, many duplicates, stale slots and unsearched roots; and the status values
against include/xq.h and torch_examples."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT

REFRESHED, NO_SLOT, DUPLICATE, STALE, UNSEARCHED = 0, 1, 2, 3, 4
NO_CLAIM = 0xFFFFFFFF


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("reanalyse_shim") / "libxq_reanalyse_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "reanalyse_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.ex_shim_refresh_statuses.argtypes = [C.c_int64, V, C.c_int64, V, V, V, V]
    H.ex_shim_refresh_status.restype = C.c_uint8
    H.ex_shim_refresh_status.argtypes = [C.c_int64, C.c_int64, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32]
    return H


def statuses_numpy(index, size, stale, total):
    """the rule of include/xq.h: NO_SLOT for an index outside [0, size), DUPLICATE for every row but the first with its index, then
    STALE, then UNSEARCHED (no visit or weight), else REFRESHED"""
    out = np.empty(len(index), np.uint8)
    first = {}
    for t, i in enumerate(index.tolist()):
        if i < 0 or i >= size:
            out[t] = NO_SLOT
        elif first.setdefault(i, t) != t:
            out[t] = DUPLICATE
        elif stale[t]:
            out[t] = STALE
        else:
            out[t] = REFRESHED if total[t] else UNSEARCHED
    return out


def run_shim(shim, index, size, stale, total, capacity):
    claim = np.full(capacity, NO_CLAIM, np.uint32)
    status = np.empty(len(index), np.uint8)
    shim.ex_shim_refresh_statuses(len(index), index.ctypes.data, size, stale.ctypes.data, total.ctypes.data, claim.ctypes.data,
                                  status.ctypes.data)
    return status, claim


@pytest.mark.parametrize("m", [1, 7, 256, 4096])
def test_status_rule_against_numpy(shim, m):
    rng = np.random.default_rng(m)
    for trial in range(40):
        capacity = int(rng.choice([1, 5, 64, 1000, 1 << 16]))
        size = int(rng.integers(0, capacity + 1)) if trial % 4 else capacity
        kind = trial % 5
        if kind == 0:       # many duplicates: a few slots
            index = rng.integers(0, max(1, min(size, 3)), m)
        elif kind == 1:     # the edges of the valid range
            index = rng.choice(np.array([-1, 0, size - 1, size, capacity, capacity + 5, -(1 << 40), 1 << 40]), m)
        elif kind == 2:     # a sweep
            index = np.arange(m) % max(size, 1)
        else:               # random, a share out of range
            index = rng.integers(-3, capacity + 3, m)
        index = index.astype(np.int64)
        stale = (rng.random(m) < rng.choice([0.0, 0.1, 0.5])).astype(np.uint8)
        total = np.where(rng.random(m) < 0.2, 0, rng.integers(1, 1 << 24, m)).astype(np.uint32)
        status, claim = run_shim(shim, index, size, stale, total, capacity)
        want = statuses_numpy(index, size, stale, total)
        assert (status == want).all(), (m, trial, np.nonzero(status != want)[0][:5])
        assert (claim == NO_CLAIM).all()                       # every winner restored its slot's word
        held = (index >= 0) & (index < size)
        assert (status[~held] == NO_SLOT).all()
        # one writer at most per slot, and it is the first row with that index
        writers = index[status == REFRESHED]
        assert len(np.unique(writers)) == len(writers)


def test_status_rule_single_row(shim):
    """the row-level rule: the order of the checks, and that a row never wins a word held by another row or by nobody"""
    f = shim.ex_shim_refresh_status
    assert f(-1, 10, 0, 0, 1, 0) == NO_SLOT and f(10, 10, 0, 0, 0, 5) == NO_SLOT and f(0, 0, 0, 0, 0, 5) == NO_SLOT
    assert f(3, 10, 2, 5, 1, 0) == DUPLICATE and f(3, 10, NO_CLAIM, 5, 0, 7) == DUPLICATE
    assert f(3, 10, 5, 5, 1, 0) == STALE and f(3, 10, 5, 5, 0, 0) == UNSEARCHED and f(3, 10, 5, 5, 0, 1) == REFRESHED


def test_status_values_match_header():
    text = open(os.path.join(ROOT, "include", "xq.h")).read()
    got = {k: int(v) for k, v in re.findall(r"(XQ_REFRESH\w*) = (\d+)", text)}
    assert got == {"XQ_REFRESHED": REFRESHED, "XQ_REFRESH_NO_SLOT": NO_SLOT, "XQ_REFRESH_DUPLICATE": DUPLICATE, "XQ_REFRESH_STALE": STALE,
                   "XQ_REFRESH_UNSEARCHED": UNSEARCHED}
    pytest.importorskip("torch")
    from cn_chess_ai_b200 import torch_examples as te
    assert (te.REFRESHED, te.NO_SLOT, te.DUPLICATE, te.STALE, te.UNSEARCHED) == (REFRESHED, NO_SLOT, DUPLICATE, STALE, UNSEARCHED)
