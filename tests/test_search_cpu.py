"""CPU suite for the batched tree search: the helpers of xq_search.cuh compiled for the host (tests/hostsim/search_shim.cpp, with
-ffp-contract=off) against the numpy restatement in search_oracle.py -- PUCT scores and the selection order bit for bit (random inputs,
forced ties, N = 0, fpu ties, c_puct = 0), the warp reduction of the select kernel, the backup's signs and value cleaning, and the priors
of an expansion against a float64 softmax."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import search_oracle as S
from conftest import ROOT


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("search_shim") / "libxq_search_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "search_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.ss_puct.argtypes = [V, V, V, C.c_int, C.c_float, C.c_float, C.c_int, V]
    H.ss_select_warp.argtypes = [V, V, V, C.c_int, C.c_float, C.c_float, C.c_int]
    H.ss_priors.argtypes = [V, C.c_int, C.c_float, V, C.c_float, V]
    H.ss_clean_value.restype = C.c_float
    H.ss_clean_value.argtypes = [C.c_float]
    H.ss_backup.argtypes = [C.c_int, C.c_float, V, V, V, V, V]
    return H


def _edges(rng, n, quantised):
    if quantised:      # few distinct values: equal scores everywhere
        p = (rng.integers(0, 4, n) / 8).astype(np.float32)
        nv = rng.integers(0, 3, n).astype(np.int32)
        w = (rng.integers(-2, 3, n) * nv / 2).astype(np.float32)
    else:
        p = rng.dirichlet(np.full(n, 0.3)).astype(np.float32)
        nv = rng.integers(0, 40, n).astype(np.int32)
        w = (rng.uniform(-1, 1, n) * nv).astype(np.float32)
    return p, nv, w


@pytest.mark.parametrize("quantised", [False, True])
def test_puct_and_selection_bit_exact(shim, quantised):
    rng = np.random.default_rng(7 + quantised)
    cases = 0
    for trial in range(3000):
        n = int(rng.integers(1, 129))
        p, nv, w = _edges(rng, n, quantised)
        c_puct = [0.0, 1.0, 1.5, 4.25][trial % 4]
        fpu = [0.0, -1.0, 0.5, 0.25][(trial // 4) % 4]
        if trial % 7 == 0:
            nv[:] = 0; w[:] = 0                       # a fresh node: every Q is fpu
        n_node = int(nv.sum()) + int(rng.integers(0, 3))
        got = np.zeros(n, np.float32)
        shim.ss_puct(p.ctypes.data, nv.ctypes.data, w.ctypes.data, n, c_puct, fpu, n_node, got.ctypes.data)
        want = S.puct(p, nv, w, c_puct, fpu, n_node)
        assert got.view(np.uint32).tolist() == want.view(np.uint32).tolist(), trial
        k = shim.ss_select_warp(p.ctypes.data, nv.ctypes.data, w.ctypes.data, n, c_puct, fpu, n_node)
        assert k == S.select_edge(p, nv, w, c_puct, fpu, n_node), trial
        cases += int((want == want.max()).sum() > 1)
    if quantised:
        assert cases > 500            # ties were exercised, many of them across lanes


def test_selection_ties_go_to_the_smaller_index(shim):
    for n in (1, 2, 31, 32, 33, 64, 100, 128):
        p = np.full(n, 1.0 / n, np.float32)
        nv = np.zeros(n, np.int32)
        w = np.zeros(n, np.float32)
        for c_puct, fpu in ((0.0, 0.0), (1.0, 0.0), (0.0, -1.0)):
            assert shim.ss_select_warp(p.ctypes.data, nv.ctypes.data, w.ctypes.data, n, c_puct, fpu, 0) == 0
        # the maximum placed at one index, equal maxima further on
        for at in {0, n // 3, n - 1}:
            q = p.copy()
            q[at:] = 2.0 / n
            assert shim.ss_select_warp(q.ctypes.data, nv.ctypes.data, w.ctypes.data, n, 1.0, 0.0, 1) == at
    # fpu equal to a visited edge's Q: the smaller index wins either way
    p = np.array([0.0, 0.0, 0.0], np.float32)
    nv = np.array([0, 2, 0], np.int32)
    w = np.array([0.0, 1.0, 0.0], np.float32)        # Q = 0.5 at index 1
    assert shim.ss_select_warp(p.ctypes.data, nv.ctypes.data, w.ctypes.data, 3, 1.0, 0.5, 2) == 0
    nv2, w2 = np.array([2, 0, 0], np.int32), np.array([1.0, 0.0, 0.0], np.float32)
    assert shim.ss_select_warp(p.ctypes.data, nv2.ctypes.data, w2.ctypes.data, 3, 1.0, 0.5, 2) == 0


def test_value_cleaning(shim):
    for v, want in ((np.nan, 0.0), (np.inf, 1.0), (-np.inf, -1.0), (3.0, 1.0), (-2.5, -1.0), (0.25, 0.25), (-1.0, -1.0), (-0.0, 0.0)):
        assert shim.ss_clean_value(v) == want
        assert S.clean_value(v) == want


def test_backup_signs(shim):
    """a chain root -> 1 -> 2 -> 3 and a sibling 4 of node 2: the edge into the leaf gets -v, the next one up +v, ..."""
    parent = np.array([-1, 0, 1, 2, 1], np.int32)
    pedge = np.array([0, 5, 3, 0, 7], np.uint8)
    rng = np.random.default_rng(1)
    for leaf, value in ((3, 0.75), (3, np.nan), (4, 7.0), (2, -0.3), (0, 0.5)):
        visits = rng.integers(0, 5, 5).astype(np.int32)
        en = rng.integers(0, 5, (5, 128)).astype(np.int32)
        ew = rng.uniform(-2, 2, (5, 128)).astype(np.float32)
        v0, n0, w0 = visits.copy(), en.copy(), ew.copy()
        shim.ss_backup(leaf, value, parent.ctypes.data, pedge.ctypes.data, visits.ctypes.data, en.ctypes.data, ew.ctypes.data)
        v = S.clean_value(value)
        j, want_v, want_n, want_w = leaf, v0.copy(), n0.copy(), w0.copy()
        want_v[j] += 1
        while j > 0:
            p = parent[j]
            v = np.float32(-v)
            want_n[p, pedge[j]] += 1
            want_w[p, pedge[j]] = np.float32(want_w[p, pedge[j]] + v)
            want_v[p] += 1
            j = p
        assert (visits == want_v).all() and (en == want_n).all() and ew.view(np.uint32).tolist() == want_w.view(np.uint32).tolist()
    # the sign: one backup of +1 from a leaf two plies down is +1 on the root's edge (same side to move as the leaf), -1 one ply down
    visits, en, ew = np.zeros(5, np.int32), np.zeros((5, 128), np.int32), np.zeros((5, 128), np.float32)
    shim.ss_backup(2, 1.0, parent.ctypes.data, pedge.ctypes.data, visits.ctypes.data, en.ctypes.data, ew.ctypes.data)
    assert ew[1, 3] == -1.0 and ew[0, 5] == 1.0 and visits.tolist() == [1, 1, 1, 0, 0]


def test_priors_against_float64(shim):
    rng = np.random.default_rng(4)
    for trial in range(2000):
        n = int(rng.integers(1, 129))
        raw = (rng.standard_normal(n) * 1.5).astype(np.float32)
        kind = trial % 6
        if kind == 1:
            raw[rng.random(n) < 0.2] = np.nan
        elif kind == 2:
            raw[rng.random(n) < 0.2] = -np.inf
        elif kind == 3:
            raw[:] = -np.inf
            raw[rng.random(n) < 0.3] = np.nan          # every legal score -inf or NaN: uniform
        elif kind == 4:
            raw[int(rng.integers(0, n))] = np.inf      # +inf -> FLT_MAX: all mass on it (and on any tie)
        t = [1.0, 0.5, 2.0][trial % 3]
        noise = rng.dirichlet(np.full(n, 0.3)).astype(np.float32) if trial % 5 == 0 else None
        eps = 0.25
        got = np.zeros(n, np.float32)
        shim.ss_priors(raw.ctypes.data, n, t, None if noise is None else noise.ctypes.data, eps, got.ctypes.data)
        want = S.priors64(raw, t, noise, eps)
        err = np.abs(got - want) / np.maximum(want, 1e-30)
        big = want > 1e-30
        # 1e-6, plus the f32 rounding of (l - m) / T, which exp turns into a relative error of |l - m| / T ulps
        l = S.P.clean(raw)
        with np.errstate(invalid="ignore"):
            arg = np.where(np.isfinite(l) & np.isfinite(l.max()), np.abs(l - l.max()) / t, 0.0)
        tol = 1e-6 + 2.0 ** -23 * arg
        assert (err[big] <= tol[big]).all(), (trial, kind, err.max())
        assert (got[~big] < 1e-30).all()
        if kind == 3 and noise is None:
            assert (got == np.float32(1.0 / n)).all()
