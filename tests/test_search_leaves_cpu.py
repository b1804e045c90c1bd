"""CPU suite for the multi-leaf selection: the helpers of xq_search.cuh compiled for the host (tests/hostsim/search_leaves_shim.cpp, with
-ffp-contract=off) against the numpy restatement in search_leaves_oracle.py -- the virtual-loss score bit for bit (random inputs, N = 0,
fpu ties, c_puct = 0, vl = 0), its reduction to the plain score at no in-flight descent, and the select kernel's per-node in-flight
counting over synthetic trees against the definition by node paths."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import search_leaves_oracle as SL
import search_oracle as S
from conftest import ROOT


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("search_leaves_shim") / "libxq_search_leaves_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "search_leaves_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.sl_puct_vl.argtypes = [V, V, V, V, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, V]
    H.sl_puct.argtypes = [V, V, V, C.c_int, C.c_float, C.c_float, C.c_int, V]
    H.sl_inflight.argtypes = [V, C.c_int, C.c_int, V, V]
    return H


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32).tolist()


@pytest.mark.parametrize("quantised", [False, True])
def test_puct_vl_bit_exact(shim, quantised):
    rng = np.random.default_rng(11 + quantised)
    ties = 0
    for trial in range(3000):
        n = int(rng.integers(1, 129))
        if quantised:            # few distinct values: equal scores everywhere, fpu equal to visited Q
            p = (rng.integers(0, 4, n) / 8).astype(np.float32)
            nv = rng.integers(0, 3, n).astype(np.int32)
            w = (rng.integers(-2, 3, n) * nv / 2).astype(np.float32)
            c = rng.integers(0, 2, n).astype(np.int32)
        else:
            p = rng.dirichlet(np.full(n, 0.3)).astype(np.float32)
            nv = rng.integers(0, 40, n).astype(np.int32)
            w = (rng.uniform(-1, 1, n) * nv).astype(np.float32)
            c = np.where(rng.random(n) < 0.3, rng.integers(1, 32, n), 0).astype(np.int32)
        if trial % 7 == 0:
            nv[:] = 0; w[:] = 0                   # a fresh node
        c_puct = [0.0, 1.0, 1.5, 4.25][trial % 4]
        fpu = [0.0, -1.0, 0.5, 0.25][(trial // 4) % 4]
        vl = [0.0, 1.0, 3.0, 0.37][(trial // 16) % 4]
        c_node = int(c.sum())
        n_node = int(nv.sum()) + int(rng.integers(0, 3))
        got = np.zeros(n, np.float32)
        shim.sl_puct_vl(p.ctypes.data, nv.ctypes.data, w.ctypes.data, c.ctypes.data, n, vl, c_puct, fpu, n_node, c_node, got.ctypes.data)
        want = SL.puct_vl(p, nv, w, c, vl, c_puct, fpu, n_node, c_node)
        assert _bits(got) == _bits(want), trial
        ties += int((want == want.max()).sum() > 1)
    if quantised:
        assert ties > 500


def test_puct_vl_without_inflight_is_puct(shim):
    rng = np.random.default_rng(5)
    for trial in range(2000):
        n = int(rng.integers(1, 129))
        p = rng.dirichlet(np.full(n, 0.3)).astype(np.float32)
        nv = rng.integers(0, 40, n).astype(np.int32)
        if trial % 5 == 0:
            nv[:] = 0
        w = (rng.uniform(-1, 1, n) * nv).astype(np.float32)
        c = np.zeros(n, np.int32)
        c_puct, fpu, vl = [0.0, 1.25, 3.0][trial % 3], [0.0, -0.1, 0.3][trial % 3], [0.0, 1.0, 2.5][(trial // 3) % 3]
        n_node = int(nv.sum())
        a, b = np.zeros(n, np.float32), np.zeros(n, np.float32)
        shim.sl_puct_vl(p.ctypes.data, nv.ctypes.data, w.ctypes.data, c.ctypes.data, n, vl, c_puct, fpu, n_node, 0, a.ctypes.data)
        shim.sl_puct(p.ctypes.data, nv.ctypes.data, w.ctypes.data, n, c_puct, fpu, n_node, b.ctypes.data)
        assert _bits(a) == _bits(b), trial
        assert _bits(b) == _bits(S.puct(p, nv, w, c_puct, fpu, n_node)), trial


def test_virtual_loss_spreads_the_descents():
    """two equal edges: the first descent takes edge 0, a second one with vl > 0 takes edge 1; vl = 0 still changes U"""
    p = np.array([0.5, 0.5], np.float32)
    nv = np.array([3, 3], np.int32)
    w = np.array([0.6, 0.6], np.float32)
    c = np.array([1, 0])
    assert int(np.argmax(SL.puct_vl(p, nv, w, c, 1.0, 1.5, 0.0, 6, 1))) == 1
    assert int(np.argmax(SL.puct_vl(p, nv, w, c * 0, 1.0, 1.5, 0.0, 6, 0))) == 0


def _synthetic_tree(rng):
    """children[j] = {edge: child}; internal nodes (with children) are expanded, the others are leaves"""
    children = [dict()]
    depth = [0]
    frontier = [0]
    while frontier:
        j = frontier.pop()
        if depth[j] >= int(rng.integers(1, 9)) or len(children) > 300:
            continue
        for e in rng.choice(128, size=int(rng.integers(1, 6)), replace=False):
            children[j][int(e)] = len(children)
            children.append(dict())
            depth.append(depth[j] + 1)
            frontier.append(len(children) - 1)
    return children


def test_inflight_counting_matches_the_path_definition(shim):
    rng = np.random.default_rng(21)
    checked = 0
    for trial in range(300):
        children = _synthetic_tree(rng)
        L = int(rng.integers(2, 33))
        node_paths, edge_paths = [], []
        for _ in range(L):
            j, nodes, edges = 0, [0], []
            while children[j]:
                e = int(rng.choice(sorted(children[j]))) if rng.random() < 0.7 or not edge_paths or len(edge_paths[-1]) <= len(edges) \
                    else edge_paths[-1][len(edges)]            # often follow the previous descent
                if e not in children[j]:
                    e = sorted(children[j])[0]
                edges.append(e)
                j = children[j][e]
                nodes.append(j)
            node_paths.append(nodes)
            edge_paths.append(edges)
        dmax = max(len(e) for e in edge_paths)
        path = np.full((max(dmax, 1), 32), 255, np.uint8)
        for k, e in enumerate(edge_paths):
            path[:len(e), k] = e
        for k in range(L):
            depth = len(edge_paths[k])
            counts = np.zeros((max(depth, 1), 128), np.int32)
            c_node = np.zeros(max(depth, 1), np.int32)
            shim.sl_inflight(path.ctypes.data, k, depth, counts.ctypes.data, c_node.ctypes.data)
            for d in range(depth):
                want = SL.inflight_counts(node_paths[:k], node_paths[k][:d + 1])
                j = node_paths[k][d]
                edge_of = {c: e for e, c in children[j].items()}
                dense = np.zeros(128, np.int32)
                for child, cnt in want.items():
                    dense[edge_of[child]] = cnt
                assert counts[d].tolist() == dense.tolist(), (trial, k, d)
                assert c_node[d] == sum(want.values()), (trial, k, d)
                checked += int(c_node[d] > 0)
    assert checked > 1000
