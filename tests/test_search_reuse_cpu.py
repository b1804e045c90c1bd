"""CPU suite for re-rooting the search trees (xq_search_advance): the helpers of xq_search.cuh compiled for the host
(tests/hostsim/search_reuse_shim.cpp, -ffp-contract=off) against a numpy restatement on thousands of random trees -- the membership
bitmap (the advance kernel's ballot iterated to a fixed point) and its prefix counts, the new indices, the in-place move order, the moved
node arrays and edge rows against an out-of-place compaction, and the root-noise mix bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

F32 = np.float32


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("search_reuse_shim") / "libxq_search_reuse_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "search_reuse_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.sr_membership.argtypes = [C.c_int, C.c_int, V, V, V]
    H.sr_new_index.argtypes = [V, V, C.c_int]
    H.sr_move.argtypes = [C.c_int, C.c_int, C.c_int] + [V] * 12 + [V, C.c_float, V]
    H.sr_mix.restype = C.c_float
    H.sr_mix.argtypes = [C.c_float, C.c_float, C.c_float]
    return H


def random_parents(rng, count):
    """parent[j] < j, parent[0] = -1; a mix of bushy trees, deep chains and trees with most nodes under one root child"""
    kind = rng.integers(0, 3)
    par = np.full(count, -1, np.int32)
    for j in range(1, count):
        if kind == 0:
            par[j] = rng.integers(0, j)
        elif kind == 1:
            par[j] = max(0, j - 1 - int(rng.integers(0, 3)))
        else:
            par[j] = 0 if j < 4 or rng.random() < 0.05 else rng.integers(max(1, j - 40), j)
    return par


def keep_numpy(par, m):
    """keep[j] = j == m or (j > m and keep[parent[j]])"""
    keep = np.zeros(len(par), bool)
    keep[m] = True
    for j in range(m + 1, len(par)):
        keep[j] = keep[par[j]]
    return keep


def test_membership_and_new_indices(shim):
    rng = np.random.default_rng(11)
    trees = 0
    for trial in range(3000):
        count = int(rng.integers(1, 200)) if trial % 4 else int(rng.integers(200, 3000))
        par = random_parents(rng, count)
        root_children = np.nonzero(par == 0)[0]
        ms = [0] + list(root_children) if trial % 10 == 0 else [0] + list(rng.choice(root_children, min(3, len(root_children)), replace=False)) if len(root_children) else [0]
        for m in ms:
            m = int(m)
            words = (count + 31) // 32
            bits = np.zeros(words, np.uint32)
            prefix = np.zeros(words, np.int32)
            kept = shim.sr_membership(count, m, par.ctypes.data, bits.ctypes.data, prefix.ctypes.data)
            keep = keep_numpy(par, m)
            assert kept == keep.sum(), (trial, m)
            want_bits = np.zeros(words, np.uint32)
            for j in np.nonzero(keep)[0]:
                want_bits[j >> 5] |= np.uint32(1 << (j & 31))
            assert (bits == want_bits).all(), (trial, m)
            cum = np.concatenate([[0], np.cumsum([bin(int(b)).count("1") for b in want_bits])[:-1]])
            lo = m >> 5
            assert (prefix[lo:] == cum[lo:] - cum[lo]).all(), (trial, m)
            new = np.cumsum(keep) - 1
            for j in np.nonzero(keep)[0]:
                assert shim.sr_new_index(bits.ctypes.data, prefix.ctypes.data, int(j)) == new[j]
            assert (new[keep] <= np.nonzero(keep)[0]).all()            # a kept node never moves up
            trees += 1
    assert trees > 6000


def _random_tree(rng, count):
    """the node arrays and edge rows of a random tree whose child fields agree with the parent array"""
    par = random_parents(rng, count)
    pedge = np.zeros(count, np.uint8)
    nedges = rng.integers(0, 119, count).astype(np.uint8)
    expanded = (rng.random(count) < 0.8).astype(np.uint8)
    child = np.full((count, 128), -1, np.int32)
    for j in range(1, count):
        p = par[j]
        expanded[p] = 1
        free = [k for k in range(128) if child[p, k] < 0]
        k = int(rng.choice(free[:max(int(nedges[p]), 1) + 8]))
        child[p, k] = j
        pedge[j] = k
        nedges[p] = max(int(nedges[p]), k + 1)
    arrays = dict(
        parent=par, pedge=pedge, visits=rng.integers(0, 1000, count).astype(np.int32), reward=rng.integers(-50, 50, count).astype(np.int32),
        depth=rng.integers(0, 60, count).astype(np.int32), nedges=nedges, expanded=expanded,
        P=rng.random((count, 128)).astype(F32), N=rng.integers(0, 500, (count, 128)).astype(np.int32),
        W=rng.uniform(-50, 50, (count, 128)).astype(F32), child=child, act=rng.integers(0, 8100, (count, 128)).astype(np.int16))
    # depths consistent along the parent pointers
    for j in range(1, count):
        arrays["depth"][j] = arrays["depth"][par[j]] + 1
    return arrays


def compact_numpy(a, m, noise, eps):
    """out-of-place compaction of the kept subtree: the expected node fields and, per kept expanded node, its n_edges edge slots"""
    keep = keep_numpy(a["parent"], m)
    old = np.nonzero(keep)[0]
    new = np.full(len(keep), -1, np.int64)
    new[old] = np.arange(len(old))
    out = []
    for j in old:
        root = j == m
        nd = dict(parent=-1 if root else int(new[a["parent"][j]]), pedge=0 if root else int(a["pedge"][j]), visits=int(a["visits"][j]),
                  reward=0 if root else int(a["reward"][j]), depth=int(a["depth"][j] - a["depth"][m]), nedges=int(a["nedges"][j]),
                  expanded=int(a["expanded"][j]))
        ne = int(a["nedges"][j]) if a["expanded"][j] else 0
        P = a["P"][j, :ne].copy()
        if root and noise is not None:
            # search_mix: (1 - eps) * P + eps * noise, each operation rounded to f32 in this order
            P = ((F32(1) + F32(-eps)) * P + F32(eps) * noise[a["act"][j, :ne].astype(np.int64)]).astype(F32)
        c = a["child"][j, :ne]
        nd["edges"] = dict(P=P, N=a["N"][j, :ne].copy(), W=a["W"][j, :ne].copy(), act=a["act"][j, :ne].copy(),
                           child=np.where(c >= 0, new[np.maximum(c, 0)], -1))
        out.append(nd)
    return out


@pytest.mark.parametrize("batch", [1, 2, 5])
def test_in_place_move_equals_out_of_place_compaction(shim, batch):
    rng = np.random.default_rng(20 + batch)
    moved_total = 0
    for trial in range(400 if batch == 2 else 150):
        count = int(rng.integers(2, 160)) if trial % 5 else int(rng.integers(160, 1200))
        a = _random_tree(rng, count)
        rc = np.nonzero(a["parent"] == 0)[0]
        m = int(rng.choice(rc))
        noise = rng.dirichlet(np.full(8100, 0.3)).astype(F32) if trial % 3 == 0 else None
        eps = [0.25, 0.0, 1.0, 0.4][trial % 4]
        want = compact_numpy(a, m, noise, eps)
        b = {k: v.copy() for k, v in a.items()}
        order = np.full(count, -1, np.int32)
        n = shim.sr_move(count, m, batch, *(b[k].ctypes.data for k in ("parent", "pedge", "visits", "reward", "depth", "nedges", "expanded", "P",
                                                                        "N", "W", "child", "act")),
                         None if noise is None else noise.ctypes.data, eps, order.ctypes.data)
        assert n == len(want), trial
        assert (np.diff(order[:n]) > 0).all() and order[0] == m       # increasing old index, the matched node first
        for i, nd in enumerate(want):
            got = {k: int(b[k][i]) for k in ("parent", "pedge", "visits", "reward", "depth", "nedges", "expanded")}
            assert got == {k: v for k, v in nd.items() if k != "edges"}, (trial, i)
            ne = len(nd["edges"]["N"])
            for k, v in nd["edges"].items():
                g = b[k][i, :ne]
                if k in ("P", "W"):
                    assert g.view(np.uint32).tolist() == v.view(np.uint32).tolist(), (trial, i, k)
                else:
                    assert (g == v).all(), (trial, i, k)
        moved_total += n
    assert moved_total > 1000


def test_in_place_order_never_overwrites_an_unread_slot(shim):
    """each batch is read before it is written and new <= old: replaying the move order, every written slot was read already or is
    not kept"""
    rng = np.random.default_rng(5)
    for trial in range(1500):
        count = int(rng.integers(2, 400))
        par = random_parents(rng, count)
        m = int(rng.choice(np.nonzero(par == 0)[0]))
        keep = keep_numpy(par, m)
        new = np.cumsum(keep) - 1
        for batch in (1, 2, 4):
            kept = np.nonzero(keep)[0]
            read = np.zeros(count, bool)
            for s in range(0, len(kept), batch):
                grp = kept[s:s + batch]
                read[grp] = True
                for j in grp:
                    assert read[new[j]] or not keep[new[j]], (trial, batch, j)


def test_noise_mix_bit_exact(shim):
    rng = np.random.default_rng(9)
    p = rng.random(20000).astype(F32)
    nz = rng.dirichlet(np.full(20000, 0.3)).astype(F32)
    for eps in (0.0, 0.25, 0.3, 1.0, float(F32(1 / 3))):
        got = np.array([shim.sr_mix(float(a), float(b), eps) for a, b in zip(p[:3000], nz[:3000])], F32)
        want = ((F32(1) + F32(-eps)) * p[:3000] + F32(eps) * nz[:3000]).astype(F32)
        assert got.view(np.uint32).tolist() == want.view(np.uint32).tolist(), eps
