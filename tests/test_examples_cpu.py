"""CPU suite for the self-play example buffer (xq_examples_*): the helpers of xq_examples.cuh compiled for the host
(tests/hostsim/examples_shim.cpp, -ffp-contract=off) against numpy on random inputs -- the result cleaning and the z sign, the
policy-target division, the view of stored actions, the sample-index draw (oracle/loader.py: rng_np) and the commit offsets of the scan
with the env lookup of the commit kernel -- and the layout of xq_example in include/xq.h against EXAMPLE_DTYPE."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

F32 = np.float32


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("examples_shim") / "libxq_examples_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "examples_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.ex_shim_z.restype = C.c_float
    H.ex_shim_z.argtypes = [C.c_float, C.c_int]
    H.ex_shim_policy.restype = C.c_float
    H.ex_shim_policy.argtypes = [C.c_uint32, C.c_uint32]
    H.ex_shim_view_index.argtypes = [C.c_int, C.c_int, C.c_int]
    H.ex_shim_sample_index.argtypes = [C.c_uint64, C.c_uint32, C.c_int64, C.c_int64, V]
    H.ex_shim_commit_offsets.restype = C.c_int64
    H.ex_shim_commit_offsets.argtypes = [C.c_int64, C.c_int, V, V, C.c_int64, V]
    H.ex_shim_find_env.restype = C.c_int64
    H.ex_shim_find_env.argtypes = [V, C.c_int64, C.c_int64]
    return H


def z_numpy(result, player):
    r = np.where(np.isnan(result), F32(0), np.clip(result, F32(-1), F32(1))).astype(F32)
    return np.where(player == 0, r, -r).astype(F32)


def test_result_cleaning_and_z_sign(shim):
    rng = np.random.default_rng(1)
    res = np.concatenate([rng.uniform(-3, 3, 4000), [np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -1.0, 1.0000001, -0.9999999, 1e-45]]).astype(F32)
    player = rng.integers(0, 3, len(res))
    got = np.array([shim.ex_shim_z(float(r), int(p)) for r, p in zip(res, player)], F32)
    assert got.view(np.uint32).tolist() == z_numpy(res, player).view(np.uint32).tolist()


def test_policy_target_division(shim):
    rng = np.random.default_rng(2)
    tot = np.concatenate([rng.integers(1, 70000, 3000), rng.integers(1 << 24, 1 << 31, 1000), [0, 0, 1, 3]]).astype(np.uint32)
    vis = np.minimum((rng.random(len(tot)) * tot.astype(np.float64)).astype(np.uint32), tot)
    vis[-4:] = [0, 0, 1, 1]
    got = np.array([shim.ex_shim_policy(int(v), int(t)) for v, t in zip(vis, tot)], F32)
    with np.errstate(invalid="ignore", divide="ignore"):
        want = np.where(tot == 0, F32(0), vis.astype(F32) / tot.astype(F32)).astype(F32)
    assert got.view(np.uint32).tolist() == want.view(np.uint32).tolist()


def test_view_of_stored_actions(shim):
    """flip (side view, Black to move) maps from * 90 + to to (89 - from) * 90 + (89 - to), the policy_index of the rotated squares"""
    for a in range(0, 8100, 7):
        for player in (0, 1, 2):
            for view in (0, 1):
                f, t = divmod(a, 90)
                want = (89 - f) * 90 + (89 - t) if (view == 1 and player == 1) else a
                assert shim.ex_shim_view_index(a, player, view) == want


def test_sample_index_draw(shim, O):
    for seed, counter, size, batch in [(0, 0, 1, 50), (7, 3, 1000, 4096), (2**63 + 5, 2**32 - 1, 123457, 999), (11, 9, 2**40 + 3, 64),
                                       (5, 1, 0, 16)]:
        got = np.empty(batch, np.int64)
        shim.ex_shim_sample_index(seed, counter, size, batch, got.ctypes.data)
        if size == 0:
            assert (got == -1).all()
            continue
        want = ((O.rng_np(seed, np.arange(batch), np.full(batch, counter)) >> np.uint64(1)) % np.uint64(size)).astype(np.int64)
        assert (got == want).all()


@pytest.mark.parametrize("threads", [1, 7, 32, 1024])
def test_commit_offsets_and_env_lookup(shim, threads):
    rng = np.random.default_rng(threads)
    for trial in range(60):
        n = int(rng.choice([1, 2, 33, 1023, 1024, 1025, 4097, 70000])) if trial % 3 else int(rng.integers(1, 3000))
        ended = (rng.random(n) < rng.choice([0.0, 0.05, 0.5, 1.0])).astype(np.uint8)
        staged = rng.integers(0, 257, n).astype(np.uint32)
        base = int(rng.integers(0, 2**40))
        off = np.empty(n, np.int64)
        total = shim.ex_shim_commit_offsets(n, threads, ended.ctypes.data, staged.ctypes.data, base, off.ctypes.data)
        cnt = np.where(ended != 0, staged, 0).astype(np.int64)
        want = base + np.concatenate([[0], np.cumsum(cnt)[:-1]])
        assert total == cnt.sum() and (off == want).all(), (n, trial)
        # every commit number belongs to the ended env the commit kernel finds for it
        owner = np.repeat(np.arange(n), cnt)
        pos = base + np.arange(len(owner))
        for p, e in list(zip(pos, owner))[:: max(1, len(owner) // 500)]:
            assert shim.ex_shim_find_env(off.ctypes.data, n, int(p)) == e


def test_example_layout_matches_header(tmp_path):
    from cn_chess_ai_b200._lib import EXAMPLE_DTYPE
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "xq.h"\n#define F(f) printf("%s %zu\\n", #f, offsetof(xq_example, f));\n'
                   'int main(void) { printf("size %zu\\n", sizeof(xq_example));\n'
                   'F(rec) F(env) F(game) F(ply) F(n_edges) F(reserved0) F(z) F(q) F(total_visits) F(reserved1) F(action) F(visits)\n'
                   'return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(out.pop("size")) == EXAMPLE_DTYPE.itemsize == 864
    assert {k: int(v) for k, v in out.items()} == {k: EXAMPLE_DTYPE.fields[k][1] for k in out}
    assert list(out) == list(EXAMPLE_DTYPE.names)
