"""CPU suite for the Gumbel root search (xq_gumbel_*): the helpers of xq_search.cuh compiled for the host (tests/hostsim/gumbel_shim.cpp,
-ffp-contract=off) against the numpy restatement in gumbel_oracle.py -- the Gumbel words and draws, the top-m considered set with ties,
the Sequential Halving sequence for many (m, n), v_mix, q^ and sigma (all-equal q, no visited edge, priors underflowed to 0), the improved
policy and its integer weights, the root rule with in-flight counts and its fallback, and the action to play.  Bit for bit where the
arithmetic is explicitly rounded; logf / expf within stated margins."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import gumbel_oracle as G
from conftest import ROOT

F32 = np.float32


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("gumbel_shim") / "libxq_gumbel_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "gumbel_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.gb_draw.restype = C.c_float
    H.gb_draw.argtypes = [C.c_uint64, C.c_int]
    H.gb_rng.restype = C.c_uint64
    H.gb_rng.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
    H.gb_considered.argtypes = [V, C.c_int, C.c_int, V]
    H.gb_seq.argtypes = [C.c_int, C.c_int, C.c_int]
    H.gb_vmix.restype = C.c_float
    H.gb_vmix.argtypes = [V, V, V, C.c_int, C.c_float]
    H.gb_root_scores.argtypes = [V, V, V, V, V, C.c_int, C.c_float, C.c_float, C.c_float, V, V]
    H.gb_policy.argtypes = [V, C.c_int, V, V]
    H.gb_pick.argtypes = [V, V, V, C.c_int, C.c_int]
    H.gb_action.argtypes = [V, V, V, C.c_int]
    return H


def p_(a):
    return a.ctypes.data


def ulps(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


def random_root(rng, n):
    """(N, W, P) of a root of n edges: some visited, some not, priors with underflowed zeros"""
    N = np.where(rng.random(n) < 0.5, rng.integers(1, 40, n), 0).astype(np.int32)
    W = np.where(N > 0, (rng.uniform(-1, 1, n) * N).astype(F32), F32(0)).astype(F32)
    P = rng.dirichlet(np.full(n, 0.3)).astype(F32)
    P[rng.random(n) < 0.1] = 0
    return N, W, P


def test_gumbel_words_and_draws(shim):
    rng = np.random.default_rng(1)
    for _ in range(200):
        seed, env = (int(x) for x in rng.integers(0, 2 ** 62, 2))
        ctr = int(rng.integers(0, 2 ** 32))
        base = int(G.rng_np(seed, env, ctr))
        assert shim.gb_rng(seed, env, ctr) == base
        assert all(shim.gb_rng(base, k, 128) == int(G.rng_np(base, k, 128)) for k in range(0, 128, 17))
        g = np.array([shim.gb_draw(base, k) for k in range(128)], F32)
        want = G.gumbel_draw(base, 128)
        # one logf rounding of the inner log is amplified where -log u is near 1 (g near 0): an absolute margin of 2^-21 there
        assert (np.abs(g.astype(np.float64) - want) <= 2.0 ** -21 * np.maximum(1.0, np.abs(want))).all()
        # the double-precision draw of the same uniforms: the f32 logs are within a few ulps of it
        u = G.gumbel_u(base, 128).astype(np.float64)
        assert np.allclose(g, -np.log(-np.log(u)), rtol=2e-6, atol=2e-6)


def test_gumbel_distribution():
    """-log(-log u) of the documented uniforms is Gumbel(0, 1): mean = Euler's gamma, variance pi^2 / 6"""
    g = np.concatenate([G.gumbel_draw(int(G.rng_np(7, e, 3)), 128) for e in range(2000)]).astype(np.float64)
    assert abs(g.mean() - 0.5772156649) < 0.01 and abs(g.var() - np.pi ** 2 / 6) < 0.03


def test_top_m_with_ties(shim):
    rng = np.random.default_rng(2)
    for trial in range(3000):
        n = int(rng.integers(1, 129))
        m = int(rng.integers(1, 129))
        key = rng.normal(size=n).astype(F32)
        if trial % 3 == 0:
            key = rng.integers(0, 4, n).astype(F32)           # many ties
        if trial % 7 == 0:
            key[rng.random(n) < 0.3] = -np.inf
        out = np.zeros(n, np.uint8)
        shim.gb_considered(p_(key), n, m, p_(out))
        assert (out.astype(bool) == G.considered(key, m)).all(), (n, m)
        assert out.sum() == min(m, n)


def test_schedule_sequence(shim):
    for m in list(range(0, 20)) + [31, 32, 33, 64, 100, 127, 128]:
        for n in list(range(1, 70)) + [100, 128, 200, 256, 512, 1000, 4096]:
            want = G.sequence(m, n)
            got = [shim.gb_seq(m, n, i) for i in range(n)]
            assert got == want, (m, n)


def test_schedule_examples():
    """mctx's documented examples and the Sequential Halving shape: each phase visits the survivors equally"""
    assert G.sequence(1, 5) == [0, 1, 2, 3, 4]
    assert G.sequence(2, 6) == [0, 0, 1, 1, 2, 2]
    assert G.sequence(4, 8) == [0, 0, 0, 0, 1, 1, 2, 2]
    assert G.sequence(16, 64)[:16] == [0] * 16


def test_vmix_sigma_and_scores(shim):
    rng = np.random.default_rng(3)
    for trial in range(3000):
        n = int(rng.integers(1, 129))
        N, W, P = random_root(rng, n)
        if trial % 5 == 0:
            N[:] = 0; W[:] = 0                                 # no visited edge: v_mix = v
        if trial % 7 == 0:
            N[:] = 3; W[:] = F32(1.5)                          # all-equal q
        if trial % 11 == 0:
            P[:] = 0; P[rng.integers(0, n)] = 1                # every other prior underflowed
        vhat = F32(np.clip(rng.normal(), -1, 1))
        cv, cs = (F32(50), F32(0.1)) if trial % 2 else (F32(rng.uniform(0, 100)), F32(rng.uniform(0, 2)))
        assert np.float32(shim.gb_vmix(p_(N), p_(W), p_(P), n, vhat)).tobytes() == G.completed_q(N, W, P, vhat)[1].tobytes()
        g = rng.gumbel(size=n).astype(F32)
        with np.errstate(divide="ignore"):
            lg = np.log(P).astype(F32)
        z, sc = np.zeros(n, F32), np.zeros(n, F32)
        shim.gb_root_scores(p_(N), p_(W), p_(P), p_(g), p_(lg), n, vhat, cv, cs, p_(z), p_(sc))
        wz, wsc = G.root_scores(N, W, P, g, lg, vhat, cv, cs)
        assert z.tobytes() == wz.tobytes() and sc.tobytes() == wsc.tobytes(), trial
        sg = G.sigma(N, W, P, vhat, cv, cs)
        assert (sg >= 0).all() and (sg <= F32(F32(cv + F32(N.max())) * cs) * F32(1.0001)).all()
        if (N == 3).all() or (N == 0).all():
            assert (sg == 0).all()                             # equal completed q: q^ = 0


def test_improved_policy_and_weights(shim):
    rng = np.random.default_rng(4)
    for trial in range(2000):
        n = int(rng.integers(1, 129))
        z = (rng.normal(size=n) * rng.uniform(0.1, 20)).astype(F32)
        if trial % 6 == 0:
            z[rng.random(n) < 0.3] = -np.inf
            z[rng.integers(0, n)] = F32(0.5)
        p, w = np.zeros(n, F32), np.zeros(n, np.uint32)
        shim.gb_policy(p_(z), n, p_(p), p_(w))
        wp, ww = G.improved_policy(z)
        assert (ulps(p, wp) <= 8).all()                           # expf of host and numpy
        assert (np.abs(w.astype(np.int64) - ww) <= 8).all()                 # 8 ulps of pi' < 1 at most 8 weight units
        assert (w.astype(np.int64) == np.rint(p.astype(np.float64) * 2 ** 24)).all()       # the weight of the host's own pi'
        with np.errstate(invalid="ignore"):
            e = np.exp(z.astype(np.float64) - z.max())
        assert np.allclose(p, e / e.sum(), rtol=1e-5, atol=1e-7)
        assert abs(int(w.sum()) - 2 ** 24) <= n


def test_root_rule_with_inflight_counts_and_fallback(shim):
    rng = np.random.default_rng(5)
    fallbacks = 0
    for trial in range(5000):
        n = int(rng.integers(1, 129))
        cons = np.zeros(n, np.uint8)
        cons[rng.choice(n, int(rng.integers(1, n + 1)), replace=False)] = 1
        nv = rng.integers(0, 5, n).astype(np.int32)
        c = rng.integers(0, 3, n).astype(np.int32) * (rng.random(n) < 0.3)
        cnt = (nv + c).astype(np.int32)
        sc = rng.integers(0, 6, n).astype(F32) if trial % 2 else rng.normal(size=n).astype(F32)
        if trial % 9 == 0:
            sc[rng.random(n) < 0.5] = -np.inf
        target = int(rng.integers(0, 6))
        got = shim.gb_pick(p_(cons), p_(cnt), p_(sc), n, target)
        assert got == G.pick(cons.astype(bool), cnt, sc, target), trial
        fallbacks += not (cons.astype(bool) & (cnt == target)).any()
        assert cons[got] == 1
    assert fallbacks > 100


def test_play_rule(shim):
    rng = np.random.default_rng(6)
    for trial in range(5000):
        n = int(rng.integers(1, 129))
        cons = (rng.random(n) < 0.5).astype(np.uint8)
        nv = rng.integers(0, 4, n).astype(np.int32) * (rng.random(n) < 0.6)
        nv = nv.astype(np.int32)
        sc = rng.integers(0, 3, n).astype(F32)
        got = shim.gb_action(p_(cons), p_(nv), p_(sc), n)
        assert got == G.action(cons.astype(bool), nv, sc), trial
        if not (cons.astype(bool) & (nv > 0)).any():
            assert got == -1


def test_sequential_halving_counts():
    """the sequence, fed to the root rule with the visits it produces, gives the considered actions exactly its visit counts"""
    rng = np.random.default_rng(7)
    for m in (1, 2, 3, 5, 8, 16, 40, 128):
        for n in (1, 7, 16, 64, 200):
            cons = np.ones(m, bool)
            sc = rng.normal(size=m).astype(F32)
            nv = np.zeros(m, np.int64)
            for i, t in enumerate(G.sequence(m, n)):
                k = G.pick(cons, nv, sc, t)
                assert nv[k] == t
                nv[k] += 1
            assert nv.sum() == n


def test_improved_policy64_bounds_the_f32_mirror():
    """improved_policy64's bound holds for the f32 mirror (sigma / improved_policy) on 1 .. 128 edges: random visits and values, every
    q equal, spans of 1e-8 (the floor), priors spread over e^-110, and a sharp float64 check: the bound is at most a few per cent of
    pi' at ordinary roots"""
    rng = np.random.default_rng(0)
    F32 = np.float32
    worst = 0.0
    for t in range(1500):
        n = int(rng.integers(1, 129))
        N = rng.integers(0, 5, n) * (rng.random(n) < 0.5)
        kind = t % 4
        W = (N * rng.uniform(-1, 1, n)).astype(F32)
        vh = F32(rng.uniform(-1, 1))
        if kind == 1:
            W, vh = (-0.5 * N).astype(F32), F32(-0.5)
        if kind == 2:
            W = (N * rng.integers(0, 2, n) * F32(1e-8)).astype(F32)
        P = rng.dirichlet(np.ones(n)).astype(F32)
        if kind == 3:
            x = rng.uniform(-110, 0, n)
            P = np.exp(x - x.max()).astype(F32)
            P = (P / P.sum()).astype(F32)
        with np.errstate(divide="ignore"):
            lg = np.log(P).astype(F32)
        p32, _ = G.improved_policy((lg + G.sigma(N, W, P, vh, 50.0, 0.1)).astype(F32))
        pi, b = G.improved_policy64(N, W, P, lg, vh, 50.0, 0.1)
        err = np.abs(p32.astype(np.float64) - pi)
        assert (err <= b).all(), t
        if kind == 0 and N.sum() > 0:
            assert (b <= 0.05 * pi + 2.0 ** -126).all(), t
        live = b > 0
        if live.any():
            worst = max(worst, float((err[live] / b[live]).max()))
    assert 0 < worst < 1
