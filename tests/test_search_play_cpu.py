"""CPU suite for playing self-play moves from the search and for the library's root noise (xq_search_play_device,
xq_search_root_noise_device): the helpers of xq_search.cuh compiled for the host (tests/hostsim/search_play_shim.cpp, -ffp-contract=off)
against numpy -- the visit-count choice bit for bit at temperature 1 and outside rounding margins at other temperatures, the log-Gamma draw
against a float64 restatement of the same random words, and the distributions against scipy (Gamma, and the Beta marginals of the
Dirichlet draw), all with fixed seeds."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

from conftest import ROOT

F32 = np.float32


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("search_play_shim") / "libxq_search_play_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "search_play_shim.cpp")], check=True)
    H = C.CDLL(so)
    V = C.c_void_p
    H.sp_sample.argtypes = [V, C.c_int, C.c_float, C.c_float, V]
    H.sp_uniform.restype = C.c_float
    H.sp_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
    H.sp_rng.restype = C.c_uint64
    H.sp_rng.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
    H.sp_dirichlet.argtypes = [C.c_uint64, C.c_int, C.c_float, V, V]
    return H


def rng_np(seed, env, ctr):
    """xq_rng on uint64 arrays (wrapping arithmetic)"""
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + np.asarray(env, np.uint64) * np.uint64(0x9E3779B97F4A7C15)
             + np.asarray(ctr, np.uint64) * np.uint64(0xD1B54A32D192ED03))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def sample_numpy(visits, tau, u):
    """(edge, weights, running sums, threshold) of the play kernel's sampled choice in float32"""
    n = visits.astype(np.int64)
    nmax = n.max()
    if tau == 1.0:
        w = n.astype(F32)
    else:
        with np.errstate(divide="ignore"):
            w = np.where(n > 0, np.exp(np.log(F32(n) / F32(nmax)) / F32(tau)), 0).astype(F32)
    run = np.cumsum(w, dtype=F32)
    thr = F32(u) * run[-1]
    hit = np.nonzero(run > thr)[0]
    k = int(hit[0]) if len(hit) else int(np.nonzero(w > 0)[0][-1])
    return k, w, run, thr


def random_visits(rng, n):
    kind = rng.integers(0, 3)
    if kind == 0:
        v = rng.integers(0, 5, n)
    elif kind == 1:
        v = rng.geometric(0.05, n) - 1
    else:
        v = np.zeros(n, np.int64)
        v[rng.integers(0, n, 3)] = rng.integers(1, 10000, 3)
    if v.max() == 0:
        v[rng.integers(0, n)] = 1
    return v.astype(np.int32)


def test_visit_choice_at_temperature_one_is_bit_exact(shim):
    rng = np.random.default_rng(5)
    for trial in range(4000):
        n = int(rng.integers(1, 129))
        visits = random_visits(rng, n)
        if trial % 50 == 0:
            visits[:] = 0
            visits[rng.integers(0, n)] = (1 << 24) - n      # the largest total a search can make
        seed, env, ctr = (int(x) for x in rng.integers(0, 1 << 62, 3))
        u = shim.sp_uniform(seed, env, ctr & 0xFFFFFFFF)
        assert u == F32(int(rng_np(seed, env, ctr & 0xFFFFFFFF)) >> 40) * F32(2.0 ** -24)
        w = np.zeros(n, F32)
        k = shim.sp_sample(visits.ctypes.data, n, 1.0, u, w.ctypes.data)
        want, w_np, _, _ = sample_numpy(visits, 1.0, u)
        assert k == want, trial
        assert w.tobytes() == w_np.tobytes()
        assert visits[k] > 0


def test_visit_choice_at_other_temperatures_outside_margins(shim):
    rng = np.random.default_rng(6)
    close = total = 0
    for tau in (0.25, 0.5, 2.0):
        for trial in range(2000):
            n = int(rng.integers(1, 129))
            visits = random_visits(rng, n)
            u = float(F32(int(rng.integers(0, 1 << 24)) * 2.0 ** -24))
            w = np.zeros(n, F32)
            k = shim.sp_sample(visits.ctypes.data, n, tau, u, w.ctypes.data)
            want, w_np, run, thr = sample_numpy(visits, tau, u)
            assert np.allclose(w, w_np, rtol=2e-5, atol=0), (tau, trial)
            assert visits[k] > 0
            total += 1
            if np.any(np.abs(run - thr) <= 1e-5 * max(float(run[-1]), 1e-30)):
                close += 1
                continue
            assert k == want, (tau, trial)
    assert close < total * 0.01, (close, total)


def test_no_visits_samples_nothing(shim):
    w = np.zeros(4, F32)
    assert shim.sp_sample(np.zeros(4, np.int32).ctypes.data, 4, 1.0, 0.5, w.ctypes.data) == -1
    v = np.array([0, 3, 0, 0], np.int32)
    for u in (0.0, 0.5, 1.0 - 2 ** -24):
        for tau in (1.0, 0.3, 4.0):
            assert shim.sp_sample(v.ctypes.data, 4, tau, u, w.ctypes.data) == 1


def u24(x, lo):
    return ((x >> np.uint64(lo)) & np.uint64(0xFFFFFF)).astype(np.float64) * 2.0 ** -24 + 2.0 ** -24


def log_gamma64(base, n, alpha, tries=32):
    """float64 restatement of search_log_gamma on the same words: (lg [n], near [n] = an acceptance test within 1e-5 of its threshold)"""
    k = np.arange(n, dtype=np.uint64)
    d = alpha + 1.0 - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    v = np.ones(n)
    done = np.zeros(n, bool)
    near = np.zeros(n, bool)
    for i in range(tries):
        xn = rng_np(base, k, 1 + 2 * i)
        z = np.sqrt(-2.0 * np.log(u24(xn, 40))) * np.cos(2.0 * np.pi * u24(xn, 16))
        cand = (1.0 + c * z) ** 3
        live = ~done & (cand > 0)
        v = np.where(live, cand, v)
        with np.errstate(invalid="ignore", divide="ignore"):
            lhs = np.log(u24(rng_np(base, k, 2 + 2 * i), 40))
            rhs = 0.5 * z * z + d - d * v + d * np.log(v)
        near |= live & (np.abs(lhs - rhs) < 1e-5)
        done |= live & (lhs < rhs)
    lg = np.log(d * v) + np.log(u24(rng_np(base, k, 0), 40)) / alpha
    return lg, near


def draw(shim, base, n, alpha):
    lg = np.zeros(n, F32)
    eta = np.zeros(n, F32)
    shim.sp_dirichlet(base, n, alpha, lg.ctypes.data, eta.ctypes.data)
    return lg, eta


def test_log_gamma_matches_float64_restatement(shim):
    rng = np.random.default_rng(7)
    near = total = 0
    for alpha in (0.03, 0.3, 1.0, 3.0, 10.0):
        for _ in range(200):
            base = int(rng.integers(0, 1 << 63))
            n = int(rng.integers(1, 129))
            lg, eta = draw(shim, base, n, alpha)
            lg64, nr = log_gamma64(base, n, alpha)
            total += n
            near += int(nr.sum())
            ok = ~nr
            assert np.allclose(lg[ok], lg64[ok], rtol=2e-6, atol=2e-5), alpha
            if not nr.any():
                e64 = np.exp(lg64 - lg64.max())
                assert np.allclose(eta, e64 / e64.sum(), rtol=1e-4, atol=1e-6), alpha
    assert near < total * 0.001, (near, total)


def gamma_sample(shim, alpha, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    while sum(len(x) for x in out) < count:
        out.append(draw(shim, int(rng.integers(0, 1 << 63)), 128, alpha)[0])
    return np.concatenate(out)[:count].astype(np.float64)


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 3.0])
def test_log_gamma_distribution(shim, alpha):
    lg = gamma_sample(shim, alpha, 6000, seed=int(alpha * 1000))
    assert np.isfinite(lg).all()
    # compare log x with the log of scipy's Gamma: the cdf of lg is gamma.cdf(exp(lg)), finite even where exp(lg) underflows
    p = stats.kstest(lg, lambda x: stats.gamma.cdf(np.exp(x), alpha)).pvalue
    assert p > 1e-3, (alpha, p)


@pytest.mark.parametrize("alpha,n", [(0.03, 40), (0.3, 40), (0.3, 8), (1.0, 5), (3.0, 20)])
def test_dirichlet_marginals_are_beta(shim, alpha, n):
    rng = np.random.default_rng(n * 100 + int(alpha * 100))
    first = np.array([draw(shim, int(rng.integers(0, 1 << 63)), n, alpha)[1][0] for _ in range(3000)], np.float64)
    assert beta_ks(first, alpha, n) > 1e-3, (alpha, n)


def beta_ks(eta, alpha, n):
    """KS p-value of eta above 1e-37 against Beta(alpha, (n - 1) alpha) conditioned on the same; the share at or below 1e-37 (where an f32
    eta ends at 0 while Beta with a small alpha still has mass: 7.8 % at alpha 0.03, n 40) must match within 4 standard deviations"""
    tiny = 1e-37
    beta = stats.beta(alpha, (n - 1) * alpha)
    f0 = beta.cdf(tiny)
    low = float(np.mean(eta <= tiny))
    assert abs(low - f0) <= 4 * np.sqrt(f0 * (1 - f0) / len(eta)) + 1e-9, (low, f0)
    return stats.kstest(eta[eta > tiny], lambda x: (beta.cdf(x) - f0) / (1 - f0)).pvalue


def test_single_edge_and_tiny_alpha(shim):
    rng = np.random.default_rng(9)
    for alpha in (1e-6, 0.03, 1.0, 50.0):
        for _ in range(50):
            _, eta = draw(shim, int(rng.integers(0, 1 << 63)), 1, alpha)
            assert eta[0] == F32(1)
    for alpha in (1e-30, 1e-6, 1e-3, 0.01):
        for _ in range(100):
            n = int(rng.integers(2, 129))
            lg, eta = draw(shim, int(rng.integers(0, 1 << 63)), n, alpha)
            assert not np.isnan(eta).any() and (eta >= 0).all()
            assert abs(eta.astype(np.float64).sum() - 1.0) <= 1e-6, alpha
