"""GPU tests of playing self-play moves from the search and of the library's root noise (xq_search_play_device,
xq_search_root_noise_device, TorchSearch.play / root_noise / run(dirichlet_alpha=...)): greedy play against root.best through
TorchEnv.step(pick="given") on a second handle, bit for bit; sampled play against a numpy restatement from get_tree visits and xq_rng; the
temperature schedule and a chi-square test of the sampled frequencies; stale and unvisited roots, errors and call order; sharding; the noise
mix bit for bit, the dense root_noise path fed with the drawn noise, the noise against the host helper and Beta(alpha, (n - 1) alpha); and an
end-to-end self-play loop of a small torch network against the oracle, committed to the example ring."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import test_search_play_cpu as H
from conftest import ROOT, harvest_positions
from test_search_gpu import _capture_next, _scores, _values

pytestmark = pytest.mark.gpu

F32 = np.float32
C_PUCT, FPU, TEMP = 1.25, -0.1, 0.8
ENV_SEED = 31


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("search_play_shim_gpu") / "libxq_search_play_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "search_play_shim.cpp")], check=True)
    L = C.CDLL(so)
    L.sp_dirichlet.argtypes = [C.c_uint64, C.c_int, C.c_float, C.c_void_p, C.c_void_p]
    return L


@pytest.fixture(scope="module")
def boards257(O, oracle_lib):
    """mid-game positions, positions one ply before the move cap, boards where a General can be captured"""
    mid = harvest_positions(O, 80, 2, 12, seed=301)
    late = harvest_positions(O, 60, 1, 15, seed=302)
    late["move_count"] = 199
    cap = _capture_next(O, oracle_lib, 37, seed=303)
    recs = np.concatenate([mid, late, cap])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 3 + 1
    return recs


def _vname(view):
    return "side" if view == 1 else "absolute"


def searched(xq, torch, recs, sims, view, seed=5, env_id0=0, inputs=None, env_seed=ENV_SEED):
    """a TorchEnv holding recs and a TorchSearch after `sims` seeded simulations; inputs: per simulation (scores, values) of the
    global rows env_id0 .. env_id0 + n (sharding), seeded per tree count otherwise"""
    n = len(recs)
    te = xq.TorchEnv(n, seed=env_seed, env_id0=env_id0)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    ts.reset()
    for s in range(sims):
        sc, va = inputs[s] if inputs else (_scores(seed, s, n), _values(seed, s, n))
        ts.select(C_PUCT, FPU)
        ts.expand_backup(torch.from_numpy(sc[env_id0:env_id0 + n] if inputs else sc).cuda(),
                         torch.from_numpy(va[env_id0:env_id0 + n] if inputs else va).cuda(), temperature=TEMP, view=_vname(view))
    torch.cuda.synchronize()
    return te, ts


def step_tuple(st):
    return tuple(None if x is None else x.cpu().numpy() for x in st)


def root_visits(ts, t):
    nodes, edges = ts.search.get_tree(t)
    ne = int(nodes[0]["n_edges"]) if nodes[0]["expanded"] else 0
    return edges[0]["visits"][:ne].astype(np.int32), edges[0]["action"][:ne].astype(np.int64), nodes[0]["rec"]


def policy_of(action, rec, view):
    return 8099 - action if view == 1 and rec["player"] == 1 else action


@pytest.mark.parametrize("view", [0, 1])
@pytest.mark.parametrize("auto_reset", [False, True])
def test_greedy_play_equals_root_best_through_given_step(xq, torch, boards257, view, auto_reset):
    for how in ("tau0", "plies0"):
        te, ts = searched(xq, torch, boards257, 24, view)
        twin = xq.TorchEnv(len(boards257), seed=ENV_SEED)
        twin.env.set_boards(boards257)
        best = ts.root(_vname(view)).best
        want = twin.step(actions=best, pick="given", view=_vname(view), auto_reset=auto_reset)
        got = ts.play(temperature=0.0 if how == "tau0" else 1.0, sample_plies=30 if how == "tau0" else 0, view=_vname(view),
                      auto_reset=auto_reset)
        torch.cuda.synchronize()
        g, w = step_tuple(got), step_tuple(want)
        assert g[1] is None
        assert (g[0] == w[0]).all() and (g[0] == best.cpu().numpy()).all(), how
        for i in range(2, 7):
            assert (g[i] == w[i]).all(), (how, i)
        assert te.env.get_boards().tobytes() == twin.env.get_boards().tobytes(), how
        assert w[3].any(), "no game-ending move was covered"
        ts.close(); te.close(); twin.close()


@pytest.mark.parametrize("tau", [1.0, 0.5, 2.0])
def test_sampled_play_against_numpy(xq, torch, boards257, tau):
    view = 1
    te, ts = searched(xq, torch, boards257, 32, view)
    recs = te.env.get_boards()
    got = step_tuple(ts.play(temperature=tau, sample_plies=1000, view="side", auto_reset=False))
    L = xq.lib()
    close = 0
    for t in range(len(recs)):
        visits, acts, rec = root_visits(ts, t)
        if visits.sum() == 0:
            assert got[0][t] == -1 and got[6][t] == 0
            continue
        u = F32(L.xq_rng(ENV_SEED, t, int(recs[t]["ctr"])) >> 40) * F32(2.0 ** -24)
        k, _, run, thr = H.sample_numpy(visits, tau, u)
        if tau != 1.0 and np.any(np.abs(run - thr) <= 1e-5 * float(run[-1])):
            close += 1
            assert got[0][t] in {policy_of(a, rec, view) for a in acts}
            continue
        assert got[0][t] == policy_of(acts[k], rec, view), t
        assert got[6][t] == 1
    assert close <= 3
    ts.close(); te.close()


def test_sample_plies_schedule_and_zero_temperature_play_best(xq, torch, boards257):
    recs = boards257.copy()
    recs["move_count"][::2] = 40             # at or past sample_plies = 40: greedy
    recs["move_count"][1::2] = 39            # below: sampled
    te, ts = searched(xq, torch, recs, 32, 1)
    best = ts.root("side").best.cpu().numpy()
    got = ts.play(temperature=1.0, sample_plies=40).actions.cpu().numpy()
    assert (got[::2] == best[::2]).all()
    assert (got[1::2] != best[1::2]).any()   # sampling does reach other edges
    ts.close(); te.close()


@pytest.mark.parametrize("tau", [1.0, 0.5])
def test_sampled_frequencies_chi_square(xq, torch, O, tau):
    n = 4096
    recs = O.new_envs(n)
    te = xq.TorchEnv(n, seed=77)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 64)
    ts.reset()
    row = torch.from_numpy(_scores(9, 0, 1)[0]).cuda().clamp(-3, 3)
    for s in range(64):
        ts.select(C_PUCT, FPU)
        ts.expand_backup(row.expand(n, -1).contiguous(), torch.zeros(n, device="cuda"), temperature=TEMP)
    visits, acts, rec = root_visits(ts, 0)
    for t in (1, n - 1):
        assert (root_visits(ts, t)[0] == visits).all()
    got = ts.play(temperature=tau, sample_plies=1000, auto_reset=False).actions.cpu().numpy()
    live = visits > 0
    p = visits[live].astype(np.float64) ** (1.0 / tau)
    p /= p.sum()
    idx = {int(a): i for i, a in enumerate(acts[live])}
    counts = np.bincount([idx[int(a)] for a in got], minlength=len(p))
    assert counts.sum() == n
    small = p * n < 5                                              # edges expected fewer than 5 times share one bin
    obs = np.append(counts[~small], counts[small].sum())
    exp = np.append(p[~small] * n, p[small].sum() * n)
    keep = exp > 0
    assert stats.chisquare(obs[keep], exp[keep]).pvalue > 1e-3
    ts.close(); te.close()


def test_stale_and_unvisited_roots_play_nothing(xq, torch, boards257):
    te, ts = searched(xq, torch, boards257, 8, 1)
    before = te.env.get_boards()
    te.step(actions=ts.root().best, pick="given")                 # every env moves: every root is stale now
    moved = te.env.get_boards()
    st = step_tuple(ts.play(temperature=1.0, auto_reset=False))
    assert (st[0] == -1).all() and (st[6] == 0).all()
    assert te.env.get_boards().tobytes() == moved.tobytes()
    assert moved.tobytes() != before.tobytes()
    ts.reset()                                                     # roots never expanded: no visited edge
    st = step_tuple(ts.play(temperature=0.0, auto_reset=False))
    assert (st[0] == -1).all() and (st[6] == 0).all()
    assert te.env.get_boards().tobytes() == moved.tobytes()
    ts.close(); te.close()


def test_errors_and_call_order(xq, torch, boards257):
    te = xq.TorchEnv(len(boards257))
    te.env.set_boards(boards257)
    ts = xq.TorchSearch(te, 4)
    with pytest.raises(xq.XQError, match="never reset"):
        ts.play()
    with pytest.raises(xq.XQError, match="never reset"):
        ts.root_noise(0.3)
    ts.reset()
    ts.select()
    with pytest.raises(xq.XQError, match="not expanded"):
        ts.play()
    with pytest.raises(xq.XQError, match="not expanded"):
        ts.root_noise(0.3)
    n = len(boards257)
    ts.expand_backup(torch.zeros((n, 8100), device="cuda"), torch.zeros(n, device="cuda"))
    for tau in (-1.0, float("nan"), float("inf")):
        with pytest.raises(xq.XQError, match="temperature"):
            ts.play(temperature=tau)
    with pytest.raises(xq.XQError, match="sample_plies"):
        ts.play(sample_plies=-1)
    with pytest.raises(xq.XQError, match="view"):
        ts.search.play_device(1.0, 0, 7, True)
    for alpha in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(xq.XQError, match="alpha"):
            ts.root_noise(alpha)
    for eps in (-0.1, 1.5, float("nan")):
        with pytest.raises(xq.XQError, match="eps"):
            ts.root_noise(0.3, eps=eps)
    ts.play()                                                      # still usable
    ts.root_noise(0.3)
    torch.cuda.synchronize()
    ts.close(); te.close()


def test_sharding(xq, torch, O):
    N = 4097
    recs = np.concatenate([harvest_positions(O, 1024, 4, 5, seed=404), harvest_positions(O, 1, 1, 9, seed=405)])
    recs["ctr"] = np.arange(N, dtype=np.uint32) % 11

    inputs = [(_scores(12, s, N), _values(12, s, N)) for s in range(12)]

    def run(lo, hi):
        te, ts = searched(xq, torch, recs[lo:hi], 12, 1, env_id0=lo, inputs=inputs)
        eta = ts.root_noise(0.3, seed=3, want_noise=True).cpu().numpy()
        st = ts.play(temperature=1.0, sample_plies=1000, auto_reset=True)
        out = (st.actions.cpu().numpy(), eta, te.env.get_boards())
        ts.close(); te.close()
        return out

    whole = run(0, N)
    parts = [run(0, 2000), run(2000, N)]
    for i in range(3):
        assert np.concatenate([p[i] for p in parts]).tobytes() == whole[i].tobytes()
    for hi in (1, 33):
        part = run(0, hi)
        for i in range(3):
            assert part[i].tobytes() == whole[i][:hi].tobytes()


def _priors(ts, n):
    out = np.zeros((n, 128), F32)
    ne = np.zeros(n, np.int64)
    for t in range(n):
        nodes, edges = ts.search.get_tree(t)
        ne[t] = nodes[0]["n_edges"] if nodes[0]["expanded"] else -1
        out[t] = edges[0]["prior"]
    return out, ne


def test_noise_mix_is_bit_exact_and_leaves_other_trees_alone(xq, torch, boards257):
    n = len(boards257)
    te, ts = searched(xq, torch, boards257, 3, 1)
    mask = torch.from_numpy((np.arange(n) % 3 != 0).astype(np.uint8)).cuda()
    before, ne = _priors(ts, n)
    eps = 0.3
    eta = ts.root_noise(0.3, eps=eps, seed=11, mask=mask, want_noise=True).cpu().numpy()
    after, _ = _priors(ts, n)
    for t in range(n):
        k = max(int(ne[t]), 0)
        if t % 3 == 0 or k == 0:
            assert after[t].tobytes() == before[t].tobytes()
            assert (eta[t] == 0).all()
            continue
        want = (F32(1) + F32(-eps)) * before[t, :k] + F32(eps) * eta[t, :k]
        assert after[t, :k].tobytes() == want.astype(F32).tobytes(), t
        assert (eta[t, k:] == 0).all() and abs(float(eta[t, :k].astype(np.float64).sum()) - 1) < 1e-5
    ts.close(); te.close()
    te2 = xq.TorchEnv(n)
    te2.env.set_boards(boards257)
    ts2 = xq.TorchSearch(te2, 2)
    ts2.reset()                                                    # unexpanded roots: nothing changes, zero rows
    eta = ts2.root_noise(0.3, want_noise=True).cpu().numpy()
    assert (eta == 0).all()
    assert (_priors(ts2, 4)[0] == 0).all()
    ts2.close(); te2.close()


@pytest.mark.parametrize("view", [0, 1])
def test_noise_equals_the_dense_path(xq, torch, boards257, view):
    n, sims, eps = len(boards257), 10, 0.25
    vn = _vname(view)
    te = xq.TorchEnv(n)
    te.env.set_boards(boards257)
    ts = xq.TorchSearch(te, sims)
    te2 = xq.TorchEnv(n)
    te2.env.set_boards(boards257)
    ts2 = xq.TorchSearch(te2, sims)
    ts.reset(); ts2.reset()
    for s in range(sims):
        sc, va = torch.from_numpy(_scores(8, s, n)).cuda(), torch.from_numpy(_values(8, s, n)).cuda()
        ts.select(C_PUCT, FPU)
        ts.expand_backup(sc, va, temperature=TEMP, view=vn)
        if s == 0:
            eta = ts.root_noise(0.3, eps=eps, seed=21, want_noise=True).cpu().numpy()
            dense = np.zeros((n, 8100), F32)
            for t in range(n):
                visits, acts, rec = root_visits(ts, t)
                dense[t, [policy_of(int(a), rec, view) for a in acts]] = eta[t, :len(acts)]
            dense_t = torch.from_numpy(dense).cuda()
        ts2.select(C_PUCT, FPU)
        ts2.expand_backup(sc, va, temperature=TEMP, view=vn, root_noise=dense_t, noise_eps=eps)
    for t in range(n):
        a, b = ts.search.get_tree(t), ts2.search.get_tree(t)
        assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes(), t
    ts.close(); te.close(); ts2.close(); te2.close()


def test_noise_distribution_on_device(xq, torch, O, shim):
    n, alpha = 65536, 0.3
    te = xq.TorchEnv(n, env_id0=1000)
    recs = O.new_envs(n)
    recs["ctr"] = np.arange(n, dtype=np.uint32) % 7
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 1)
    ts.reset()
    ts.select()
    ts.expand_backup(torch.zeros((n, 8100), device="cuda"), torch.zeros(n, device="cuda"))
    eta = ts.root_noise(alpha, eps=0.0, seed=123, want_noise=True).cpu().numpy()
    ne = int(ts.search.get_tree(0)[0][0]["n_edges"])
    assert ne > 30 and (eta[:, ne:] == 0).all()
    L = xq.lib()
    off = 0
    for t in range(0, n, 37):
        base = L.xq_rng(123, 1000 + t, int(recs[t]["ctr"]))
        lg, want = np.zeros(ne, F32), np.zeros(ne, F32)
        shim.sp_dirichlet(base, ne, alpha, lg.ctypes.data, want.ctypes.data)
        off += not np.allclose(eta[t, :ne], want, rtol=1e-4, atol=1e-6)
    assert off <= 3, off                                          # an acceptance test within rounding of its threshold
    assert H.beta_ks(eta[:, 0].astype(np.float64), alpha, ne) > 1e-3
    assert H.beta_ks(eta[:, 17].astype(np.float64), alpha, ne) > 1e-3
    assert abs(eta.astype(np.float64).sum(1) - 1).max() < 1e-5
    # the same seed gives the same bits (the priors were not changed at eps 0), another seed other noise
    assert ts.root_noise(alpha, eps=0.0, seed=123, want_noise=True).cpu().numpy().tobytes() == eta.tobytes()
    other = ts.root_noise(alpha, eps=0.0, seed=124, want_noise=True).cpu().numpy()
    assert (other[:, :ne] != eta[:, :ne]).mean() > 0.99
    ts.close(); te.close()


def test_self_play_loop_end_to_end(xq, torch, O, oracle_lib):
    n, sims, moves = 256, 16, 12
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(1260, 64), torch.nn.Tanh(), torch.nn.Linear(64, 8101)).cuda()

    @torch.no_grad()
    def evaluate(planes):
        out = net(planes.float())
        return out[:, :8100].contiguous(), torch.tanh(out[:, 8100])

    def play(noise, tau):
        recs = O.new_envs(n)
        recs["move_count"][n // 2:] = 190                          # the second half reaches the move cap after 10 moves
        te = xq.TorchEnv(n, seed=4)
        te.env.set_boards(recs)
        ts = xq.TorchSearch(te, 2 * sims)
        ex = xq.TorchExamples(ts, 4096, 32)
        distinct = []
        last_end = np.full(n, -1)
        for mv in range(moves):
            if mv:
                ts.advance(sims)
            ts.run(evaluate, sims, obs_dtype=torch.float32, reset=mv == 0, dirichlet_alpha=0.3 if noise else None)
            ex.record(ts)
            pre = te.env.get_boards()
            st = ts.play(temperature=tau, sample_plies=8)
            ex.finish(st)
            post = te.env.get_boards()
            a = st.actions.cpu().numpy()
            assert (st.valid.cpu().numpy() == 1).all()
            absa = np.where(pre["player"] == 1, 8099 - a, a)
            ref = pre.copy()
            rew = np.zeros(n, np.int32)
            done, win, cap, valid = (np.zeros(n, np.uint8) for _ in range(4))
            oracle_lib.xqo_batch_step(ref.ctypes.data, n, ((absa // 90) << 7 | absa % 90).astype(np.uint16), rew, done, win, cap, valid)
            assert (valid == 1).all() and (rew == st.reward.cpu().numpy()).all() and (done == st.done.cpu().numpy()).all()
            assert (cap == st.captured.cpu().numpy()).all() and (win == st.winner.cpu().numpy()).all()
            live = done == 0
            assert post[live].tobytes() == ref[live].tobytes()
            assert (post["move_count"][~live] == 0).all()
            last_end[done == 1] = mv
            distinct.append(len({r.tobytes() for r in post[: n // 2][["sq", "move_count", "player", "red_score", "black_score"]]}))
        info = ex.info()
        # every example of a game that ended was committed, every later one is staged
        assert info["size"] == (last_end + 1).sum() and info["pending"] == n * moves - info["size"] and info["stale"] == 0
        assert (last_end[n // 2:] >= 0).all()                     # at the move cap if no General fell before
        ts.close(); te.close()
        return distinct

    assert max(play(noise=False, tau=0.0)) == 1                   # one network, no noise, greedy: the games from the opening are one
    assert play(noise=True, tau=1.0)[7] > n // 8                   # sampled moves and root noise: they spread out
