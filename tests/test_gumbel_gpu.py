"""GPU tests of the Gumbel root search (xq_gumbel_*, TorchGumbel, TorchExamples.record_gumbel): whole searches replayed by the numpy
restatement in gumbel_oracle.py node by node (257 varied roots, L in {1, 4, 8}, max_considered in {1, 2, 16, 128}, n_simulations in
{1, 7, 64}, both views, f32 and bf16 scores), the Sequential Halving counts, begin against select + expand_backup, the schedule after
advance, play against TorchEnv.step, the Gumbel-max property (chi-square), independence of sizes and sharding, call order and argument
errors, the recorded policy targets, and a self-play loop of a small torch network."""
import numpy as np
import pytest
from scipy import stats

import gumbel_oracle as G
import search_oracle as S
from test_search_gpu import _scores, _values
from test_search_leaves_gpu import _net, roots257  # noqa: F401
from test_search_reuse_gpu import assert_tree_equal

pytestmark = pytest.mark.gpu

F32 = np.float32
FIELDS = ("status", "winner", "reward", "depth")
C_PUCT, FPU, VL, T = 1.25, -0.1, 1.0, 0.8


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _vname(view):
    return "side" if view == 1 else "absolute"


def _plan(n_sims, L):
    out, used = [], 0
    while used < n_sims:
        out.append(min(L, n_sims - used))
        used += out[-1]
    return out


def gumbel_search(xq, torch, recs, L, m, n_sims, view, seed, sdt=None, cv=50.0, cs=0.1, max_leaves=8):
    """reset, begin on seeded root scores / values, then the selections of _plan(n_sims, L): (log, root scores, root values, ts, tg)"""
    n = len(recs)
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, n_sims, max_leaves)
    tg = xq.TorchGumbel(ts, m)
    ts.reset()
    sc0, v0 = _scores(seed, 999, n), _values(seed, 999, n)
    x = torch.from_numpy(sc0).cuda()
    tg.begin(x if sdt is None else x.to(sdt), torch.from_numpy(v0).cuda(), n_sims, seed=seed, temperature=T, c_visit=cv, c_scale=cs,
             view=_vname(view))
    log = []
    for s, k in enumerate(_plan(n_sims, L)):
        sel = tg.select(k, C_PUCT, FPU, VL)
        leaves = ts.leaves().clone()
        sc = torch.from_numpy(_scores(seed, s, n * k)).cuda()
        ts.expand_backup(sc if sdt is None else sc.to(sdt), torch.from_numpy(_values(seed, s, n * k)).cuda(), temperature=T, view=_vname(view))
        log.append({f: getattr(sel, f).cpu().numpy() for f in FIELDS} | {"leaves": leaves.cpu().numpy()})
    torch.cuda.synchronize()
    return log, v0, ts, tg


def check_state(recs, tg, dev, i, m, v0, seed):
    """the begin state of tree i against the oracle: the Gumbel words within margins, logf(P) within margins, the considered set exactly
    from the device's g and logit; returns the state"""
    st = tg.gumbel.get(i)
    nodes, edges = dev
    ne = int(nodes[0]["n_edges"]) if nodes[0]["expanded"] else 0
    assert st["m"] == min(m, ne), i
    if ne == 0:
        return st
    base = int(G.rng_np(seed, i, recs[i]["ctr"]))
    want = G.gumbel_draw(base, ne)
    assert (np.abs(st["gumbel"][:ne].astype(np.float64) - want) <= 2.0 ** -21 * np.maximum(1.0, np.abs(want))).all(), i
    P = edges[0]["prior"][:ne]
    with np.errstate(divide="ignore"):
        lp = np.log(P.astype(np.float64))
    fin = np.isfinite(lp)
    assert (np.isneginf(st["logit"][:ne]) == ~fin).all() and np.allclose(st["logit"][:ne][fin], lp[fin], rtol=1e-6, atol=1e-6), i
    key = (st["gumbel"][:ne] + st["logit"][:ne]).astype(F32)
    assert (st["considered"][:ne] == G.considered(key, m)).all() and not st["considered"][ne:].any(), i
    assert (st["n0"][:ne] == 0).all() and np.float32(st["root_value"]).tobytes() == S.clean_value(v0[i]).tobytes(), i
    return st


def replay(L_oracle, recs, log, v0, ts, tg, L, m, n_sims, view, seed, bf16=False, cv=50.0, cs=0.1):
    import torch
    n = len(recs)
    dev = {i: ts.search.get_tree(i) for i in range(n)}
    trees = {}
    for i in range(n):
        Tr = G.GumbelTree(L_oracle, recs[i])
        if Tr.status[0] == 0:          # begin expands and backs up the root
            Tr.expand(0, dev[i][1][0]["prior"])
            Tr.backup(0, v0[i])
        Tr.begin(check_state(recs, tg, dev[i], i, m, v0, seed), n_sims, cv, cs)
        trees[i] = Tr
    for s, k in enumerate(_plan(n_sims, L)):
        vals = _values(seed, s, n * k)
        for i in range(n):
            Tr = trees[i]
            slots = Tr.select_gumbel(k, C_PUCT, FPU, VL)
            for kk, (j, st) in enumerate(slots):
                r = i * k + kk
                assert log[s]["leaves"][r].tobytes() == Tr.rec[j].tobytes(), (s, i, kk, j)
                got = {f: int(log[s][f].reshape(-1)[r]) for f in FIELDS}
                assert got == {"status": st, "winner": Tr.winner[j], "reward": Tr.reward[j], "depth": Tr.depth[j]}, (s, i, kk, j)
            Tr.expand_backup_slots(slots, lambda j: dev[i][1][j]["prior"], vals[i * k:(i + 1) * k])
    for i in range(n):
        assert_tree_equal(dev[i], trees[i], i)
    return trees


CASES = [(1, 16, 64, 1, False), (4, 16, 64, 0, True), (8, 2, 64, 1, True), (8, 128, 64, 0, False), (1, 1, 7, 0, False), (4, 1, 7, 1, True),
         (1, 128, 7, 1, False), (8, 16, 7, 0, False), (1, 2, 1, 1, True), (4, 128, 1, 0, False)]


@pytest.mark.parametrize("L,m,n_sims,view,bf16", CASES)
def test_replay_against_oracle(xq, torch, oracle_lib, roots257, L, m, n_sims, view, bf16):
    seed = 700 + 13 * L + m + n_sims + view
    log, v0, ts, tg = gumbel_search(xq, torch, roots257, L, m, n_sims, view, seed, sdt=torch.bfloat16 if bf16 else None)
    trees = replay(oracle_lib, roots257, log, v0, ts, tg, L, m, n_sims, view, seed, bf16)
    pol, act = (x.cpu().numpy() for x in tg.root(_vname(view)))
    for i, Tr in trees.items():
        wp, wa, _ = Tr.gumbel_root(view)
        assert int(act[i]) == wa, i
        assert np.allclose(pol[i], wp, rtol=4e-6, atol=1e-12), i
        if Tr.gs["m"]:
            assert abs(float(pol[i].astype(np.float64).sum()) - 1.0) < 1e-5
    tg.close()
    ts.close()


@pytest.mark.parametrize("m,n_sims", [(2, 7), (4, 64), (16, 64), (16, 7), (40, 64)])
def test_sequential_halving_counts(xq, torch, roots257, m, n_sims):
    """one leaf per selection: on a fresh root with m <= n_edges the considered edges' visits this move are Sequential Halving's counts;
    no other root edge is visited"""
    log, v0, ts, tg = gumbel_search(xq, torch, roots257, 1, m, n_sims, 1, 31 + m)
    checked = 0
    for i in range(len(roots257)):
        nodes, edges = ts.search.get_tree(i)
        ne = int(nodes[0]["n_edges"]) if nodes[0]["expanded"] else 0
        if ne < m or nodes[0]["status"]:
            continue
        st = tg.gumbel.get(i)
        nv = edges[0]["visits"][:ne]
        cons = st["considered"][:ne]
        want = [0] * m
        for t in G.sequence(m, n_sims):
            want[want.index(t)] += 1
        assert sorted(nv[cons].tolist()) == sorted(want) and (nv[~cons] == 0).all(), i
        checked += 1
    assert checked > 100


def test_begin_is_select_then_expand_backup(xq, torch, roots257):
    n = len(roots257)
    sc, v = torch.from_numpy(_scores(5, 0, n)).cuda(), torch.from_numpy(_values(5, 0, n)).cuda()
    out = []
    for use_begin in (True, False):
        te = xq.TorchEnv(n)
        te.env.set_boards(roots257)
        ts = xq.TorchSearch(te, 8)
        ts.reset()
        if use_begin:
            tg = xq.TorchGumbel(ts, 16)
            tg.begin(sc, v, 8, seed=1, temperature=T)
        else:
            ts.select()
            ts.expand_backup(sc, v, temperature=T)
        out.append([ts.search.get_tree(i) for i in range(n)])
    live = 0
    for (na, ea), (nb, eb) in zip(*out):
        if nb[0]["status"] in (1, 2):           # a terminal root: begin leaves it alone, a select backs its value up
            assert na[0]["visits"] == 0 and nb[0]["visits"] == 1 and len(na) == len(nb) == 1
            continue
        assert na.tobytes() == nb.tobytes() and ea.tobytes() == eb.tobytes()
        live += 1
    assert live > 150


def test_schedule_after_advance(xq, torch):
    """after play + advance the kept root's edges keep their N; N0 records them, and this move's visits follow the schedule again"""
    evaluate = _net(torch)
    n, sims, m = 128, 16, 4
    te = xq.TorchEnv(n, seed=9)
    ts = xq.TorchSearch(te, 2 * sims)
    tg = xq.TorchGumbel(ts, m)
    tg.run(evaluate, sims, seed=3, obs_dtype=torch.float32)
    tg.play(auto_reset=False)
    kept = ts.advance(sims).cpu().numpy()
    assert (kept > 1).sum() > n // 2
    root = tg.run(evaluate, sims, seed=4, obs_dtype=torch.float32, reset=False)
    assert (root.action.cpu().numpy() >= 0).sum() > n // 2
    want = [0] * m
    for t in G.sequence(m, sims):
        want[want.index(t)] += 1
    checked = 0
    for i in range(n):
        nodes, edges = ts.search.get_tree(i)
        st = tg.gumbel.get(i)
        ne = int(nodes[0]["n_edges"]) if nodes[0]["expanded"] else 0
        if ne < m or nodes[0]["status"] or not kept[i]:
            continue
        nv = edges[0]["visits"][:ne] - st["n0"][:ne]
        cons = st["considered"][:ne]
        assert sorted(nv[cons].tolist()) == sorted(want) and (nv[~cons] == 0).all(), i
        checked += (st["n0"][:ne] > 0).any()
    assert checked > 10


@pytest.mark.parametrize("auto_reset", [False, True])
def test_play_is_step_with_root_action(xq, torch, roots257, auto_reset):
    for view in (0, 1):
        log, v0, ts, tg = gumbel_search(xq, torch, roots257, 4, 16, 64, view, 77 + view)
        te2 = xq.TorchEnv(len(roots257))
        te2.env.set_boards(roots257)
        act = tg.root(_vname(view)).action
        want = te2.step(actions=act, pick="given", view=_vname(view), auto_reset=auto_reset)
        got = tg.play(view=_vname(view), auto_reset=auto_reset)
        for f in ("actions", "reward", "done", "winner", "captured", "valid"):
            assert torch.equal(getattr(got, f), getattr(want, f)), f
        assert ts.tenv.env.get_boards().tobytes() == te2.env.get_boards().tobytes()
        again = tg.play(view=_vname(view))             # the roots are stale now: nothing is played
        assert (again.actions.cpu().numpy() == -1).all() and (again.valid.cpu().numpy() == 0).all()


def test_gumbel_max_follows_priors(xq, torch, oracle_lib):
    """m = 1, one simulation: the played action is argmax(g + log P), a sample from the priors (chi-square over 65,536 envs)"""
    n = 65536
    te = xq.TorchEnv(n)
    ts = xq.TorchSearch(te, 1)
    tg = xq.TorchGumbel(ts, 1)
    rng = np.random.default_rng(11)
    row = (rng.standard_normal(8100) * 1.0).astype(F32)
    sc = torch.from_numpy(np.broadcast_to(row, (n, 8100)).copy()).cuda()
    root = tg.run(lambda planes: (sc, torch.zeros(planes.shape[0], device=planes.device)), 1, seed=123, obs_dtype=torch.float32)
    nodes, edges = ts.search.get_tree(0)
    ne = int(nodes[0]["n_edges"])
    acts, P = edges[0]["action"][:ne], edges[0]["prior"][:ne].astype(np.float64)
    got = root.action.cpu().numpy()
    assert (got >= 0).all()
    counts = np.array([(got == a).sum() for a in acts])
    assert counts.sum() == n
    exp = P / P.sum() * n
    big = exp >= 5                          # the edges expected fewer than 5 times pooled into one cell, if there are any
    obs, ex = counts[big], exp[big]
    if (~big).any():
        obs, ex = np.append(obs, counts[~big].sum()), np.append(ex, exp[~big].sum())
    assert stats.chisquare(obs, ex).pvalue > 1e-4
    tg.close()
    ts.close()


def test_draws_do_not_depend_on_size_or_sharding(xq, torch):
    evaluate = _net(torch)
    states = {}
    for n, id0 in ((4097, 0), (33, 0), (1, 0), (2048, 0), (2049, 2048), (1, 4000)):
        te = xq.TorchEnv(n, seed=1, env_id0=id0)
        ts = xq.TorchSearch(te, 4)
        tg = xq.TorchGumbel(ts, 8)
        tg.run(evaluate, 4, seed=21, obs_dtype=torch.float32)
        for i in sorted({0, n - 1, min(n - 1, 32)}):
            states.setdefault(id0 + i, []).append(tg.gumbel.get(i))
        tg.close()
        ts.close()
    for e, lst in states.items():
        for st in lst[1:]:
            assert st["gumbel"].tobytes() == lst[0]["gumbel"].tobytes() and (st["considered"] == lst[0]["considered"]).all(), e


def test_call_order_budget_and_arguments(xq, torch):
    n = 16
    te = xq.TorchEnv(n)
    ts = xq.TorchSearch(te, 8, 4)
    sc, v = torch.zeros((n, 8100), device="cuda"), torch.zeros(n, device="cuda")
    for bad in (0, 129):
        with pytest.raises(xq.XQError):
            xq.TorchGumbel(ts, bad)
    tg = xq.TorchGumbel(ts, 16)
    with pytest.raises(xq.XQError):
        tg.begin(sc, v, 8)                      # never reset
    ts.reset()
    with pytest.raises(xq.XQError):
        tg.select()                             # no begin
    with pytest.raises(xq.XQError):
        tg.root()
    with pytest.raises(xq.XQError):
        tg.play()
    for kw in ({"n_simulations": 0}, {"n_simulations": 9}, {"n_simulations": 8, "c_visit": -1.0}, {"n_simulations": 8, "c_scale": float("nan")},
               {"n_simulations": 8, "c_visit": float("inf")}, {"n_simulations": 8, "temperature": 0.0}):
        with pytest.raises(xq.XQError):
            tg.begin(sc, v, **kw)
    with pytest.raises(ValueError):
        tg.begin(sc, v, 8, view="sideways")
    tg.begin(sc, v, 6)
    with pytest.raises(xq.XQError):
        tg.select(5)                            # leaves past max_leaves
    tg.select(4)
    with pytest.raises(xq.XQError):
        tg.select(1)                            # selection pending
    with pytest.raises(xq.XQError):
        tg.root()
    ts.expand_backup(torch.zeros((4 * n, 8100), device="cuda"), torch.zeros(4 * n, device="cuda"))
    with pytest.raises(xq.XQError):
        tg.select(3)                            # past n_simulations
    tg.select(2)
    ts.expand_backup(torch.zeros((2 * n, 8100), device="cuda"), torch.zeros(2 * n, device="cuda"))
    tg.root()
    ts.reset()
    with pytest.raises(xq.XQError):
        tg.root()                               # the roots changed since begin
    ex = xq.TorchExamples(ts, 64)
    with pytest.raises(xq.XQError):
        ex.record_gumbel(tg)
    te2 = xq.TorchEnv(n)
    ex2 = xq.TorchExamples(te2, 64)
    tg.begin(sc, v, 8)
    with pytest.raises(xq.XQError):
        ex2.record_gumbel(tg)                   # another env
    ex.record_gumbel(tg)
    with pytest.raises(xq.XQError):
        xq.gumbel_bytes(0, 8)
    pad = lambda b: (b + 255) // 256 * 256          # noqa: E731  each of the seven arrays is 256-byte aligned
    for t in (1, 10, 4097):
        assert xq.gumbel_bytes(t, 8) == 4 * pad(512 * t) + pad(16 * t) + 2 * pad(4 * t)
        assert 2072 * t <= xq.gumbel_bytes(t, 8) < 2072 * t + 7 * 256


def test_recorded_targets_are_the_improved_policy(xq, torch):
    evaluate = _net(torch)
    n = 512
    te = xq.TorchEnv(n, seed=5)
    te.env.rollout_random(6)
    ts = xq.TorchSearch(te, 16, 4)
    tg = xq.TorchGumbel(ts, 16)
    ex = xq.TorchExamples(ts, 4 * n)
    root = tg.run(evaluate, 16, seed=8, leaves=4, obs_dtype=torch.float32)
    ex.record_gumbel(tg)
    ex.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.zeros(n, device="cuda"))
    smp = ex.sample(2048, seed=1, counter=0)
    env = ex.get(0, n)["env"]
    idx = smp.index.cpu().numpy()
    raw = ex.get(0, n)
    # q is the example's root q as record() stores it: sum W / sum N, bit for bit TorchSearch.root().q
    q = ts.root().q.cpu().numpy()
    assert raw["q"].view(np.uint32).tolist() == q[raw["env"].astype(np.int64)].view(np.uint32).tolist()
    assert np.isfinite(raw["q"]).all() and np.abs(raw["q"]).max() > 0.01
    tot = raw["visits"].astype(np.int64).sum(1)
    assert (tot == raw["total_visits"]).all() and (np.abs(tot - 2 ** 24) <= raw["n_edges"].astype(np.int64)).all()
    # w_k / sum w: the rounding of each weight (half a unit) and of the division, and the renormalisation by sum w, which is 2^24 within a
    # few units (each pi' carries its own rounding): |w_k / sum w - pi'_k| <= (1.5 + pi'_k |sum w - 2^24|) 2^-24
    pol, want = smp.policy.cpu().numpy().astype(np.float64), root.policy.cpu().numpy()[env[idx].astype(np.int64)].astype(np.float64)
    dev = np.abs(tot[idx] - 2 ** 24)[:, None]
    assert (np.abs(pol - want) <= (1.5 + want * dev) * 2.0 ** -24).all()
    assert np.abs(pol - want).max() <= 2.0 ** -21


def test_self_play_loop(xq, torch):
    """256 envs, advance -> run -> record_gumbel -> play -> finish, committed to the ring"""
    evaluate = _net(torch)
    n, sims, moves = 256, 16, 6
    te = xq.TorchEnv(n, seed=12)
    ts = xq.TorchSearch(te, 3 * sims, 8)
    tg = xq.TorchGumbel(ts, 8)
    ex = xq.TorchExamples(ts, 8 * n)
    ts.reset()
    ended = 0
    for mv in range(moves):
        if mv:
            ts.advance(sims)
        root = tg.run(evaluate, sims, seed=mv, leaves=8, obs_dtype=torch.float32, reset=False)
        assert (root.action.cpu().numpy() >= 0).all()
        ex.record_gumbel(tg)
        step = tg.play()
        assert torch.equal(step.actions, root.action) and (step.valid.cpu().numpy() == 1).all()
        ended += int(ex.finish(step).sum())
    ex.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.zeros(n, device="cuda"))
    info = ex.info()
    assert info["total_committed"] == n * moves and info["stale"] == 0 and info["dropped"] == 0
    smp = ex.sample(512, seed=2, counter=1, want_mask=True)
    s = smp.policy.double().sum(1).cpu().numpy()
    assert (np.abs(s - 1) < 1e-5).all()
