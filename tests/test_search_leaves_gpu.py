"""GPU tests of the multi-leaf selection (xq_search_select_leaves_device, TorchSearch.select_leaves / run(leaves=...)): whole searches of
mixed selection sizes replayed by the numpy restatement in search_leaves_oracle.py slot by slot and node by node, one leaf against the
plain select, duplicates, the budget and argument checks, observe over n * L leaves, root / play / advance / example recording after a
multi-leaf search, sizes, reruns and sharding, and a self-play loop of a small torch network."""
import numpy as np
import pytest

import policy_oracle as P
import search_leaves_oracle as SL
import search_oracle as S
from conftest import harvest_positions, random_boards
from test_search_gpu import _capture_next, _scores, _values
from test_search_reuse_gpu import advance_oracle, assert_tree_equal

pytestmark = pytest.mark.gpu

FIELDS = ("status", "winner", "reward", "depth")


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def roots257(O, oracle_lib):
    """reachable positions, arbitrary boards (the generic kernel), move counts 197..199, boards with a capturable General"""
    reach = harvest_positions(O, 40, 2, 7, seed=241)
    arb = random_boards(O, 60, seed=212)
    late = harvest_positions(O, 60, 1, 13, seed=205)
    late["move_count"] = 197 + np.arange(60) % 3
    cap = _capture_next(O, oracle_lib, 57, seed=277)
    recs = np.concatenate([reach, arb, late, cap])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 7 + 3
    return recs


def _vname(view):
    return "side" if view == 1 else "absolute"


def _plan(max_sims, L):
    """selection sizes of one search: L straight after the reset (duplicates at the root), then single and L-leaf calls to the budget"""
    out, used = [], 0
    while used < max_sims:
        k = min(L if len(out) % 3 != 1 else 1, max_sims - used)
        out.append(k)
        used += k
    return out


def search_leaves(xq, torch, recs, plan, view, seed, vl, c_puct=1.25, fpu=-0.1, t=0.8, sdt=None, max_leaves=32, record=True, ts=None):
    """one search of the selection sizes `plan` on seeded inputs (call s: scores / values of seed (seed, s) over its n * k rows)"""
    n = len(recs)
    if ts is None:
        te = xq.TorchEnv(n)
        te.env.set_boards(recs)
        ts = xq.TorchSearch(te, sum(plan), max_leaves)
    ts.reset()
    log = []
    for s, k in enumerate(plan):
        sel = ts.select_leaves(k, c_puct, fpu, vl)
        leaves = ts.leaves().clone() if record else None
        sc = torch.from_numpy(_scores(seed, s, n * k)).cuda()
        if sdt is not None:
            sc = sc.to(sdt)
        ts.expand_backup(sc, torch.from_numpy(_values(seed, s, n * k)).cuda(), temperature=t, view=_vname(view))
        if record:
            log.append({f: getattr(sel, f).cpu().numpy() for f in FIELDS} | {"leaves": leaves.cpu().numpy()})
    torch.cuda.synchronize()
    return log, ts


def replay_leaves(L, recs, log, ts, plan, view, seed, vl, c_puct=1.25, fpu=-0.1, t=0.8, bf16=False, which=None, check_priors=True):
    """the oracle's search with the device's priors, compared slot by slot after every call, then node by node and edge by edge; priors
    checked against float64 on the score row of the slot that expanded the node"""
    import torch
    n = len(recs)
    which = range(n) if which is None else which
    dev = {i: ts.search.get_tree(i) for i in which}
    trees = {i: SL.LeavesTree(L, recs[i]) for i in which}
    raw_at = {}
    for s, k in enumerate(plan):
        vals = _values(seed, s, n * k)
        sc = _scores(seed, s, n * k)
        if bf16:
            sc = torch.from_numpy(sc).to(torch.bfloat16).float().numpy()
        for i in which:
            T = trees[i]
            slots = T.select_leaves(k, c_puct, fpu, vl)
            for kk, (j, st) in enumerate(slots):
                r = i * k + kk
                assert log[s]["leaves"][r].tobytes() == T.rec[j].tobytes(), (s, i, kk, j)
                got = {f: int(log[s][f].reshape(-1)[r]) for f in FIELDS}
                assert got == {"status": st, "winner": T.winner[j], "reward": T.reward[j], "depth": T.depth[j]}, (s, i, kk, j)
                if st == 0:
                    flip = view == 1 and T.rec[j]["player"] == 1
                    acts = T.lists(j)
                    raw_at[(i, j)] = sc[r, np.where(flip, 8099 - acts, acts)]
            T.expand_backup_slots(slots, lambda j: dev[i][1][j]["prior"], vals[i * k:(i + 1) * k])
    for i in which:
        T, (nodes, edges) = trees[i], dev[i]
        assert_tree_equal((nodes, edges), T, i)
        if not check_priors:
            continue
        for j in range(len(T.rec)):
            c = len(T.act[j]) if T.expanded[j] else 0
            if c == 0:
                continue
            raw = raw_at[(i, j)]
            want = S.priors64(raw, t)
            l = P.clean(raw)
            with np.errstate(invalid="ignore"):
                arg = np.where(np.isfinite(l) & np.isfinite(l.max()), np.abs(l - l.max()) / t, 0.0)
            tol = 1e-6 + 2.0 ** -23 * arg
            got = edges[j]["prior"][:c].astype(np.float64)
            big = want > 1e-30
            assert (np.abs(got - want)[big] <= tol[big] * want[big]).all() and (got[~big] < 1e-30).all(), (i, j)
    return trees


@pytest.mark.parametrize("L,vl,view,bf16,c_puct", [(2, 1.0, 0, False, 1.25), (3, 0.0, 1, True, 1.25), (8, 3.0, 1, False, 0.0),
                                                   (8, 1.0, 0, True, 2.0), (32, 1.0, 1, False, 1.25), (32, 3.0, 0, True, 0.0)])
def test_replay_against_oracle(xq, torch, oracle_lib, roots257, L, vl, view, bf16, c_puct):
    plan = _plan(64, L)
    seed = 400 + L + view
    log, ts = search_leaves(xq, torch, roots257, plan, view, seed, vl, c_puct=c_puct, sdt=torch.bfloat16 if bf16 else None)
    trees = replay_leaves(oracle_lib, roots257, log, ts, plan, view, seed, vl, c_puct=c_puct, bf16=bf16)
    st = np.concatenate([x["status"].reshape(-1) for x in log])
    assert {0, 1, 2, 4}.issubset(set(st.tolist()))
    # root results after the multi-leaf search
    vis, q, best = (x.cpu().numpy() for x in ts.root(_vname(view)))
    for i, T in trees.items():
        wv, wq, wb = T.root(view)
        assert np.array_equal(vis[i], wv) and int(best[i]) == wb, i
        assert (np.isnan(q[i]) and np.isnan(wq)) or q[i].view(np.uint32) == wq.view(np.uint32), i
    ts.close()


def test_one_leaf_is_select(xq, torch, O, oracle_lib, roots257):
    n, sims, seed = len(roots257), 24, 17
    outs = []
    for one in (False, True):
        te = xq.TorchEnv(n)
        te.env.set_boards(roots257)
        ts = xq.TorchSearch(te, sims, 8)
        ts.reset()
        log = []
        for s in range(sims):
            sel = ts.select_leaves(1, 1.25, -0.1, 2.0) if one else ts.select(1.25, -0.1)
            log.append([getattr(sel, f).reshape(-1).cpu().numpy() for f in FIELDS] + [ts.leaves().cpu().numpy()])
            ts.expand_backup(torch.from_numpy(_scores(seed, s, n)).cuda(), torch.from_numpy(_values(seed, s, n)).cuda(), temperature=0.8)
        outs.append((log, [ts.search.get_tree(i) for i in range(n)]))
        ts.close()
    (la, ta), (lb, tb) = outs
    for a, b in zip(la, lb):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    for (na, ea), (nb, eb) in zip(ta, tb):
        assert na.tobytes() == nb.tobytes() and ea.tobytes() == eb.tobytes()


def _net(torch):
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Conv2d(14, 16, 3, padding=1), torch.nn.ReLU(), torch.nn.Flatten(), torch.nn.Linear(16 * 90, 8101)).cuda()

    def evaluate(planes):
        with torch.no_grad():
            out = net(planes.float())
        return out[:, :8100].contiguous(), torch.tanh(out[:, 8100])
    return evaluate


def test_run_with_one_leaf_is_run(xq, torch):
    evaluate = _net(torch)
    trees = []
    for kw in ({}, {"leaves": 1, "virtual_loss": 2.0}):
        te = xq.TorchEnv(64, seed=3)
        te.env.rollout_random(10)
        ts = xq.TorchSearch(te, 20, 4)
        ts.run(evaluate, 20, view="side", obs_dtype=torch.float32, **kw)
        trees.append([ts.search.get_tree(i) for i in range(64)])
        ts.close()
    for (na, ea), (nb, eb) in zip(*trees):
        assert na.tobytes() == nb.tobytes() and ea.tobytes() == eb.tobytes()


def test_duplicates(xq, torch, O, oracle_lib):
    recs = harvest_positions(O, 16, 1, 9, seed=31)
    L = 8
    te = xq.TorchEnv(16)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 40, L)
    ts.reset()
    sel = ts.select_leaves(L, 1.5, 0.0, 1.0)
    st = sel.status.cpu().numpy()
    assert (st[:, 0] == 0).all() and (st[:, 1:] == SL.DUPLICATE).all()
    assert (sel.depth.cpu().numpy() == 0).all()
    assert (ts.leaves().cpu().numpy().reshape(16, L, 64) == recs.view(np.uint8).reshape(16, 1, 64)).all()
    sc = torch.zeros((16 * L, 8100), device="cuda")
    val = torch.full((16 * L,), 0.5, device="cuda")
    ts.expand_backup(sc, val)
    for i in range(16):
        nodes, _ = ts.search.get_tree(i)
        assert len(nodes) == 1 and nodes[0]["visits"] == 1 and nodes[0]["expanded"] == 1

    # NaN scores and values in duplicate slots change nothing
    trees = []
    for poison in (False, True):
        ts.reset()
        dups = 0
        for s in range(4):
            sel = ts.select_leaves(L, 1.5, 0.0, 1.0)
            sc = torch.from_numpy(_scores(9, s, 16 * L)).cuda()
            val = torch.from_numpy(_values(9, s, 16 * L)).cuda()
            dup = sel.status.reshape(-1) == SL.DUPLICATE
            dups += int(dup.sum())
            if poison:
                sc[dup] = float("nan")
                val[dup] = float("nan")
            ts.expand_backup(sc, val)
        assert dups >= 16 * (L - 1)
        trees.append([ts.search.get_tree(i) for i in range(16)])
    for (na, ea), (nb, eb) in zip(*trees):
        assert na.tobytes() == nb.tobytes() and ea.tobytes() == eb.tobytes()
    ts.close()


def test_single_legal_move_root(xq, torch, O, oracle_lib):
    cand = random_boards(O, 3000, seed=5, max_pieces=6)
    counts, _ = P.oracle_lists(oracle_lib, cand)
    ok = [i for i in range(len(cand)) if counts[i] == 1 and not S.generals_missing(cand[i])]
    recs = cand[ok[:8]]
    assert len(recs) == 8
    plan, seed = [1, 4, 4, 4], 12
    log, ts = search_leaves(xq, torch, recs, plan, 1, seed, 1.0, max_leaves=4)
    replay_leaves(oracle_lib, recs, log, ts, plan, 1, seed, 1.0)
    # every descent of the second call takes the only edge; the first makes the child, the rest are its duplicates
    st = log[1]["status"]
    child_open = st[:, 0] == 0
    assert (st[child_open, 1:] == SL.DUPLICATE).all()
    ts.close()


def test_budget_and_errors(xq, torch, O):
    from cn_chess_ai_b200 import XQError, search_bytes_per_tree

    def refused(f, *a, **k):
        with pytest.raises(XQError):
            f(*a, **k)

    for m in (1, 7, 64, 200):
        assert search_bytes_per_tree(m, 1) == search_bytes_per_tree(m) == (m + 1) * 2389 + 73
        for L in (2, 8, 32):
            assert search_bytes_per_tree(m, L) == (m + 1) * 2389 + 4 + 69 * L
    for m, L in ((0, 1), (4, 0), (4, 33), (4, -1)):
        refused(search_bytes_per_tree, m, L)
    te = xq.TorchEnv(40)
    for L in (0, 33, -2):
        refused(xq.BatchedSearch, te.env, 8, L)
    ts = xq.TorchSearch(te, 10, 4)
    refused(ts.select_leaves, 2)                                           # never reset
    ts.reset()
    for L in (0, 5, 33):
        refused(ts.select_leaves, L)
    for vl in (-1.0, float("nan"), float("inf")):
        refused(ts.select_leaves, 2, virtual_loss=vl)
    refused(ts.select_leaves, 2, c_puct=-1.0)
    refused(ts.select_leaves, 2, fpu=float("nan"))

    def sim(L):
        ts.select_leaves(L)
        ts.expand_backup(torch.zeros((40 * L, 8100), device="cuda"), torch.zeros(40 * L, device="cuda"))

    ts.select_leaves(4)
    refused(ts.select_leaves, 1)                                           # a selection pending
    with pytest.raises(ValueError):                                        # the rows of the last selection are 40 * 4
        ts.expand_backup(torch.zeros((40, 8100), device="cuda"), torch.zeros(40, device="cuda"))
    ts.expand_backup(torch.zeros((160, 8100), device="cuda"), torch.zeros(160, device="cuda"))
    sim(4)
    refused(ts.select_leaves, 3)                                           # 8 + 3 > 10
    sim(2)
    refused(ts.select)
    assert ts.search.get_tree(0)[0][0]["visits"] == 10 - 3                 # the three duplicates of the first call are not backed up
    # after advance(min_free) the budget is min_free slots
    ts.advance(5)
    sim(4)
    refused(ts.select_leaves, 2)
    sim(1)
    refused(ts.select_leaves, 1)
    ts.close()


@pytest.mark.parametrize("view", [0, 1])
def test_observe_leaves(xq, torch, O, view):
    recs = np.concatenate([harvest_positions(O, 50, 1, 11, seed=44), random_boards(O, 14, seed=45)])
    n, L = len(recs), 6
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 19, L)
    search_leaves(xq, torch, recs, [1, 6, 6], view, 3, 1.0, ts=ts, record=False)
    ts.select_leaves(L)
    leaves = ts.leaves().clone().cpu().numpy()
    ref = xq.TorchEnv(n * L)
    ref.env.set_boards(leaves.view(recs.dtype).reshape(-1))
    for dt in (torch.float32, torch.bfloat16, torch.uint8):
        planes, aux = ts.observe(dt, _vname(view))
        assert planes.shape[0] == n * L
        wp, wa = ref.observe(dt, _vname(view))
        assert torch.equal(planes, wp) and torch.equal(aux, wa), dt
    ts.close()


def test_play_advance_and_record_after_a_multi_leaf_search(xq, torch, O, oracle_lib):
    recs = harvest_positions(O, 96, 1, 9, seed=61)
    n, L, seed, view = len(recs), 8, 21, 1
    plan = _plan(40, L)
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 40, L)
    log, _ = search_leaves(xq, torch, recs, plan, view, seed, 1.0, ts=ts)
    trees = replay_leaves(oracle_lib, recs, log, ts, plan, view, seed, 1.0, check_priors=False)
    ex = xq.TorchExamples(ts, 4 * n)
    ex.record(ts)
    root = ts.root("side")
    step = ts.play(temperature=0.0, view="side", auto_reset=False)
    assert torch.equal(step.actions, root.best) and (step.valid.cpu().numpy() == 1).all()
    ex.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.zeros(n, device="cuda"))
    got = ex.get(0, n)
    for i, T in trees.items():
        c = len(T.act[0])
        assert got[i]["rec"].tobytes() == recs[i].tobytes() and int(got[i]["n_edges"]) == c
        assert (got[i]["action"][:c] == T.act[0]).all() and (got[i]["visits"][:c] == T.N[0]).all(), i
    # advance: the played child's subtree, as the oracle re-roots it
    boards = te.env.get_boards()
    min_free = 16
    ts.advance(min_free)
    torch.cuda.synchronize()
    for i, T in trees.items():
        U, _ = advance_oracle(oracle_lib, T, boards[i], min_free, 41)
        assert_tree_equal(ts.search.get_tree(i), U, i)
    ex.close()
    ts.close()


@pytest.mark.parametrize("n", [1, 33, 4097])
def test_sizes(xq, torch, O, oracle_lib, n):
    recs = harvest_positions(O, n, 1, 9 + n % 2, seed=n + 7)
    plan, seed = [8, 1, 8, 8], 500 + n
    log, ts = search_leaves(xq, torch, recs, plan, 1, seed, 1.0, max_leaves=8)
    which = sorted(set(range(0, n, max(1, n // 40))) | {n - 1})
    replay_leaves(oracle_lib, recs, log, ts, plan, 1, seed, 1.0, which=which)
    ts.close()


def test_rerun_and_sharding(xq, torch, O):
    recs = np.concatenate([harvest_positions(O, 150, 2, 5, seed=19), random_boards(O, 40, seed=13)])
    n, plan, seed = len(recs), [1, 8, 8, 8, 5], 77
    roots = []
    for _ in range(2):
        _, ts = search_leaves(xq, torch, recs, plan, 1, seed, 1.0, max_leaves=8, record=False)
        roots.append(ts.root("side"))
        ts.close()
    assert torch.equal(roots[0].visits, roots[1].visits) and torch.equal(roots[0].q.view(torch.int32), roots[1].q.view(torch.int32))
    h = 101
    parts = []
    for part in (slice(0, h), slice(h, n)):
        m = len(recs[part])
        te = xq.TorchEnv(m)
        te.env.set_boards(recs[part])
        ts = xq.TorchSearch(te, sum(plan), 8)
        ts.reset()
        for s, k in enumerate(plan):
            ts.select_leaves(k, 1.25, -0.1, 1.0)
            rows = np.arange(n * k).reshape(n, k)[part].reshape(-1)
            ts.expand_backup(torch.from_numpy(_scores(seed, s, n * k)[rows]).cuda(), torch.from_numpy(_values(seed, s, n * k)[rows]).cuda(),
                             temperature=0.8)
        parts.append(ts.root("side"))
        ts.close()
    assert torch.equal(torch.cat([p.visits for p in parts]), roots[0].visits)
    assert torch.equal(torch.cat([p.q for p in parts]).view(torch.int32), roots[0].q.view(torch.int32))


def test_self_play_with_eight_leaves(xq, torch, O, oracle_lib):
    """256 envs, run(leaves=8) per move with a small torch network; every call's network output is captured and the oracle replays
    the search on it; the greedy move is then played on the env and on the oracle's boards"""
    evaluate = _net(torch)
    n, sims, L, moves, cap_value = 256, 33, 8, 3, 0.0
    te = xq.TorchEnv(n, seed=4)
    ts = xq.TorchSearch(te, sims, L)
    ref = O.new_envs(n)
    for mv in range(moves):
        calls = []

        def capture(planes):
            sc, v = evaluate(planes)
            calls.append((sc.float().cpu().numpy(), v.float().cpu().numpy()))
            return sc, v

        root = ts.run(capture, sims, c_puct=1.5, view="side", obs_dtype=torch.float32, leaves=L, virtual_loss=1.0, cap_value=cap_value)
        assert [len(c[1]) for c in calls] == [n] + [n * L] * 4
        which = range(0, n, 5)
        dev = {i: ts.search.get_tree(i) for i in which}
        for i in which:
            T = SL.LeavesTree(oracle_lib, ref[i].copy())
            for sc, v in calls:
                k = len(v) // n
                slots = T.select_leaves(k, 1.5, 0.0, 1.0)
                vals = []
                for kk, (j, st) in enumerate(slots):
                    x = v[i * k + kk]
                    if st in (1, 2, 3):
                        x = {1: 1.0 if T.winner[j] == T.rec[j]["player"] else -1.0, 2: cap_value, 3: -1.0}[st]
                    vals.append(np.float32(x))
                T.expand_backup_slots(slots, lambda j: dev[i][1][j]["prior"], vals)
            assert_tree_equal(dev[i], T, (mv, i))
            wv, _, wb = T.root(1)
            assert int(root.best[i]) == wb and np.array_equal(root.visits[i].cpu().numpy(), wv), (mv, i)
        best = root.best.cpu().numpy()
        r = te.step(actions=root.best, pick="given", view="side")
        assert (r.valid.cpu().numpy() == 1).all(), mv
        a = np.where(ref["player"] == 1, 8099 - best, best)
        act = ((a // 90) << 7 | (a % 90)).astype(np.uint16)
        rew = np.zeros(n, np.int32)
        done, win, cap, valid = (np.zeros(n, np.uint8) for _ in range(4))
        oracle_lib.xqo_batch_step(ref.ctypes.data, n, act, rew, done, win, cap, valid)
        for i in np.nonzero(done)[0]:
            c = ref[i]["ctr"]
            oracle_lib.xqo_reset(ref[i:i + 1].ctypes.data)
            ref[i]["ctr"] = c
        assert te.env.get_boards().tobytes() == ref.tobytes(), mv
    ts.close()
