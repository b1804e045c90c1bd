"""GPU tests of subtree reuse between moves (xq_search_advance, TorchSearch.advance / run(reset=False)): after a move, every tree's
get_tree must equal a numpy compaction of its pre-advance tree (search_oracle.Tree, re-rooted by `advance_oracle` below) field by field
and bit for bit; rebuilt trees must equal a fresh reset; the simulations that follow are replayed leaf by leaf and node by node against
the oracle continuing from its compacted tree; root noise on kept and rebuilt roots, the call-order and argument checks, the budget,
sizes, sharding, and an end-to-end game of a small torch network."""
import numpy as np
import pytest

import policy_oracle as P
import search_oracle as S
from conftest import harvest_positions, random_boards
from test_search_gpu import _capture_next, _scores, _values

pytestmark = pytest.mark.gpu

F32 = np.float32
C_PUCT, FPU, TEMP = 1.25, -0.1, 0.8


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
    """reachable positions, arbitrary boards (the generic path), move counts 197..199, boards with a capturable General"""
    reach = harvest_positions(O, 40, 2, 7, seed=141)
    arb = random_boards(O, 60, seed=112)
    late = harvest_positions(O, 60, 1, 13, seed=105)
    late["move_count"] = 197 + np.arange(60) % 3
    cap = _capture_next(O, oracle_lib, 57, seed=177)
    recs = np.concatenate([reach, arb, late, cap])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 5 + 2
    return recs


def _vname(view):
    return "side" if view == 1 else "absolute"


def simulate(torch, ts, sims, seed, view, noise=None, eps=0.25, record=True):
    """sims seeded simulations on the current trees; the per-simulation log of leaves and select outputs"""
    n = ts.n
    nz = None if noise is None else torch.from_numpy(noise).cuda()
    log = []
    for s in range(sims):
        sel = ts.select(C_PUCT, FPU)
        leaves = ts.leaves().clone() if record else None
        ts.expand_backup(torch.from_numpy(_scores(seed, s, n)).cuda(), torch.from_numpy(_values(seed, s, n)).cuda(), temperature=TEMP,
                         root_noise=nz, noise_eps=eps, view=_vname(view))
        if record:
            log.append({k: getattr(sel, k).cpu().numpy() for k in ("status", "winner", "reward", "depth")} | {"leaves": leaves.cpu().numpy()})
    torch.cuda.synchronize()
    return log


def tree_from_device(L, nodes, edges):
    """a search_oracle.Tree holding a device tree as read back by get_tree"""
    T = S.Tree(L, nodes[0]["rec"])
    T.rec = [nd["rec"].copy() for nd in nodes]
    for f, k in (("parent", "parent"), ("pedge", "parent_edge"), ("visits", "visits"), ("reward", "reward"), ("depth", "depth"),
                 ("winner", "winner"), ("status", "status")):
        setattr(T, f, [int(nd[k]) for nd in nodes])
    T.expanded = [bool(nd["expanded"]) for nd in nodes]
    T.act, T.P, T.N, T.W, T.child = [], [], [], [], []
    for nd, e in zip(nodes, edges):
        if not nd["expanded"]:
            for a in (T.act, T.P, T.N, T.W, T.child):
                a.append(None)
            continue
        c = int(nd["n_edges"])
        T.act.append(e["action"][:c].astype(np.int64)); T.P.append(e["prior"][:c].copy()); T.N.append(e["visits"][:c].astype(np.int64))
        T.W.append(e["value_sum"][:c].copy()); T.child.append(e["child"][:c].astype(np.int64))
    return T


def advance_oracle(L, T, env_rec, min_free, cap, noise=None, eps=0.25, view=1):
    """xq_search_advance on one oracle tree: (new tree, kept)"""
    key = env_rec.tobytes()
    m = None
    if T.rec[0].tobytes() == key:
        m = 0
    elif T.expanded[0]:
        hits = [int(c) for c in T.child[0] if c >= 0 and T.rec[int(c)].tobytes() == key]
        assert len(hits) <= 1
        m = hits[0] if hits else None
    if m is not None:
        keep = np.zeros(len(T.rec), bool)
        keep[m] = True
        for j in range(m + 1, len(T.rec)):
            keep[j] = keep[T.parent[j]]
        old = np.nonzero(keep)[0]
    if m is None or len(old) > cap - min_free:
        return S.Tree(L, env_rec.copy()), 0
    new = np.full(len(T.rec), -1, np.int64)
    new[old] = np.arange(len(old))
    U = S.Tree(L, T.rec[m].copy())
    dm = T.depth[m]
    U.rec = [T.rec[j].copy() for j in old]
    U.parent = [-1 if j == m else int(new[T.parent[j]]) for j in old]
    U.pedge = [0 if j == m else T.pedge[j] for j in old]
    U.visits = [T.visits[j] for j in old]
    U.reward = [0 if j == m else T.reward[j] for j in old]
    U.depth = [T.depth[j] - dm for j in old]
    U.winner = [T.winner[j] for j in old]
    U.status = [T.status[j] for j in old]
    U.expanded = [T.expanded[j] for j in old]
    U.act = [None if T.act[j] is None else T.act[j].copy() for j in old]
    U.N = [None if T.N[j] is None else T.N[j].copy() for j in old]
    U.W = [None if T.W[j] is None else T.W[j].copy() for j in old]
    U.child = [None if T.child[j] is None else np.where(T.child[j] >= 0, new[np.maximum(T.child[j], 0)], -1) for j in old]
    U.P = [None if T.P[j] is None else T.P[j].copy() for j in old]
    if noise is not None and U.expanded[0]:
        flip = view == 1 and U.rec[0]["player"] == 1
        idx = np.where(flip, 8099 - U.act[0], U.act[0])
        U.P[0] = ((F32(1) + F32(-eps)) * U.P[0] + F32(eps) * noise[idx]).astype(F32)
    return U, len(old)


def assert_tree_equal(dev, T, tag):
    nodes, edges = dev
    assert len(nodes) == len(T.rec), tag
    for j in range(len(T.rec)):
        nd = nodes[j]
        assert nd["rec"].tobytes() == T.rec[j].tobytes(), (tag, j)
        assert (int(nd["parent"]), int(nd["parent_edge"]), int(nd["visits"]), int(nd["reward"]), int(nd["depth"]), int(nd["expanded"]),
                int(nd["status"]), int(nd["winner"])) == \
            (T.parent[j], T.pedge[j], T.visits[j], T.reward[j], T.depth[j], int(T.expanded[j]), T.status[j], T.winner[j]), (tag, j)
        if not T.expanded[j]:
            continue
        c = len(T.act[j])
        e = edges[j]
        assert int(nd["n_edges"]) == c and (e["action"][c:] == -1).all(), (tag, j)
        assert (e["action"][:c] == T.act[j]).all() and (e["child"][:c] == T.child[j]).all() and (e["visits"][:c] == T.N[j]).all(), (tag, j)
        assert e["value_sum"][:c].view(np.uint32).tolist() == T.W[j].view(np.uint32).tolist(), (tag, j)
        assert e["prior"][:c].view(np.uint32).tolist() == np.asarray(T.P[j], F32).view(np.uint32).tolist(), (tag, j)


def continue_replay(L, trees, log, ts, sims, seed, which):
    """the oracle continuing from its compacted trees, compared leaf by leaf; then node by node with the device's final trees (the
    priors of new expansions taken from the device, as test_search_gpu._replay does)"""
    n = ts.n
    dev = {i: ts.search.get_tree(i) for i in which}
    for s in range(sims):
        vals = _values(seed, s, n)
        for i in which:
            T = trees[i]
            j = T.select(C_PUCT, FPU)
            assert log[s]["leaves"][i].tobytes() == T.rec[j].tobytes(), (s, i, j)
            got = {k: int(log[s][k][i]) for k in ("status", "winner", "reward", "depth")}
            assert got == {"status": T.status[j], "winner": T.winner[j], "reward": T.reward[j], "depth": T.depth[j]}, (s, i, j)
            if T.status[j] == 0 and not T.expanded[j]:
                T.expand(j, dev[i][1][j]["prior"])
            T.backup(j, vals[i])
    for i in which:
        assert_tree_equal(dev[i], trees[i], ("final", i))


def root_moves(L, T, view, best, kind):
    """the policy index (frame of view) tree T's env plays: kind 0 the root's best, 1 a root edge without a child, 2 a move that ends
    the game, 3 a rejected index"""
    if kind == 3:
        return 8100 + 17
    if not T.expanded[0] or len(T.act[0]) == 0:
        return best
    flip = view == 1 and T.rec[0]["player"] == 1
    to_view = lambda a: int(8099 - a) if flip else int(a)       # noqa: E731
    if kind == 1:
        free = np.nonzero(T.child[0] < 0)[0]
        return to_view(T.act[0][free[0]]) if len(free) else best
    if kind == 2:
        for a in T.act[0]:
            r = T.rec[0][None].copy()
            act = np.array([(int(a) // 90) << 7 | (int(a) % 90)], np.uint16)
            rew = np.zeros(1, np.int32)
            done, win, cap, valid = (np.zeros(1, np.uint8) for _ in range(4))
            L.xqo_batch_step(r.ctypes.data, 1, act, rew, done, win, cap, valid)
            if done[0]:
                return to_view(a)
    return best


@pytest.mark.parametrize("view,min_free", [(0, 40), (1, 12), (1, 56)])
def test_advance_against_oracle_and_continuation(xq, torch, oracle_lib, roots257, view, min_free):
    L = oracle_lib
    recs = roots257
    n, max_sims, sims, seed = len(recs), 64, 48, 500 + view + min_free
    cap = max_sims + 1
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, max_sims)
    ts.reset()
    simulate(torch, ts, sims, seed, view, record=False)
    pre = {i: tree_from_device(L, *ts.search.get_tree(i)) for i in range(n)}
    root = ts.root(_vname(view))
    best = root.best.cpu().numpy()
    kinds = np.arange(n) % 4
    moves = np.array([root_moves(L, pre[i], view, int(best[i]), int(kinds[i])) for i in range(n)], np.int64)
    r = te.step(actions=torch.from_numpy(moves).cuda(), pick="given", view=_vname(view), auto_reset=True)
    valid, done = r.valid.cpu().numpy(), r.done.cpu().numpy()
    envs = te.env.get_boards()
    kept = ts.advance(min_free, view=_vname(view)).cpu().numpy()
    torch.cuda.synchronize()
    want_trees, want_kept = {}, np.zeros(n, np.int64)
    for i in range(n):
        want_trees[i], want_kept[i] = advance_oracle(L, pre[i], envs[i], min_free, cap)
    assert (kept == want_kept).all(), np.nonzero(kept != want_kept)
    fresh = xq.TorchSearch(te, max_sims)
    fresh.reset()
    for i in range(n):
        dev = ts.search.get_tree(i)
        assert_tree_equal(dev, want_trees[i], ("advance", i))
        if kept[i] == 0:
            assert dev[0].tobytes() == fresh.search.get_tree(i)[0].tobytes(), i
    fresh.close()
    # every kind of move was seen, each with its outcome
    sizes = np.array([len(pre[i].rec) for i in range(n)])
    rej = (kinds == 3) & (valid == 0) & (done == 0)                      # a rejected move on a finished game still resets the env
    assert rej.sum() > 40 and (kept[rej] == np.where(sizes[rej] <= cap - min_free, sizes[rej], 0)).all()     # rejected: the whole tree
    assert (kept[(valid == 0) & (done == 1)] == 0).all()
    assert ((kinds == 2) & (done == 1) & (kept == 0)).sum() > 5                                                 # game over: rebuilt
    assert ((kinds == 1) & (valid == 1) & (kept == 0)).sum() > 5                                                # no child: rebuilt
    too_large = [i for i in range(n) if kinds[i] == 0 and kept[i] == 0 and valid[i] == 1 and done[i] == 0]
    if min_free == 12:
        assert ((kinds == 0) & (kept > 1)).sum() > 10                                                           # best: subtree kept
    if min_free == 56:
        assert len(too_large) >= 3                                                                              # subtrees over budget
    # the continuation: exactly min_free simulations on the compacted trees
    seed2 = seed + 1000
    log = simulate(torch, ts, min_free, seed2, view)
    with pytest.raises(xq.XQError):
        ts.select()
    which = sorted(set(range(0, n, 3)) | set(too_large[:5]))
    continue_replay(L, want_trees, log, ts, min_free, seed2, which)
    vis, q, bst = (x.cpu().numpy() for x in ts.root(_vname(view)))
    for i in which:
        wv, wq, wb = want_trees[i].root(view)
        assert np.array_equal(vis[i], wv) and int(bst[i]) == wb, i
        assert (np.isnan(q[i]) and np.isnan(wq)) or q[i].view(np.uint32) == wq.view(np.uint32), i
    ts.close()


def test_root_noise_on_kept_and_rebuilt_roots(xq, torch, O, oracle_lib):
    L = oracle_lib
    recs = harvest_positions(O, 64, 1, 9, seed=18)
    n, max_sims, sims, seed, eps, view = 64, 40, 24, 71, 0.3, 1
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, max_sims)
    ts.reset()
    simulate(torch, ts, sims, seed, view, record=False)
    pre = {i: tree_from_device(L, *ts.search.get_tree(i)) for i in range(n)}
    best = ts.root("side").best.cpu().numpy()
    moves = np.where(np.arange(n) % 2 == 0, best, 8100 + 3)          # odd trees: rejected, the whole tree is kept
    moves[::8] = [root_moves(L, pre[i], view, int(best[i]), 1) for i in range(0, n, 8)]   # every 8th: a root edge without a child
    te.step(actions=torch.from_numpy(moves.astype(np.int64)).cuda(), pick="given", view="side")
    envs = te.env.get_boards()
    rng = np.random.default_rng(4)
    noise = rng.dirichlet(np.full(8100, 0.3), n).astype(F32)
    kept = ts.advance(16, root_noise=torch.from_numpy(noise).cuda(), noise_eps=eps, view="side").cpu().numpy()
    want = {i: advance_oracle(L, pre[i], envs[i], 16, max_sims + 1, noise[i], eps, view) for i in range(n)}
    assert (kept == np.array([want[i][1] for i in range(n)])).all()
    for i in range(n):
        assert_tree_equal(ts.search.get_tree(i), want[i][0], i)          # kept roots: search_mix(P_old, noise, eps) bit for bit
    mixed = [i for i in range(n) if kept[i] > 0 and want[i][0].expanded[0]]
    assert len(mixed) > 20
    assert any(np.abs(want[i][0].P[0] - pre[i].P[0]).max() > 1e-3 for i in mixed if i % 2)   # the mix changed kept priors
    # rebuilt roots get their noise when the next simulation expands them
    rebuilt = [i for i in range(n) if kept[i] == 0]
    assert len(rebuilt) >= 4
    seed2 = 900
    simulate(torch, ts, 1, seed2, view, noise=noise, eps=eps, record=False)
    counts, acts = P.oracle_lists(L, envs)
    idx = P.policy_indices(envs, counts, acts, 1)
    raw = _scores(seed2, 0, n)
    for i in rebuilt:
        nodes, edges = ts.search.get_tree(i)
        c = counts[i]
        w = S.priors64(raw[i, idx[i, :c]], TEMP, noise[i, idx[i, :c]], eps)
        got = edges[0]["prior"][:c].astype(np.float64)
        assert np.allclose(got, w, rtol=1e-5, atol=1e-7), i
    ts.close()


def test_call_order_budget_and_arguments(xq, torch, O):
    from cn_chess_ai_b200 import SEARCH_ADVANCE_MAX_SIMULATIONS, XQError
    n, ms = 40, 6
    te = xq.TorchEnv(n)
    ts = xq.TorchSearch(te, ms)
    sc = torch.zeros((n, 8100), device="cuda")
    val = torch.zeros(n, device="cuda")

    def refused(f, *a, **k):
        with pytest.raises(XQError):
            f(*a, **k)

    refused(ts.advance, 2)                                                # never reset
    ts.reset()
    for mf in (0, -1, ms + 1):
        refused(ts.advance, mf)
    for e in (-0.1, 1.5, float("nan")):
        refused(ts.advance, 2, noise_eps=e)
    refused(ts.search.advance_device, 2, None, 0.0, 5, None)             # view
    ts.select()
    refused(ts.advance, 2)                                                # a selection is pending
    ts.expand_backup(sc, val)
    for mf in (1, 2, 3, ms):
        size = len(ts.search.get_tree(0)[0])
        kept = ts.advance(mf)                              # the env did not move: the whole tree is kept while it leaves min_free free
        assert (kept.cpu().numpy() == (size if size <= ms + 1 - mf else 0)).all(), mf
        assert mf < ms or (kept.cpu().numpy() == 0).all()
        for _ in range(mf):
            ts.select()
            ts.expand_backup(sc, val)
        refused(ts.select)                                                 # exactly min_free selects
    ts.reset()
    for _ in range(ms):                                                    # a reset restores the full budget
        ts.select()
        ts.expand_backup(sc, val)
    refused(ts.select)
    ts.close()
    # the size bound of the compaction's shared-memory bitmap
    te1 = xq.TorchEnv(1)
    for ms, ok in ((SEARCH_ADVANCE_MAX_SIMULATIONS, True), (SEARCH_ADVANCE_MAX_SIMULATIONS + 1, False)):
        t1 = xq.TorchSearch(te1, ms)
        t1.reset()
        if ok:
            t1.select()
            t1.expand_backup(torch.zeros((1, 8100), device="cuda"), torch.zeros(1, device="cuda"))
            assert int(t1.advance(ms).item()) == 1
            nodes, edges = t1.search.get_tree(0)
            assert len(nodes) == 1 and nodes[0]["visits"] == 1 and nodes[0]["expanded"] == 1
        else:
            refused(t1.advance, 1)
        t1.close()


def _play_round(xq, torch, recs, max_sims, sims, min_free, seed, parts):
    """one search, a move of the root's best, an advance and min_free more simulations, on handles split at `parts`"""
    out = []
    for part in parts:
        te = xq.TorchEnv(len(recs[part]))
        te.env.set_boards(recs[part])
        ts = xq.TorchSearch(te, max_sims)
        ts.reset()
        n = len(recs)
        for s in range(sims):
            ts.select(C_PUCT, FPU)
            ts.expand_backup(torch.from_numpy(_scores(seed, s, n)[part]).cuda(), torch.from_numpy(_values(seed, s, n)[part]).cuda(),
                             temperature=TEMP, view="side")
        te.step(actions=ts.root("side").best, pick="given", view="side")
        kept = ts.advance(min_free)
        for s in range(min_free):
            ts.select(C_PUCT, FPU)
            ts.expand_backup(torch.from_numpy(_scores(seed + 1, s, n)[part]).cuda(), torch.from_numpy(_values(seed + 1, s, n)[part]).cuda(),
                             temperature=TEMP, view="side")
        out.append((kept, ts.root("side"), ts, te))
    return out


@pytest.mark.parametrize("n", [1, 33, 4097])
def test_sizes(xq, torch, O, oracle_lib, n):
    L = oracle_lib
    recs = harvest_positions(O, n, 1, 9 + n % 2, seed=n + 7)
    max_sims, sims, min_free, seed = 24, 12, 10, 40 + n
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, max_sims)
    ts.reset()
    simulate(torch, ts, sims, seed, 1, record=False)
    which = sorted(set(range(0, n, max(1, n // 40))) | {n - 1})
    pre = {i: tree_from_device(L, *ts.search.get_tree(i)) for i in which}
    te.step(actions=ts.root("side").best, pick="given", view="side")
    envs = te.env.get_boards()
    kept = ts.advance(min_free).cpu().numpy()
    trees = {}
    for i in which:
        trees[i], k = advance_oracle(L, pre[i], envs[i], min_free, max_sims + 1)
        assert kept[i] == k, i
        assert_tree_equal(ts.search.get_tree(i), trees[i], i)
    log = simulate(torch, ts, min_free, seed + 1, 1)
    continue_replay(L, trees, log, ts, min_free, seed + 1, which)
    ts.close()


def test_sharding(xq, torch, O):
    recs = np.concatenate([harvest_positions(O, 150, 2, 5, seed=19), random_boards(O, 40, seed=13)])
    n = len(recs)
    (k1, r1, t1, e1), = _play_round(xq, torch, recs, 32, 20, 12, 77, [slice(0, n)])
    halves = _play_round(xq, torch, recs, 32, 20, 12, 77, [slice(0, 91), slice(91, n)])
    assert torch.equal(torch.cat([h[0] for h in halves]), k1)
    assert torch.equal(torch.cat([h[1].visits for h in halves]), r1.visits)
    assert torch.equal(torch.cat([h[1].q for h in halves]).view(torch.int32), r1.q.view(torch.int32))
    assert torch.equal(torch.cat([h[1].best for h in halves]), r1.best)
    for i, j in ((0, 0), (90, 90), (91, 0), (n - 1, n - 92)):
        h = halves[0] if i < 91 else halves[1]
        a, b = t1.search.get_tree(i), h[2].search.get_tree(j)
        assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes(), i
    for _, _, t, _ in [(k1, r1, t1, e1)] + halves:
        t.close()


def test_end_to_end_with_a_torch_network(xq, torch, O, oracle_lib):
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Conv2d(14, 16, 3, padding=1), torch.nn.ReLU(), torch.nn.Flatten(), torch.nn.Linear(16 * 90, 8101)).cuda()

    def evaluate(planes):
        with torch.no_grad():
            out = net(planes.float())
        return out[:, :8100].contiguous(), torch.tanh(out[:, 8100])

    n, max_sims, sims, moves = 64, 64, 32, 8
    te = xq.TorchEnv(n, seed=1)
    ts = xq.TorchSearch(te, max_sims)
    ref = O.new_envs(n)
    kept_share = []
    for mv in range(moves):
        if mv == 0:
            root = ts.run(evaluate, sims, c_puct=1.5, view="side", obs_dtype=torch.float32)
        else:
            kept = ts.advance(sims)
            kept_share.append(float((kept > 0).float().mean()))
            root = ts.run(evaluate, sims, c_puct=1.5, view="side", obs_dtype=torch.float32, reset=False)
        for i in range(0, n, 7):
            nodes, edges = ts.search.get_tree(i)
            c = int(nodes[0]["n_edges"])
            assert int(edges[0]["visits"][:c].sum()) == int(nodes[0]["visits"]) - 1, (mv, i)
        best = root.best.cpu().numpy()
        r = te.step(actions=root.best, pick="given", view="side")
        assert (r.valid.cpu().numpy() == 1).all(), mv
        flip = ref["player"] == 1
        a = np.where(flip, 8099 - best, best)
        act = ((a // 90) << 7 | (a % 90)).astype(np.uint16)
        rew = np.zeros(n, np.int32)
        done, win, cap, valid = (np.zeros(n, np.uint8) for _ in range(4))
        oracle_lib.xqo_batch_step(ref.ctypes.data, n, act, rew, done, win, cap, valid)
        assert (valid == 1).all()
        for i in np.nonzero(done)[0]:
            c = ref[i]["ctr"]
            oracle_lib.xqo_reset(ref[i:i + 1].ctypes.data)
            ref[i]["ctr"] = c
        assert te.env.get_boards().tobytes() == ref.tobytes(), mv
    assert np.mean(kept_share) > 0.5, kept_share                       # most trees keep a subtree
    ts.close()
