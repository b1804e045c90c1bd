"""GPU tests of the batched tree search (xq_search_*, TorchSearch): whole searches replayed by the numpy restatement in search_oracle.py
(oracle lists and steps, f32 PUCT and backup) leaf by leaf and node by node, terminal roots, the root noise, the call-order and argument
checks, rerun and sharding invariance, sizes with partly empty warps and CTAs, and an end-to-end game of a small torch network."""
import numpy as np
import pytest

import policy_oracle as P
import search_oracle as S
from conftest import harvest_positions, random_boards

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _capture_next(O, L, m, seed):
    """boards where the side to move can capture the enemy General next ply (both Generals present)"""
    cand = np.concatenate([random_boards(O, 3000, seed=seed), harvest_positions(O, 400, 3, 21, seed=seed)])
    counts, acts = P.oracle_lists(L, cand)
    keep = []
    for i in range(len(cand)):
        if S.generals_missing(cand[i]) or counts[i] >= 128:
            continue
        codes = O.codes_of(cand[i])
        tgt = 8 if cand[i]["player"] == 0 else 1
        if any(codes[a & 127] == tgt for a in acts[i, :counts[i]]):
            keep.append(i)
        if len(keep) == m:
            break
    assert len(keep) == m
    return cand[keep]


@pytest.fixture(scope="module")
def trees257(O, oracle_lib):
    """257 roots: reachable positions with both colours to move, arbitrary boards (the generic path), move_count 197..199, and boards
    where a General can be captured next ply"""
    reach = harvest_positions(O, 40, 2, 7, seed=41)
    arb = random_boards(O, 60, seed=12)
    late = harvest_positions(O, 60, 1, 13, seed=5)
    late["move_count"] = 197 + np.arange(60) % 3
    cap = _capture_next(O, oracle_lib, 57, seed=77)
    recs = np.concatenate([reach, arb, late, cap])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 3 + 1
    assert len(recs) == 257 and (recs["player"] == 1).sum() > 50
    return recs


def _scores(seed, s, n):
    """seeded scores of simulation s: normal, with NaN, +-inf and all -inf rows"""
    rng = np.random.default_rng([seed, s])
    x = (rng.standard_normal((n, 8100)) * 1.5).astype(np.float32)
    x[rng.random((n, 8100)) < 0.01] = np.nan
    x[rng.random((n, 8100)) < 0.01] = -np.inf
    x[rng.random((n, 8100)) < 0.002] = np.inf
    x[rng.random(n) < 0.05] = -np.inf
    return x


def _values(seed, s, n):
    rng = np.random.default_rng([seed, s, 1])
    v = rng.uniform(-1.6, 1.6, n).astype(np.float32)
    v[rng.random(n) < 0.05] = np.nan
    return v


def _search(xq, torch, recs, sims, view, seed, c_puct=1.25, fpu=-0.1, t=0.8, sdt=None, noise=None, eps=0.25, inject=True, record=True):
    """one whole search through TorchSearch on seeded inputs: (per-simulation log, root result, trees, the search)"""
    n = len(recs)
    te = xq.TorchEnv(n)
    if inject:
        te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    ts.reset()
    nz = None if noise is None else torch.from_numpy(noise).cuda()
    log = []
    for s in range(sims):
        sel = ts.select(c_puct, fpu)
        leaves = ts.leaves().clone() if record else None
        sc = torch.from_numpy(_scores(seed, s, n)).cuda()
        if sdt is not None:
            sc = sc.to(sdt)
        ts.expand_backup(sc, torch.from_numpy(_values(seed, s, n)).cuda(), temperature=t, root_noise=nz, noise_eps=eps,
                         view="side" if view == 1 else "absolute")
        if record:
            log.append({k: getattr(sel, k).cpu().numpy() for k in ("status", "winner", "reward", "depth")} | {"leaves": leaves.cpu().numpy()})
    root = ts.root("side" if view == 1 else "absolute")
    torch.cuda.synchronize()
    return log, root, ts


def _replay(L, recs, log, ts, root, sims, view, seed, c_puct=1.25, fpu=-0.1, t=0.8, bf16=False, noise=None, eps=0.25, which=None):
    """the oracle's search with the device's priors, compared leaf by leaf, then node by node; priors checked against float64 on the
    scores as the device read them (bf16: rounded to nearest even)"""
    import torch
    n = len(recs)
    which = range(n) if which is None else which
    dev = {i: ts.search.get_tree(i) for i in which}
    trees = {i: S.Tree(L, recs[i]) for i in which}
    raw_at = {}
    for s in range(sims):
        vals = _values(seed, s, n)
        sc = _scores(seed, s, n)
        if bf16:
            sc = torch.from_numpy(sc).to(torch.bfloat16).float().numpy()
        for i in which:
            T = trees[i]
            j = T.select(c_puct, fpu)
            assert log[s]["leaves"][i].tobytes() == T.rec[j].tobytes(), (s, i, j)
            got = {k: int(log[s][k][i]) for k in ("status", "winner", "reward", "depth")}
            assert got == {"status": T.status[j], "winner": T.winner[j], "reward": T.reward[j], "depth": T.depth[j]}, (s, i, j)
            if T.status[j] == 0 and not T.expanded[j]:
                T.expand(j, dev[i][1][j]["prior"])
                flip = view == 1 and T.rec[j]["player"] == 1
                raw_at[(i, j)] = sc[i, np.where(flip, 8099 - T.act[j], T.act[j])]
            T.backup(j, vals[i])
    for i in which:
        T, (nodes, edges) = trees[i], dev[i]
        assert len(nodes) == len(T.rec), i
        for j in range(len(T.rec)):
            nd = nodes[j]
            assert nd["rec"].tobytes() == T.rec[j].tobytes(), (i, j)
            assert (int(nd["parent"]), int(nd["visits"]), int(nd["depth"]), int(nd["expanded"]), int(nd["status"]), int(nd["winner"])) == \
                (T.parent[j], T.visits[j], T.depth[j], int(T.expanded[j]), T.status[j], T.winner[j]), (i, j)
            if not T.expanded[j]:
                continue
            c = len(T.act[j])
            e = edges[j]
            assert int(nd["n_edges"]) == c and (e["action"][c:] == -1).all()
            assert (e["action"][:c] == T.act[j]).all() and (e["child"][:c] == T.child[j]).all() and (e["visits"][:c] == T.N[j]).all(), (i, j)
            assert e["value_sum"][:c].view(np.uint32).tolist() == T.W[j].view(np.uint32).tolist(), (i, j)
            if c == 0:
                continue
            # priors against float64: 1e-6 relative plus the f32 rounding of (l - m) / T, which exp turns into |l - m| / T ulps
            raw = raw_at[(i, j)]
            flip = view == 1 and T.rec[j]["player"] == 1
            nz = noise[i, np.where(flip, 8099 - T.act[j], T.act[j])] if (noise is not None and j == 0) else None
            want = S.priors64(raw, t, nz, eps)
            l = P.clean(raw)
            with np.errstate(invalid="ignore"):
                arg = np.where(np.isfinite(l) & np.isfinite(l.max()), np.abs(l - l.max()) / t, 0.0)
            tol = 1e-6 + 2.0 ** -23 * arg
            got = e["prior"][:c].astype(np.float64)
            big = want > 1e-30
            assert (np.abs(got - want)[big] <= tol[big] * want[big]).all() and (got[~big] < 1e-30).all(), (i, j)
    vis, q, best = (x.cpu().numpy() for x in root)
    for i in which:
        wv, wq, wb = trees[i].root(view)
        assert np.array_equal(vis[i], wv) and int(best[i]) == wb, i
        assert (np.isnan(q[i]) and np.isnan(wq)) or q[i].view(np.uint32) == wq.view(np.uint32), i
    return trees


@pytest.mark.parametrize("view", [0, 1])
def test_replay_against_oracle(xq, torch, oracle_lib, trees257, view):
    sims, seed = 48, 100 + view
    sdt = torch.bfloat16 if view == 1 else None
    log, root, ts = _search(xq, torch, trees257, sims, view, seed, sdt=sdt)
    trees = _replay(oracle_lib, trees257, log, ts, root, sims, view, seed, bf16=sdt is not None)
    st = np.concatenate([x["status"] for x in log])
    assert {0, 1, 2, 3}.issubset(set(st.tolist()))                   # captures, move caps and boards without a legal action were reached
    assert max(len(t.rec) for t in trees.values()) == sims             # the first simulation expands the root, each later one adds a node
    ts.close()


def test_terminal_roots(xq, torch, O, oracle_lib):
    recs = O.new_envs(4)
    recs[0]["move_count"] = 200
    codes = O.codes_of(recs[1])
    codes[codes == 1] = 0                                               # Red General gone
    recs[1]["sq"] = O.pack_codes(codes)
    recs[2]["player"] = 2
    recs[3]["player"] = 255
    sims = 5
    te = xq.TorchEnv(4)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    ts.reset()
    for s in range(sims):
        sel = ts.select(1.0, 0.0)
        st = sel.status.cpu().numpy()
        assert st.tolist() == [2, 1, 0 if s == 0 else 3, 0 if s == 0 else 3], s
        assert (sel.depth.cpu().numpy() == 0).all() and (sel.reward.cpu().numpy() == 0).all()
        assert ts.leaves().cpu().numpy().tobytes() == recs.tobytes()
        ts.expand_backup(torch.zeros((4, 8100), device="cuda"), torch.full((4,), 0.5, device="cuda"), view="side")
    vis, q, best = ts.root("side")
    assert (vis.cpu().numpy() == 0).all() and np.isnan(q.cpu().numpy()).all() and (best.cpu().numpy() == -1).all()
    assert sel.winner.cpu().numpy()[1] == 1                             # getWinner: the first General in square order is Black's
    for i in range(4):
        nodes, _ = ts.search.get_tree(i)
        assert len(nodes) == 1 and nodes[0]["visits"] == sims


def test_root_noise(xq, torch, O, oracle_lib):
    recs = harvest_positions(O, 64, 1, 9, seed=8)
    n, sims, seed, eps = 64, 6, 7, 0.3
    counts, acts = P.oracle_lists(oracle_lib, recs)
    idx = P.policy_indices(recs, counts, acts, 1)
    rng = np.random.default_rng(3)
    noise = np.zeros((n, 8100), np.float32)
    for i in range(n):
        noise[i, idx[i, :counts[i]]] = rng.dirichlet(np.full(counts[i], 0.3))
    log, root, ts = _search(xq, torch, recs, sims, 1, seed, noise=noise, eps=eps, inject=True)
    _replay(oracle_lib, recs, log, ts, root, sims, 1, seed, noise=noise, eps=eps)      # root priors checked with the mix, others without
    # the mix is visible: root priors differ from the plain softmax
    nodes, edges = ts.search.get_tree(0)
    c = counts[0]
    plain = S.priors64(_scores(seed, 0, n)[0, idx[0, :c]], 0.8)
    assert np.abs(edges[0]["prior"][:c] - plain).max() > 1e-3
    ts.close()


def test_call_order_and_argument_errors(xq, torch, O):
    from cn_chess_ai_b200 import XQError
    te = xq.TorchEnv(40)
    ts = xq.TorchSearch(te, 2)
    sc = torch.zeros((40, 8100), device="cuda")
    val = torch.zeros(40, device="cuda")
    B = ts.search

    def refused(f, *a, **k):
        with pytest.raises(XQError):
            f(*a, **k)

    refused(ts.select)                                                   # never reset
    ts.reset()
    refused(ts.observe)                                                  # observe before the first select
    refused(ts.expand_backup, sc, val)                                   # expand_backup without a select
    for c, f in ((-1.0, 0.0), (float("nan"), 0.0), (float("inf"), 0.0), (1.0, float("nan")), (1.0, float("inf"))):
        refused(ts.select, c, f)
    ts.select()
    refused(ts.select)                                                   # select twice
    planes = torch.empty(40 * 1260 + 4, dtype=torch.float32, device="cuda")
    refused(B.observe_leaves_device, planes.data_ptr() + 4, 0, 1, None)  # misaligned planes
    refused(B.observe_leaves_device, planes.data_ptr(), 3, 1, None)      # dtype
    refused(B.observe_leaves_device, planes.data_ptr(), 0, 2, None)      # view
    for t in (0.0, -1.0, float("nan"), float("inf")):
        refused(ts.expand_backup, sc, val, temperature=t)
    for e in (-0.1, 1.5, float("nan")):
        refused(ts.expand_backup, sc, val, noise_eps=e)
    refused(B.expand_backup_device, sc.data_ptr(), 2, 1.0, 1, val.data_ptr())        # scores dtype
    refused(B.expand_backup_device, sc.data_ptr(), 0, 1.0, 5, val.data_ptr())        # view
    refused(B.root_device, 5, None, None, None)                         # view
    # the handle is still usable: both simulations run and the tree has them
    ts.observe()
    ts.expand_backup(sc, val)
    ts.select()
    ts.expand_backup(sc, val)
    refused(ts.select)                                                   # past max_simulations
    nodes, _ = B.get_tree(0)
    assert nodes[0]["visits"] == 2 and len(nodes) == 2
    ts.reset()
    ts.select()
    ts.expand_backup(sc, val)
    ts.close()


def test_rerun_and_sharding(xq, torch, O):
    recs = np.concatenate([harvest_positions(O, 150, 2, 5, seed=9), random_boards(O, 40, seed=3)])
    n, sims, seed = len(recs), 24, 55
    _, r1, t1 = _search(xq, torch, recs, sims, 1, seed, record=False)
    _, r2, t2 = _search(xq, torch, recs, sims, 1, seed, record=False)
    assert torch.equal(r1.visits, r2.visits) and torch.equal(r1.q.view(torch.int32), r2.q.view(torch.int32)) and torch.equal(r1.best, r2.best)
    h = 137
    out = []
    for part in (slice(0, h), slice(h, n)):
        te = xq.TorchEnv(len(recs[part]))
        te.env.set_boards(recs[part])
        ts = xq.TorchSearch(te, sims)
        ts.reset()
        for s in range(sims):
            ts.select(1.25, -0.1)
            ts.expand_backup(torch.from_numpy(_scores(seed, s, n)[part]).cuda(), torch.from_numpy(_values(seed, s, n)[part]).cuda(),
                             temperature=0.8, view="side")
        out.append(ts.root("side"))
    assert torch.equal(torch.cat([o.visits for o in out]), r1.visits)
    assert torch.equal(torch.cat([o.q for o in out]).view(torch.int32), r1.q.view(torch.int32))
    for t in (t1, t2):
        t.close()


@pytest.mark.parametrize("n", [1, 33, 4097])
def test_sizes(xq, torch, O, oracle_lib, n):
    recs = harvest_positions(O, n, 1, 9 + n % 2, seed=n)
    sims, seed = 6, 300 + n
    log, root, ts = _search(xq, torch, recs, sims, 1, seed, inject=True)
    which = sorted(set(range(0, n, max(1, n // 40))) | {n - 1})
    _replay(oracle_lib, recs, log, ts, root, sims, 1, seed, which=which)
    ts.close()


def test_end_to_end_with_a_torch_network(xq, torch, O, oracle_lib):
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Conv2d(14, 16, 3, padding=1), torch.nn.ReLU(), torch.nn.Flatten(), torch.nn.Linear(16 * 90, 8101)).cuda()

    def evaluate(planes):
        with torch.no_grad():
            out = net(planes.float())
        return out[:, :8100].contiguous(), torch.tanh(out[:, 8100])

    n, sims, moves = 64, 32, 8
    te = xq.TorchEnv(n, seed=1)
    ts = xq.TorchSearch(te, sims)
    ref = O.new_envs(n)
    for mv in range(moves):
        root = ts.run(evaluate, sims, c_puct=1.5, view="side", obs_dtype=torch.float32)
        assert (root.visits.sum(1) == sims - 1).all(), mv           # the first simulation expands the root itself
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
    ts.close()
