"""GPU tests of the compact rows (include/xq.h: XQ_COMPACT_ACTIONS): the action lists of envs and search leaves against the oracle, and
every compact reader or writer against its dense counterpart bit for bit -- the dense row D holds garbage (NaN, +-inf) off the legal
entries and the compact row is C[k] = D[actions[k]] -- for the env step, the tree search, the Gumbel begin, the example sample and the
torch layer's run(compact=True); one compact call at 65,536 trees x 32 leaves; and the argument and call-order checks."""

import numpy as np
import pytest

import compact as CP
from conftest import harvest_positions, random_boards
from test_search_gpu import _scores, _values

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _boards(O, n, seed):
    """n boards: reachable positions of both colours to move, arbitrary boards (generic path), player bytes 2 (no legal action)"""
    reach = np.concatenate([harvest_positions(O, max(1, n // 2), 1, 7, seed=seed), harvest_positions(O, max(1, n // 2), 1, 4, seed=seed + 1)])
    arb = random_boards(O, max(1, n // 8), seed=seed + 2)
    recs = np.concatenate([reach, arb])[:n].copy()
    rng = np.random.default_rng(seed)
    recs = recs[rng.permutation(len(recs))]
    if n >= 8:
        recs["player"][rng.choice(n, max(1, n // 64), replace=False)] = 2
    recs["ctr"] = np.arange(n, dtype=np.uint32) * 11 + 3
    return recs


def _tenv(xq, recs, seed=0):
    te = xq.TorchEnv(len(recs), seed=seed)
    te.env.set_boards(recs)
    return te


def _vname(view):
    return "side" if view == 1 else "absolute"


def _gather(torch, D, actions):
    """C[k] = D[actions[k]] on the device (entries past the count take D[0]: never read)"""
    return torch.gather(D, 1, actions.clamp(min=0).to(torch.int64)).contiguous()


# ---- lists ----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 33, 4097])
def test_env_legal_actions_equal_oracle(xq, torch, O, oracle_lib, n):
    recs = _boards(O, n, seed=100 + n)
    te = _tenv(xq, recs)
    for view in (0, 1):
        want, wc = CP.compact_lists(oracle_lib, recs, view)
        acts, counts = te.legal_actions(_vname(view))
        assert acts.shape == (n, 128) and acts.dtype == torch.int32 and counts.dtype == torch.uint8
        assert (counts.cpu().numpy() == wc).all(), view
        assert (acts.cpu().numpy() == want).all(), view
    te.close()


def test_env_legal_actions_standard_handle(xq, torch, O, oracle_lib):
    """a handle without injected boards runs the generator only; non-standard piece sets injected later take the generic kernel"""
    te = xq.TorchEnv(300, seed=4)
    for _ in range(5):
        te.step(torch.randn(300, 8100, device=te.device), pick="sample")
    recs = te.env.get_boards()
    want, wc = CP.compact_lists(oracle_lib, recs, 1)
    acts, counts = te.legal_actions()
    assert (acts.cpu().numpy() == want).all() and (counts.cpu().numpy() == wc).all()
    odd = random_boards(O, 300, seed=9)
    te.env.set_boards(odd)
    want, wc = CP.compact_lists(oracle_lib, odd, 1)
    acts, counts = te.legal_actions()
    assert (acts.cpu().numpy() == want).all() and (counts.cpu().numpy() == wc).all()
    te.close()


def test_leaf_actions_equal_oracle(xq, torch, O, oracle_lib):
    recs = _boards(O, 97, seed=7)
    te = _tenv(xq, recs)
    ts = xq.TorchSearch(te, 40, max_leaves=8)
    ts.reset()
    for s, L in enumerate((8, 1, 8, 3)):
        sel = ts.select() if L == 1 else ts.select_leaves(L)
        leaves = ts.leaves().cpu().numpy().view(O.ENV_DTYPE).reshape(-1)
        for view in (0, 1):
            want, wc = CP.compact_lists(oracle_lib, leaves, view)
            acts, counts = ts.leaf_actions(_vname(view))
            assert acts.shape == (97 * L, 128)
            assert (acts.cpu().numpy() == want).all() and (counts.cpu().numpy() == wc).all(), (s, view)
        if s == 0:
            # every descent after the first stops at the unexpanded root (terminal roots are ordinary slots): duplicates get its list
            open_root = sel.status[:, 0] == 0
            assert open_root.sum() > 50 and (sel.status[open_root, 1:] == 4).all()
        acts, _ = ts.leaf_actions("absolute")
        D = torch.from_numpy(_scores(5, s, 97 * L)).cuda()
        ts.expand_backup_compact(_gather(torch, D, acts), torch.from_numpy(_values(5, s, 97 * L)).cuda())
    # after compact expansion, every expanded node's edges are its record's list (absolute)
    for t in range(0, 97, 7):
        nodes, edges = ts.search.get_tree(t)
        ex = nodes["expanded"] == 1
        want, wc = CP.compact_lists(oracle_lib, nodes["rec"][ex], 0)
        assert (edges["action"][ex] == want).all() and (nodes["n_edges"][ex] == wc).all(), t
    ts.close()
    te.close()


# ---- env step -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("view", [0, 1])
@pytest.mark.parametrize("sdt", ["f32", "bf16"])
def test_step_compact_equals_dense(xq, torch, O, view, sdt):
    n = 2085
    recs = _boards(O, n, seed=300 + view)
    a, b = _tenv(xq, recs, seed=11), _tenv(xq, recs, seed=11)
    dt = torch.float32 if sdt == "f32" else torch.bfloat16
    rng = np.random.default_rng(view)
    vn = _vname(view)
    for ply in range(12):
        pick = ("greedy", "sample", "given")[ply % 3]
        D = torch.from_numpy(CP.garbage_dense(rng, n)).cuda()
        D[rng.random(n) < 0.05] = -float("inf")                              # all -inf rows
        D = D.to(dt)
        acts, counts = a.legal_actions(vn)
        Cm = _gather(torch, D, acts)
        given = None
        if pick == "given":
            k = torch.from_numpy(rng.integers(0, 130, n)).cuda()
            given = torch.gather(acts, 1, k.clamp(max=127)[:, None].to(torch.int64))[:, 0].to(torch.int64)
            given = torch.where(k >= 128, torch.from_numpy(rng.integers(-2, 8200, n)).cuda(), given).contiguous()
        ra = a.step(D if ply % 6 != 5 else None if pick == "given" else D, actions=given, pick=pick, temperature=0.7, view=vn)
        rb = b.step_compact(Cm if ply % 6 != 5 else None if pick == "given" else Cm, actions=given, pick=pick, temperature=0.7, view=vn)
        for f in ("actions", "reward", "done", "winner", "captured", "valid"):
            assert torch.equal(getattr(ra, f), getattr(rb, f)), (ply, f)
        assert (ra.logp.cpu().numpy().view(np.uint32) == rb.logp.cpu().numpy().view(np.uint32)).all(), ply
        assert a.env.get_boards().tobytes() == b.env.get_boards().tobytes(), ply
    a.close()
    b.close()


# ---- search ---------------------------------------------------------------------------------------------------------------------------
def _trees_equal(sa, sb, n):
    for t in range(n):
        na, ea = sa.get_tree(t)
        nb, eb = sb.get_tree(t)
        assert na.tobytes() == nb.tobytes(), t
        for j in range(len(na)):
            c = int(na["n_edges"][j])
            assert ea[j, :c].tobytes() == eb[j, :c].tobytes(), (t, j)
            assert (ea["action"][j] == eb["action"][j]).all() and (ea["child"][j] == eb["child"][j]).all(), (t, j)


def _twin_move(torch, ta, tb, plan, view, seed, t=0.8):
    """one move on twin searches: dense expand_backup on ta, compact on tb, the same seeded D"""
    vn = _vname(view)
    for s, L in enumerate(plan):
        sa = ta.select() if L == 1 else ta.select_leaves(L, virtual_loss=0.5)
        sb = tb.select() if L == 1 else tb.select_leaves(L, virtual_loss=0.5)
        for f in sa._fields:
            assert torch.equal(getattr(sa, f), getattr(sb, f)), (s, f)
        rows = ta._rows
        D = torch.from_numpy(_scores(seed, s, rows)).cuda()
        v = torch.from_numpy(_values(seed, s, rows)).cuda()
        acts, _ = tb.leaf_actions(vn)
        ta.expand_backup(D, v, t, view=vn)
        tb.expand_backup_compact(_gather(torch, D, acts), v, t)


@pytest.mark.parametrize("L", [1, 8, 32])
def test_search_compact_equals_dense(xq, torch, O, L):
    n = 70
    recs = _boards(O, n, seed=500 + L)
    view = L % 2
    vn = _vname(view)
    ea, eb = _tenv(xq, recs, seed=3), _tenv(xq, recs, seed=3)
    ta, tb = xq.TorchSearch(ea, 96, max_leaves=L), xq.TorchSearch(eb, 96, max_leaves=L)
    plan = [1] + [L] * ((64 - 1) // L) + ([(64 - 1) % L] if (64 - 1) % L else [])
    ta.reset(); tb.reset()
    _twin_move(torch, ta, tb, plan, view, seed=L)
    _trees_equal(ta.search, tb.search, n)
    for f, x, y in zip(("visits", "q", "best"), ta.root(vn), tb.root(vn)):
        assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes(), f
    pa, pb = ta.play(1.0, 30, vn), tb.play(1.0, 30, vn)
    for f in ("actions", "reward", "done", "winner", "captured", "valid"):
        assert torch.equal(getattr(pa, f), getattr(pb, f)), f
    assert ea.env.get_boards().tobytes() == eb.env.get_boards().tobytes()
    ka, kb = ta.advance(32, view=vn), tb.advance(32, view=vn)
    assert torch.equal(ka, kb)
    _twin_move(torch, ta, tb, [1] + [min(L, 31)], view, seed=100 + L)
    _trees_equal(ta.search, tb.search, n)
    for x, y in zip(ta.root(vn), tb.root(vn)):
        assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()
    for o in (ta, tb, ea, eb):
        o.close()


# ---- Gumbel ---------------------------------------------------------------------------------------------------------------------------
def test_gumbel_begin_compact_equals_dense(xq, torch, O):
    n, L = 90, 4
    recs = _boards(O, n, seed=700)
    ea, eb = _tenv(xq, recs, seed=5), _tenv(xq, recs, seed=5)
    ta, tb = xq.TorchSearch(ea, 40, max_leaves=L), xq.TorchSearch(eb, 40, max_leaves=L)
    ga, gb = xq.TorchGumbel(ta, 8), xq.TorchGumbel(tb, 8)
    for dt in (torch.float32, torch.bfloat16):
        ta.reset(); tb.reset()
        D = torch.from_numpy(_scores(70, 0, n)).cuda().to(dt)
        v = torch.from_numpy(_values(70, 0, n)).cuda()
        acts, _ = eb.legal_actions("side")
        ga.begin(D, v, 24, seed=9)
        gb.begin_compact(_gather(torch, D, acts), v, 24, seed=9)
        for t in range(n):
            x, y = ga.gumbel.get(t), gb.gumbel.get(t)
            for k in x:
                assert np.asarray(x[k]).tobytes() == np.asarray(y[k]).tobytes(), (t, k)
        _trees_equal(ta.search, tb.search, n)
        for s in range(6):
            sa, sb = ga.select(L), gb.select(L)
            for f in sa._fields:
                assert torch.equal(getattr(sa, f), getattr(sb, f)), (s, f)
            D = torch.from_numpy(_scores(71, s, n * L)).cuda()
            v = torch.from_numpy(_values(71, s, n * L)).cuda()
            acts, _ = tb.leaf_actions("side")
            ta.expand_backup(D, v)
            tb.expand_backup_compact(_gather(torch, D, acts), v)
        _trees_equal(ta.search, tb.search, n)
        for x, y in zip(ga.root(), gb.root()):
            assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()
    pa, pb = ga.play(), gb.play()
    for f in ("actions", "reward", "done", "winner", "captured", "valid"):
        assert torch.equal(getattr(pa, f), getattr(pb, f)), f
    for o in (ga, gb, ta, tb, ea, eb):
        o.close()


# ---- examples -------------------------------------------------------------------------------------------------------------------------
def _dense_eval(torch, n_rows, seed):
    state = {"s": 0}

    def ev(planes, actions=None):
        s = state["s"]
        state["s"] += 1
        D = torch.from_numpy(_scores(seed, s, planes.shape[0])).cuda()
        v = torch.from_numpy(_values(seed, s, planes.shape[0])).cuda()
        return (D if actions is None else _gather(torch, D, actions)), v
    return ev


def test_sample_compact_equals_dense(xq, torch, O):
    n = 64
    te = xq.TorchEnv(n, seed=21)
    ts = xq.TorchSearch(te, 24, max_leaves=4)
    tg = xq.TorchGumbel(ts, 8)
    ex = xq.TorchExamples(ts, 1000)
    for view in ("side", "absolute"):
        s = ex.sample(300, 5, 1, view=view, compact=True)
        assert (s.index == -1).all() and (s.counts == 0).all() and (s.actions == -1).all() and (s.policy == 0).all()
        assert torch.isnan(s.value).all() and torch.isnan(s.q).all() and (s.planes == 0).all()
    ev = _dense_eval(torch, n, 33)
    for move in range(8):
        if move % 2:
            tg.run(ev, 16, seed=move, leaves=4)
            ex.record_gumbel(tg)
            st = tg.play()
        else:
            ts.run(ev, 16, leaves=4)
            ex.record(ts)
            st = ts.play(1.0, 30)
        ended = torch.ones(n, dtype=torch.bool, device=te.device) if move == 7 else st.done != 0
        ex.end_games(ended.contiguous(), torch.ones(n, dtype=torch.float32, device=te.device))
    assert len(ex) > 100
    for view in ("side", "absolute"):
        for dt in (torch.float32, torch.bfloat16):
            d = ex.sample(4099, 17, 3, view=view, dtype=dt)
            c = ex.sample(4099, 17, 3, view=view, dtype=dt, compact=True)
            assert torch.equal(d.index, c.index) and torch.equal(d.planes, c.planes)
            assert d.value.cpu().numpy().tobytes() == c.value.cpu().numpy().tobytes()
            assert d.q.cpu().numpy().tobytes() == c.q.cpu().numpy().tobytes()
            idx = c.index.cpu().numpy()
            raw = ex.get()[idx]
            assert (c.counts.cpu().numpy() == raw["n_edges"]).all()
            acts = c.actions.cpu().numpy()
            live = acts >= 0
            assert (live.sum(1) == raw["n_edges"]).all()
            pol, dp = c.policy.cpu().numpy(), d.policy.cpu().numpy()
            assert (pol[~live] == 0).all()
            got = np.take_along_axis(dp, np.maximum(acts, 0).astype(np.int64), axis=1)
            assert (got[live].view(np.uint32) == pol[live].view(np.uint32)).all()
            rest = dp.copy()
            np.put_along_axis(rest, np.maximum(acts, 0).astype(np.int64), 0.0, axis=1)
            assert (rest == 0).all()
            flip = (raw["rec"]["player"] == 1) & (view == "side")
            stored = raw["action"].astype(np.int32)
            want = np.where(flip[:, None] & (stored >= 0), 8099 - stored, stored)
            assert (acts == want).all()
    for o in (ex, tg, ts, te):
        o.close()


# ---- torch layer ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gumbel", [False, True])
def test_run_compact_equals_dense(xq, torch, O, gumbel):
    n = 80
    recs = _boards(O, n, seed=900)
    ea, eb = _tenv(xq, recs, seed=8), _tenv(xq, recs, seed=8)
    ta, tb = xq.TorchSearch(ea, 64, max_leaves=8), xq.TorchSearch(eb, 64, max_leaves=8)
    if gumbel:
        ga, gb = xq.TorchGumbel(ta, 8), xq.TorchGumbel(tb, 8)
    for move in range(3):
        if gumbel:
            ra = ga.run(_dense_eval(torch, n, 40 + move), 32, seed=move, leaves=8, reset=move == 0)
            rb = gb.run(_dense_eval(torch, n, 40 + move), 32, seed=move, leaves=8, reset=move == 0, compact=True)
            pa, pb = ga.play(), gb.play()
        else:
            kw = dict(leaves=8, dirichlet_alpha=0.3, noise_seed=move, reset=move == 0)
            ra = ta.run(_dense_eval(torch, n, 40 + move), 32, **kw)
            rb = tb.run(_dense_eval(torch, n, 40 + move), 32, compact=True, **kw)
            pa, pb = ta.play(1.0, 30), tb.play(1.0, 30)
        for x, y in zip(ra, rb):
            assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes(), move
        for f in ("actions", "reward", "done", "winner", "captured", "valid"):
            assert torch.equal(getattr(pa, f), getattr(pb, f)), (move, f)
        ta.advance(32); tb.advance(32)
    _trees_equal(ta.search, tb.search, n)
    with pytest.raises(ValueError):
        tb.run(_dense_eval(torch, n, 1), 4, compact=True, root_noise=torch.zeros(n, 8100, device=eb.device))
    for o in ([ga, gb] if gumbel else []) + [ta, tb, ea, eb]:
        o.close()


# ---- scale ----------------------------------------------------------------------------------------------------------------------------
def test_compact_search_65536_trees_32_leaves(xq, torch, O):
    """the configuration whose dense scores (2,097,152 rows x 8,100 f32 = 68 GB) do not fit: one compact call at 65,536 x 32, checked
    against the dense call on a sample of trees restated as a small search of the same boards"""
    n, L = 65536, 32
    te = xq.TorchEnv(n, seed=2)
    for _ in range(3):
        te.step(torch.randn(n, 8100, device=te.device, dtype=torch.bfloat16), pick="sample")
    recs = te.env.get_boards()
    ts = xq.TorchSearch(te, 40, max_leaves=L)
    ts.reset()
    ts.select()
    g = torch.Generator(device=te.device).manual_seed(1)
    c1 = torch.randn(n, 128, device=te.device, generator=g)
    v1 = torch.rand(n, device=te.device, generator=g) * 2 - 1
    ts.expand_backup_compact(c1, v1)
    ts.select_leaves(L)
    acts, _ = ts.leaf_actions()
    c2 = torch.randn(n * L, 128, device=te.device, generator=g)
    v2 = torch.rand(n * L, device=te.device, generator=g) * 2 - 1
    ts.expand_backup_compact(c2, v2)
    torch.cuda.synchronize()
    sample = np.random.default_rng(0).choice(n, 48, replace=False)
    sample[-1] = n - 1
    small = _tenv(xq, recs[sample], seed=2)
    ss = xq.TorchSearch(small, 40, max_leaves=L)
    ss.reset()
    ss.select()
    idx = torch.from_numpy(sample).cuda()

    def dense(Cm, A):
        """the dense row of compact row Cm: entry k at A[k], NaN off the list (padding goes to a spare column)"""
        D = torch.full((Cm.shape[0], 8101), float("nan"), device=te.device)
        D.scatter_(1, torch.where(A >= 0, A, 8100).to(torch.int64), Cm)
        return D[:, :8100].contiguous()
    a1, _ = small.legal_actions()
    ss.expand_backup(dense(c1[idx], a1), v1[idx].contiguous())
    ss.select_leaves(L)
    rows = (idx[:, None] * L + torch.arange(L, device=te.device)[None, :]).reshape(-1)
    a2, _ = ss.leaf_actions()
    assert torch.equal(a2, acts[rows])
    ss.expand_backup(dense(c2[rows], a2), v2[rows].contiguous())
    for i, t in enumerate(sample):
        na, ea_ = ts.search.get_tree(int(t))
        nb, eb_ = ss.search.get_tree(i)
        assert na.tobytes() == nb.tobytes(), t
        for j in range(len(na)):
            c = int(na["n_edges"][j])
            assert ea_[j, :c].tobytes() == eb_[j, :c].tobytes(), (t, j)
    for o in (ss, small, ts, te):
        o.close()


# ---- errors ---------------------------------------------------------------------------------------------------------------------------
def test_compact_errors(xq, torch, O):
    n = 40
    te = xq.TorchEnv(n, seed=1)
    ts = xq.TorchSearch(te, 8, max_leaves=2)
    tg = xq.TorchGumbel(ts, 4)
    ex = xq.TorchExamples(ts, 16)
    L = xq.lib()
    dev = te.device
    buf = torch.zeros(n * 2 * 128 + 8, dtype=torch.float32, device=dev)
    ok, mis = buf.data_ptr(), buf.data_ptr() + 4
    ib = torch.zeros(n * 2 * 128 + 8, dtype=torch.int32, device=dev)
    v = torch.zeros(n * 2, dtype=torch.float32, device=dev)
    E, S, G, X = te.env._h, ts.search._h, tg.gumbel._h, ex.examples._h
    te._enter()
    assert L.xq_env_legal_actions_device(E, 1, None, None) == 1
    assert L.xq_env_legal_actions_device(E, 1, ib.data_ptr() + 4, None) == 1
    assert L.xq_env_legal_actions_device(E, 3, ib.data_ptr(), None) == 1
    args = (0, 0.0, 1, 1, None, None, None, None, None, None, None)
    assert L.xq_env_policy_step_compact_device(E, ok, 2, *args) == 1           # dtype
    assert L.xq_env_policy_step_compact_device(E, mis, 0, *args) == 1          # misaligned
    assert L.xq_env_policy_step_compact_device(E, None, 0, *args) == 1         # GREEDY without scores
    # call order: XQ_ERR_STATE exactly where the dense calls give it
    for dense_rc, comp_rc in (
        (L.xq_search_expand_backup_device(S, ok, 0, 1.0, 1, v.data_ptr(), None, 0.0), L.xq_search_expand_backup_compact_device(S, ok, 0, 1.0, v.data_ptr())),
        (L.xq_search_observe_leaves_device(S, None, 0, 1, None), L.xq_search_leaf_actions_device(S, 1, ib.data_ptr(), None)),
    ):
        assert dense_rc == comp_rc == 5
    ts.reset()
    assert L.xq_search_leaf_actions_device(S, 1, ib.data_ptr(), None) == 5
    assert L.xq_search_expand_backup_compact_device(S, ok, 0, 1.0, v.data_ptr()) == 5
    ts.select_leaves(2)
    assert L.xq_search_leaf_actions_device(S, 1, ib.data_ptr(), None) == 0
    assert L.xq_search_leaf_actions_device(S, 1, None, None) == 1
    assert L.xq_search_leaf_actions_device(S, 1, ib.data_ptr() + 8, None) == 1
    assert L.xq_search_expand_backup_compact_device(S, ok, 2, 1.0, v.data_ptr()) == 1
    assert L.xq_search_expand_backup_compact_device(S, mis, 0, 1.0, v.data_ptr()) == 1
    assert L.xq_search_expand_backup_compact_device(S, ok, 0, 1.0, None) == 1
    assert L.xq_search_expand_backup_compact_device(S, ok, 0, 0.0, v.data_ptr()) == 1
    assert L.xq_gumbel_begin_compact_device(G, ok, 0, 1.0, v.data_ptr(), 4, 0, 50.0, 0.1) == 5      # a selection is pending
    assert L.xq_gumbel_begin_device(G, ok, 0, 1.0, 1, v.data_ptr(), 4, 0, 50.0, 0.1) == 5
    assert L.xq_search_expand_backup_compact_device(S, ok, 0, 1.0, v.data_ptr()) == 0
    assert L.xq_search_expand_backup_compact_device(S, ok, 0, 1.0, v.data_ptr()) == 5                # no selection pending
    assert L.xq_gumbel_begin_compact_device(G, mis, 0, 1.0, v.data_ptr(), 4, 0, 50.0, 0.1) == 1
    assert L.xq_gumbel_begin_compact_device(G, ok, 1, 1.0, None, 4, 0, 50.0, 0.1) == 1
    assert L.xq_gumbel_begin_compact_device(G, ok, 0, 1.0, v.data_ptr(), 0, 0, 50.0, 0.1) == 1
    assert L.xq_gumbel_begin_compact_device(G, ok, 0, 1.0, v.data_ptr(), 4, 0, 50.0, 0.1) == 0
    pl = torch.zeros(n * 1260 + 16, dtype=torch.float32, device=dev)
    args = (None, v.data_ptr(), v.data_ptr(), None)
    assert L.xq_examples_sample_compact_device(X, n, 1, 0, 1, pl.data_ptr(), 0, None, ok, *args) == 1
    assert L.xq_examples_sample_compact_device(X, n, 1, 0, 1, pl.data_ptr(), 0, ib.data_ptr(), None, *args) == 1
    assert L.xq_examples_sample_compact_device(X, n, 1, 0, 1, pl.data_ptr(), 0, ib.data_ptr(), mis, *args) == 1
    assert L.xq_examples_sample_compact_device(X, n, 1, 0, 1, pl.data_ptr(), 7, ib.data_ptr(), ok, *args) == 1
    assert L.xq_examples_sample_compact_device(X, 0, 1, 0, 1, pl.data_ptr(), 0, ib.data_ptr(), ok, *args) == 1
    assert L.xq_examples_sample_compact_device(X, n, 1, 0, 1, None, 0, ib.data_ptr(), ok, *args) == 0
    with pytest.raises(ValueError):
        te.step_compact(torch.zeros(n, 8100, device=dev))
    with pytest.raises(ValueError):
        ts.run(_dense_eval(torch, n, 1), 2, compact=True, root_noise=torch.zeros(n, 8100, device=dev))
    torch.cuda.synchronize()
    for o in (ex, tg, ts, te):
        o.close()
