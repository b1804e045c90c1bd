"""GPU tests of the self-play example buffer (xq_examples_*, TorchExamples): seeded self-play of 257 envs against a numpy oracle that
reads every root with get_tree before each record and keeps its own staging areas and ring (the ring read back with get() must equal it
bit for bit after every finish, in both views); the counters and edge cases (masks, stale roots, staging overflow, discard, ring wrap,
a root without a legal action, NaN and out-of-range results); sampled batches against TorchEnv.observe / legal_mask of the same boards
and numpy policy targets; the call-state and argument errors; sizes and a two-handle split; one training step of a small torch network."""
import numpy as np
import pytest

from conftest import harvest_positions
from test_search_gpu import _capture_next

pytestmark = pytest.mark.gpu

F32 = np.float32
C_PUCT, FPU = 1.25, -0.1


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
    """reachable positions, boards at move counts 197..199 (cap endings within three moves) and boards with a capturable General"""
    reach = harvest_positions(O, 40, 2, 7, seed=141)
    more = harvest_positions(O, 60, 1, 5, seed=9)
    late = harvest_positions(O, 60, 1, 13, seed=105)
    late["move_count"] = 197 + np.arange(60) % 3
    cap = _capture_next(O, oracle_lib, 57, seed=177)
    recs = np.concatenate([reach, more, late, cap])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 3 + 1
    return recs


def _vname(view):
    return "side" if view == 1 else "absolute"


class Oracle:
    """numpy restatement of the buffer: staging per env, ring, counters"""

    def __init__(self, xq, n, capacity, maxg, env_id0=0):
        self.dt = xq.EXAMPLE_DTYPE
        self.n, self.capacity, self.maxg, self.env_id0 = n, capacity, maxg, env_id0
        self.staged = [[] for _ in range(n)]
        self.games = [0] * n
        self.ring = np.zeros(capacity, self.dt)
        self.total = self.dropped = self.stale = 0

    def example(self, e, nodes, edges):
        x = np.zeros((), self.dt)
        r = nodes[0]
        ne = int(r["n_edges"]) if r["expanded"] else 0
        x["rec"] = r["rec"]
        x["env"] = self.env_id0 + e
        x["ply"] = len(self.staged[e])
        x["n_edges"] = ne
        x["action"][:] = -1
        x["action"][:ne] = edges[0]["action"][:ne]
        x["visits"][:ne] = edges[0]["visits"][:ne]
        tot = int(x["visits"].sum())
        sw = F32(0)
        for w in edges[0]["value_sum"][:ne]:
            sw = F32(sw + w)
        x["total_visits"] = tot
        x["q"] = F32(sw / F32(tot)) if tot else F32(np.nan)
        return x

    def record(self, trees, envs, mask=None):
        for e in range(self.n):
            if mask is not None and not mask[e]:
                continue
            nodes, edges = trees[e]
            if nodes[0]["rec"].tobytes() != envs[e].tobytes():
                self.stale += 1
            elif len(self.staged[e]) >= self.maxg:
                self.dropped += 1
            else:
                self.staged[e].append(self.example(e, nodes, edges))

    def end_games(self, ended, result):
        for e in range(self.n):
            if not ended[e]:
                continue
            r = F32(0) if np.isnan(result[e]) else F32(np.clip(result[e], F32(-1), F32(1)))
            for x in self.staged[e]:
                x["z"] = r if x["rec"]["player"] == 0 else -r
                x["game"] = self.games[e]
                self.ring[self.total % self.capacity] = x
                self.total += 1
            self.games[e] += 1
            self.staged[e] = []

    def info(self):
        return dict(size=min(self.total, self.capacity), capacity=self.capacity, total_committed=self.total,
                    pending=sum(len(s) for s in self.staged), dropped=self.dropped, stale=self.stale)


def step_result_numpy(done, captured, cap_value):
    r = np.full(len(done), F32(cap_value), F32)
    r[captured == 8] = 1
    r[captured == 1] = -1
    return done != 0, r


def targets_numpy(ring, idx, view):
    """the policy rows and packed masks of ring slots idx in the frame of view"""
    pol = np.zeros((len(idx), 8100), F32)
    mask = np.zeros((len(idx), 254), np.uint32)
    for i, s in enumerate(idx):
        if s < 0:
            continue
        x = ring[s]
        ne = int(x["n_edges"])
        a = x["action"][:ne].astype(np.int64)
        if view == 1 and x["rec"]["player"] == 1:
            a = 8099 - a
        tot = x["total_visits"]
        if tot:
            pol[i, a] = x["visits"][:ne].astype(F32) / F32(tot)
        for j in a:
            mask[i, j >> 5] |= np.uint32(1 << (j & 31))
    return pol, mask


def search_move(torch, ts, sims, gen, first):
    """reset (first move) or advance, then `sims` simulations on seeded random scores and values"""
    n = ts.n
    if first:
        ts.reset()
    else:
        ts.advance(sims, view="side")
    for _ in range(sims):
        ts.select(C_PUCT, FPU)
        sc = torch.randn((n, 8100), generator=gen, device="cuda") * 1.5
        v = torch.rand(n, generator=gen, device="cuda") * 3.2 - 1.6
        ts.expand_backup(sc, v, temperature=0.8, view="side")


def trees_of(ts):
    return [ts.search.get_tree(i) for i in range(ts.n)]


@pytest.mark.parametrize("view", [0, 1])
def test_self_play_against_oracle(xq, torch, roots257, view):
    recs = roots257
    n, sims, moves, cap_value = len(recs), 16, 7, -0.5
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 2 * sims)
    tx = xq.TorchExamples(ts, 900, max_game_examples=256)
    orc = Oracle(xq, n, 900, 256)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(31 + view)
    ended_kinds = {"capture": 0, "cap": 0}
    for mv in range(moves):
        search_move(torch, ts, sims, gen, mv == 0)
        trees = trees_of(ts)
        envs = te.env.get_boards()
        orc.record(trees, envs)
        tx.record(ts)
        best = ts.root(_vname(view)).best
        st = te.step(actions=best, pick="given", view=_vname(view), auto_reset=True)
        ended = tx.finish(st, cap_value=cap_value)
        done, captured = st.done.cpu().numpy(), st.captured.cpu().numpy()
        e_np, r_np = step_result_numpy(done, captured, cap_value)
        assert (ended.cpu().numpy() == e_np).all()
        orc.end_games(e_np, r_np)
        ended_kinds["capture"] += int(((done != 0) & np.isin(captured, (1, 8))).sum())
        ended_kinds["cap"] += int(((done != 0) & ~np.isin(captured, (1, 8))).sum())
        got = tx.get()
        assert got.tobytes() == orc.ring.tobytes(), (mv, [i for i in range(900) if got[i].tobytes() != orc.ring[i].tobytes()][:5])
        assert tx.info() == orc.info(), mv
    assert ended_kinds["capture"] >= 1 and ended_kinds["cap"] >= 30, ended_kinds
    assert orc.total > 100 and len(tx) == orc.total
    zs = np.abs(orc.ring["z"][:orc.total])
    assert (zs == 1).any() and (zs == 0.5).any()
    tx.close()
    ts.close()


def _setup(xq, torch, recs, capacity, maxg, sims=8, seed=5):
    n = len(recs)
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    tx = xq.TorchExamples(te, capacity, maxg)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    search_move(torch, ts, sims, gen, True)
    return te, ts, tx, gen


def test_counters_and_edge_cases(xq, torch, O, oracle_lib):
    recs = harvest_positions(O, 48, 1, 9, seed=23)
    n = len(recs)
    te, ts, tx, gen = _setup(xq, torch, recs, capacity=50, maxg=3)
    orc = Oracle(xq, n, 50, 3)
    trees, envs = trees_of(ts), te.env.get_boards()
    # mask subsets
    rng = np.random.default_rng(3)
    for _ in range(2):
        m = rng.random(n) < 0.5
        tx.record(ts, torch.from_numpy(m).cuda())
        orc.record(trees, envs, m)
        assert tx.info() == orc.info()
    # overflow: the first three of each env kept, the rest dropped
    for _ in range(3):
        tx.record(ts)
        orc.record(trees, envs)
    info = tx.info()
    assert info == orc.info() and info["pending"] == 3 * n and info["dropped"] > n // 2
    # discard: half the envs lose their staged examples, and their game counts stay
    half = np.arange(n) % 2 == 0
    tx.discard(torch.from_numpy(half).cuda())
    for e in np.nonzero(half)[0]:
        orc.staged[e] = []
    assert tx.info() == orc.info()
    # NaN and out-of-range results; ring wrap (50 < 3 * 24 committed)
    res = np.array([np.nan, 5.0, -7.0, 0.3, -0.0, np.inf, -np.inf, 1.0] * (n // 8), F32)
    allend = np.ones(n, bool)
    tx.end_games(torch.from_numpy(allend).cuda(), torch.from_numpy(res).cuda())
    orc.end_games(allend, res)
    got = tx.get()
    assert orc.total == 3 * (n // 2) > 50
    assert got.tobytes() == orc.ring.tobytes() and tx.info() == orc.info()
    assert set(got["z"].tolist()) <= set(F32([0, 1, -1, 0.3, -0.3]).tolist()) and np.isfinite(got["z"]).all()
    # the ring holds the last 50 examples in commit order
    order = (np.arange(orc.total - 50, orc.total)) % 50
    assert (got[order]["env"][1:] >= got[order]["env"][:-1]).all()
    # a second game: game numbers advance (discarded envs too, they were ended)
    tx.record(ts)
    orc.record(trees, envs)
    tx.discard()
    for e in range(n):
        orc.staged[e] = []
    assert tx.info()["pending"] == 0
    tx.record(ts)
    orc.record(trees, envs)
    tx.end_games(torch.from_numpy(allend).cuda(), torch.zeros(n, device="cuda"))
    orc.end_games(allend, np.zeros(n, F32))
    assert tx.get().tobytes() == orc.ring.tobytes() and (orc.ring["game"] >= 1).any()
    # stale: record after the step without a new search
    best = ts.root("side").best
    st = te.step(actions=best, pick="given", view="side", auto_reset=False)
    moved = int((st.valid.cpu().numpy() != 0).sum())
    before = tx.info()
    tx.record(ts)
    after = tx.info()
    assert moved > 40 and after["stale"] - before["stale"] == moved and after["pending"] - before["pending"] == n - moved
    assert tx.get().tobytes() == orc.ring.tobytes()
    tx.close()
    ts.close()


def test_no_legal_action_root_ended_by_end_games(xq, torch, O):
    """Black to move without a piece left: the action list is empty, so no step can end the game and the root has no edge; the game
    is ended through end_games"""
    recs = harvest_positions(O, 4, 1, 3, seed=2)
    codes = O.codes_of(recs[0])
    codes[codes >= 8] = 0
    recs[0]["sq"] = O.pack_codes(codes)
    recs[0]["player"] = 1
    te, ts, tx, gen = _setup(xq, torch, recs, capacity=16, maxg=8, sims=4)
    tx.record(ts)
    tx.end_games(torch.tensor([1, 0, 0, 0], dtype=torch.uint8, device="cuda"), torch.tensor([1.0, 0, 0, 0], device="cuda"))
    got = tx.get(0, 1)[0]
    assert got["n_edges"] == 0 and got["total_visits"] == 0 and np.isnan(got["q"]) and got["z"] == -1 and (got["action"] == -1).all()
    s = tx.sample(4, 1, 0, want_mask=True)
    assert (s.index.cpu() == 0).all() and (s.policy.cpu() == 0).all() and (s.mask.cpu() == 0).all() and (s.value.cpu() == -1).all()
    tx.close()
    ts.close()


@pytest.mark.parametrize("view", [0, 1])
def test_sample(xq, torch, roots257, view):
    recs = roots257
    n = len(recs)
    te, ts, tx, gen = _setup(xq, torch, recs, capacity=700, maxg=4, sims=12, seed=77 + view)
    # the empty ring
    s = tx.sample(33, 9, 2, view=_vname(view), dtype=torch.float32, want_mask=True)
    assert (s.index.cpu() == -1).all() and (s.planes.cpu() == 0).all() and (s.policy.cpu() == 0).all() and (s.mask.cpu() == 0).all()
    assert s.value.isnan().all() and s.q.isnan().all()
    for mv in range(2):
        if mv:
            search_move(torch, ts, 12, gen, False)
        tx.record(ts)
        te.step(actions=ts.root().best, pick="given", auto_reset=True)
    ended = torch.ones(n, dtype=torch.bool, device="cuda")
    tx.end_games(ended, torch.linspace(-1, 1, n, device="cuda"))
    size = tx.info()["size"]
    assert size == 2 * n
    ring = tx.get()
    batch, seed, counter = 1500, 123456789, 7
    want_idx = (_draw(seed, batch, counter) % np.uint64(size)).astype(np.int64)
    pol_w, mask_w = None, None
    for dt in (torch.float32, torch.bfloat16, torch.uint8):
        s = tx.sample(batch, seed, counter, view=_vname(view), dtype=dt, want_mask=True)
        idx = s.index.cpu().numpy()
        assert (idx == want_idx).all()
        chk = xq.TorchEnv(batch)
        chk.env.set_boards(ring[idx]["rec"])
        planes, _ = chk.observe(dtype=dt, view=_vname(view))
        assert torch.equal(planes, s.planes), dt
        if pol_w is None:
            pol_w, mask_w = targets_numpy(ring, idx, view)
            legal = chk.legal_mask(packed=True, view=_vname(view)).cpu().numpy().view(np.uint32)
            assert (legal == mask_w).all()          # the stored action lists are the legal sets
        assert s.policy.cpu().numpy().view(np.uint32).tolist() == pol_w.view(np.uint32).tolist()
        assert (s.mask.cpu().numpy().view(np.uint32) == mask_w).all()
        assert s.value.cpu().numpy().view(np.uint32).tolist() == ring[idx]["z"].view(np.uint32).tolist()
        assert s.q.cpu().numpy().view(np.uint32).tolist() == ring[idx]["q"].view(np.uint32).tolist()
        chk.close()
    s2 = tx.sample(batch, seed, counter, view=_vname(view))
    assert s2.mask is None and torch.equal(s2.policy, s.policy)
    tx.close()
    ts.close()


def _draw(seed, batch, counter):
    """xq_replay_sample's (xq_rng(seed, i, counter) >> 1) for i < batch"""
    from oracle import loader
    return loader.rng_np(seed, np.arange(batch), np.full(batch, counter)) >> np.uint64(1)


def test_errors(xq, torch, O):
    from cn_chess_ai_b200 import XQError
    from cn_chess_ai_b200.env import BatchedExamples
    n = 40
    te, te2 = xq.TorchEnv(n), xq.TorchEnv(n)
    ts, ts2 = xq.TorchSearch(te, 4), xq.TorchSearch(te2, 4)
    tx = xq.TorchExamples(te, 100, 8)
    with pytest.raises(XQError, match="error 5"):
        tx.record(ts)                                   # never reset
    ts.reset()
    ts.select()
    with pytest.raises(XQError, match="error 5"):
        tx.record(ts)                                   # selection pending
    ts.expand_backup(torch.zeros((n, 8100), device="cuda"), torch.zeros(n, device="cuda"))
    tx.record(ts)
    ts2.reset()
    with pytest.raises(XQError, match="error 1"):
        tx.record(ts2)                                  # another env
    for cap, mg in ((0, 8), (10, 0), (10, 65536)):
        with pytest.raises(XQError, match="error 1"):
            BatchedExamples(te.env, cap, mg)
    assert xq.examples_bytes(n, 100, 8) >= (100 + n * 8) * 864
    with pytest.raises(XQError, match="error 1"):
        xq.examples_bytes(n, 0, 8)
    planes = torch.empty((4, 14, 10, 9), dtype=torch.bfloat16, device="cuda")
    pol = torch.empty((4, 8100), device="cuda")
    for args in ((0, planes.data_ptr(), 1, pol.data_ptr(), 1), (4, None, 1, pol.data_ptr(), 1), (4, planes.data_ptr(), 1, None, 1),
                 (4, planes.data_ptr(), 7, pol.data_ptr(), 1), (4, planes.data_ptr(), 1, pol.data_ptr(), 5),
                 (4, planes.data_ptr() + 2, 1, pol.data_ptr(), 1)):
        b, pp, dt, po, v = args
        with pytest.raises(XQError, match="error 1"):
            tx.examples.sample_device(b, 0, 0, v, pp, dt, po)
    with pytest.raises(XQError, match="error 1"):
        tx.examples.end_games_device(None, None)
    with pytest.raises(XQError, match="error 1"):
        tx.examples.get(90, 20)
    with pytest.raises(ValueError):
        tx.sample(0, 0, 0)
    with pytest.raises(ValueError):
        tx.end_games(torch.ones(n - 1, dtype=torch.bool, device="cuda"), torch.zeros(n - 1, device="cuda"))
    tx.close()
    ts.close()
    ts2.close()


@pytest.mark.parametrize("n", [1, 33, 4097])
def test_sizes(xq, torch, O, n):
    """examples against the root's dense visits and q and the env boards (TorchSearch.root as the reference)"""
    recs = harvest_positions(O, n, 1, 11, seed=n)
    te, ts, tx, gen = _setup(xq, torch, recs, capacity=3 * n, maxg=2, sims=6, seed=n)
    envs = te.env.get_boards()
    root = ts.root("absolute")
    tx.record(ts)
    tx.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.full((n,), 0.5, device="cuda"))
    got = tx.get(0, n)
    vis, q = root.visits.cpu().numpy(), root.q.cpu().numpy()
    assert got["rec"].tobytes() == envs.tobytes() and (got["env"] == np.arange(n)).all() and (got["ply"] == 0).all()
    assert got["q"].view(np.uint32).tolist() == q.view(np.uint32).tolist()
    dense = np.zeros((n, 8100), np.int64)
    for i in range(n):
        ne = int(got[i]["n_edges"])
        dense[i, got[i]["action"][:ne]] = got[i]["visits"][:ne]
        assert (got[i]["action"][ne:] == -1).all() and (got[i]["visits"][ne:] == 0).all()
    assert (dense == vis).all() and (got["total_visits"] == vis.sum(1)).all()
    assert (got["z"] == np.where(envs["player"] == 0, F32(0.5), F32(-0.5))).all()
    tx.close()
    ts.close()


def test_two_handle_split(xq, torch, O):
    """env ids are global: the examples of two handles (env_id0 0 and n0) merge into those of one handle"""
    recs = harvest_positions(O, 70, 1, 9, seed=44)
    n, n0 = len(recs), 30
    sc = torch.randn((n, 8100), generator=torch.Generator(device="cuda").manual_seed(3), device="cuda")
    vals = torch.rand(n, generator=torch.Generator(device="cuda").manual_seed(4), device="cuda") * 2 - 1

    def run(lo, hi):
        te = xq.TorchEnv(hi - lo, env_id0=lo)
        te.env.set_boards(recs[lo:hi])
        ts = xq.TorchSearch(te, 3)
        tx = xq.TorchExamples(ts, 300, 4)
        ts.reset()
        for _ in range(3):
            ts.select()
            ts.expand_backup(sc[lo:hi].contiguous(), vals[lo:hi].contiguous())
        tx.record(ts)
        tx.record(ts)
        tx.end_games(torch.ones(hi - lo, dtype=torch.bool, device="cuda"), torch.full((hi - lo,), -1.0, device="cuda"))
        out = tx.get(0, 2 * (hi - lo))
        tx.close()
        ts.close()
        return out

    whole = run(0, n)
    parts = np.concatenate([run(0, n0), run(n0, n)])
    assert whole.tobytes() == parts.tobytes()


def test_end_to_end_training_step(xq, torch, O):
    """a small policy/value network plays a few moves with the search, its examples are committed and sampled, and one optimiser step
    on cross-entropy(pi, masked log-softmax) + MSE(z) runs on the batch"""
    nn = torch.nn
    torch.manual_seed(0)

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.body = nn.Sequential(nn.Flatten(), nn.Linear(1260, 64), nn.ReLU())
            self.pi = nn.Linear(64, 8100)
            self.v = nn.Linear(64, 1)

        def forward(self, x):
            h = self.body(x.float())
            return self.pi(h), torch.tanh(self.v(h)).squeeze(1)

    net = Net().cuda()
    n = 64
    te = xq.TorchEnv(n)
    te.env.set_boards(harvest_positions(O, n, 1, 4, seed=8))
    ts = xq.TorchSearch(te, 16)
    tx = xq.TorchExamples(ts, 2048)

    @torch.no_grad()
    def evaluate(planes):
        return net(planes)

    for mv in range(4):
        if mv:
            ts.advance(8)
        root = ts.run(evaluate, 8, reset=(mv == 0))
        tx.record(ts)
        st = te.step(actions=root.best, pick="given", auto_reset=True)
        tx.finish(st)
    result = torch.where(torch.arange(n, device="cuda") % 3 == 0, 1.0, -1.0)
    tx.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), result)
    assert len(tx) == 4 * n
    b = tx.sample(256, 11, 0, want_mask=True)
    ring = tx.get()
    idx = b.index.cpu().numpy()
    pol_w, mask_w = targets_numpy(ring, idx, 1)
    assert b.policy.cpu().numpy().view(np.uint32).tolist() == pol_w.view(np.uint32).tolist()
    assert (b.mask.cpu().numpy().view(np.uint32) == mask_w).all()
    assert (b.value.cpu().numpy() == ring[idx]["z"]).all()
    bits = b.mask.view(torch.int32)
    ar = torch.arange(8100, device="cuda")
    legal = ((bits[:, ar >> 5] >> (ar & 31)) & 1).bool()
    opt = torch.optim.SGD(net.parameters(), lr=0.01)
    logits, v = net(b.planes)
    logp = torch.log_softmax(logits.masked_fill(~legal, -1e9), dim=1)
    loss = -(b.policy * logp).sum(1).mean() + ((v - b.value) ** 2).mean()
    opt.zero_grad()
    loss.backward()
    assert torch.isfinite(loss)
    assert all(p.grad is not None and p.grad.abs().sum() > 0 for p in net.parameters())
    opt.step()
    tx.close()
    ts.close()
