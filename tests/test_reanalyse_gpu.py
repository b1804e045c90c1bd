"""GPU tests of reanalyse (xq_examples_load_device, xq_examples_refresh_device / _gumbel_device, TorchExamples.load / refresh /
reanalyse): loaded env boards against get() and sample(); refreshed slots against a second buffer that records the same trees and
against the numpy oracle of test_examples_gpu (both root rules, both views, one and four leaves per selection, dense and compact rows);
untouched fields and slots byte for byte; a fixed point (self-play with an evaluator that is exact per row, then every slot reanalysed
with the same settings reads back identical); every status; sampling after a refresh; 65,536 rows against a wrapped ring of 2^21 slots;
the call-order and argument errors."""
import numpy as np
import pytest

from conftest import harvest_positions
from test_examples_gpu import Oracle, search_move, targets_numpy, trees_of

pytestmark = pytest.mark.gpu

F32 = np.float32
REFRESHED, NO_SLOT, DUPLICATE, STALE, UNSEARCHED = 0, 1, 2, 3, 4
TARGETS = ["n_edges", "q", "total_visits", "action", "visits"]          # the fields a refresh writes
KEEP = ["rec", "env", "game", "ply", "reserved0", "z", "reserved1"]     # the fields it leaves


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


def fill_ring(xq, torch, recs, capacity, moves, sims=8, seed=3):
    """self-play of len(recs) envs for `moves` moves on seeded random scores (a reset every move), every game ended after the last one:
    len(recs) * moves committed examples"""
    n = len(recs)
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    tx = xq.TorchExamples(te, capacity, moves)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    for _ in range(moves):
        search_move(torch, ts, sims, gen, True)
        tx.record(ts)
        tx.finish(te.step(actions=ts.root().best, pick="given", auto_reset=True), cap_value=-0.5)
    tx.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.linspace(-1, 1, n, device="cuda"))
    return te, ts, tx


def proj_eval(torch, seed):
    """a scoring function unlike self-play's random scores: a fixed random projection of the planes; compact rows gather the dense row"""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    w = torch.randn((1260, 32), generator=g, device="cuda") * 0.3
    p = torch.randn((32, 8100), generator=g, device="cuda")

    def ev(planes, actions=None):
        h = torch.tanh(planes.float().reshape(len(planes), -1) @ w)
        scores, v = h @ p, torch.tanh(h.sum(1))
        return (scores, v) if actions is None else (scores.gather(1, actions.clamp(min=0).long()), v)
    return ev


def recorded(xq, torch, runner, gumbel):
    """the examples record() (record_gumbel()) stores from the trees of `runner`, one per env in env order"""
    te = runner.tenv
    m = te.n
    tx2 = xq.TorchExamples(te, m, 1)
    if gumbel:
        tx2.record_gumbel(runner)
    else:
        tx2.record(runner)
    tx2.end_games(torch.ones(m, dtype=torch.bool, device="cuda"), torch.zeros(m, device="cuda"))
    out = tx2.get(0, m)
    assert tx2.info()["stale"] == 0
    tx2.close()
    return out


def check_refreshed(before, after, index, rows, rec2):
    """rows REFRESHED: the slot's targets are rec2's, everything else of the slot and every other slot is as before"""
    slots = index[rows]
    for f in TARGETS:
        assert after[slots][f].tobytes() == rec2[rows][f].tobytes(), f
    for f in KEEP:
        assert after[slots][f].tobytes() == before[slots][f].tobytes(), f
    rest = np.setdiff1d(np.arange(len(before)), slots)
    assert after[rest].tobytes() == before[rest].tobytes()


@pytest.mark.parametrize("view", [0, 1])
def test_load(xq, torch, O, view):
    te, ts, tx = fill_ring(xq, torch, harvest_positions(O, 48, 1, 7, seed=21), capacity=300, moves=4)
    ring, size = tx.get(), tx.info()["size"]
    assert size == 192
    m = 80
    te2 = xq.TorchEnv(m)
    te2.env.set_boards(harvest_positions(O, m, 1, 3, seed=22))
    orig = te2.env.get_boards()
    rng = np.random.default_rng(view)
    index = rng.integers(0, size, m).astype(np.int64)
    index[[0, 13]] = -1
    index[[7, 70]] = size
    index[50] = 300 + 3
    tx.load(te2, torch.from_numpy(index).cuda())
    got = te2.env.get_boards()
    held = (index >= 0) & (index < size)
    assert got[held].tobytes() == ring[index[held]]["rec"].tobytes()
    assert got[~held].tobytes() == orig[~held].tobytes()
    # the loaded env shows what sample() shows for the same slots
    for dt in (torch.float32, torch.bfloat16):
        s = tx.sample(m, 99, 5 + view, view=_vname(view), dtype=dt)
        tx.load(te2, s.index)
        planes, _ = te2.observe(dt, _vname(view))
        assert torch.equal(planes, s.planes)
    tx.close()
    ts.close()


@pytest.mark.parametrize("compact", [False, True], ids=["dense", "compact"])
@pytest.mark.parametrize("leaves", [1, 4])
@pytest.mark.parametrize("view", [0, 1])
@pytest.mark.parametrize("gumbel", [False, True], ids=["puct", "gumbel"])
def test_refresh_against_record(xq, torch, O, gumbel, view, leaves, compact):
    te, ts, tx = fill_ring(xq, torch, harvest_positions(O, 64, 1, 7, seed=11 + view), capacity=400, moves=5)
    before, size = tx.get(), tx.info()["size"]
    m = 96
    rng = np.random.default_rng(leaves + 2 * view + 4 * compact)
    index = rng.permutation(size)[:m].astype(np.int64)
    index[[5, 40]] = -1
    index[77] = size
    index[90] = 1 << 40
    te2 = xq.TorchEnv(m, env_id0=1000)
    ts2 = xq.TorchSearch(te2, 24, max_leaves=leaves)
    runner = xq.TorchGumbel(ts2, max_considered=8) if gumbel else ts2
    status = tx.reanalyse(runner, proj_eval(torch, 5), torch.from_numpy(index).cuda(), 16, leaves=leaves, compact=compact,
                          view=_vname(view)).cpu().numpy()
    after = tx.get()
    rec2 = recorded(xq, torch, runner, gumbel)
    held = (index >= 0) & (index < size)
    want = np.where(held, np.where(rec2["total_visits"] == 0, UNSEARCHED, REFRESHED), NO_SLOT)
    assert (status == want).all()
    rows = np.nonzero(status == REFRESHED)[0]
    assert len(rows) >= 80
    assert rec2[rows]["rec"].tobytes() == before[index[rows]]["rec"].tobytes()       # the roots were the stored positions
    check_refreshed(before, after, index, rows, rec2)
    assert (after[index[rows]]["visits"] != before[index[rows]]["visits"]).any()
    # the numpy oracle of the trees (the visits are weights after a Gumbel search)
    orc = Oracle(xq, m, m, 1)
    trees = trees_of(ts2)
    fields = ["n_edges", "action", "q"] + ([] if gumbel else ["visits", "total_visits"])
    for t in rows:
        x = orc.example(t, *trees[t])
        for f in fields:
            assert after[index[t]][f].tobytes() == x[f].tobytes(), (t, f)
    if gumbel:
        runner.close()
    ts2.close()
    tx.close()
    ts.close()


def int_eval(torch, seed):
    """an evaluator whose output for a row depends on that row's planes only, bit for bit: integer arithmetic, then exact conversions"""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    wk = torch.randint(1, 1 << 20, (1260,), generator=g, device="cuda", dtype=torch.int64)
    a = torch.randint(1, 1 << 16, (8100,), generator=g, device="cuda", dtype=torch.int64)
    c = torch.randint(0, 1 << 16, (8100,), generator=g, device="cuda", dtype=torch.int64)

    def ev(planes):
        key = (planes.reshape(len(planes), -1).to(torch.int64) * wk).sum(1)
        scores = ((key[:, None] * a + c) % 1021).to(torch.float32) / 256.0
        values = ((key * 7919) % 2001 - 1000).to(torch.float32) / 1000.0
        return scores, values
    return ev


def test_fixed_point(xq, torch, O):
    """self-play with PUCT, a reset every move and no noise, then every slot reanalysed with the same evaluator and settings: the ring
    reads back identical"""
    recs = harvest_positions(O, 48, 1, 5, seed=31)
    n, sims, moves = len(recs), 12, 4
    ev = int_eval(torch, 7)
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    tx = xq.TorchExamples(te, 512, moves)
    for _ in range(moves):
        root = ts.run(ev, sims)
        tx.record(ts)
        tx.finish(te.step(actions=root.best, pick="given", auto_reset=True))
    tx.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.linspace(-1, 1, n, device="cuda"))
    before, size = tx.get(), tx.info()["size"]
    assert size == n * moves
    m = 64
    te2 = xq.TorchEnv(m)
    ts2 = xq.TorchSearch(te2, sims)
    status = []
    for first in range(0, size, m):
        index = torch.arange(first, first + m, dtype=torch.int64, device="cuda")
        status.append(tx.reanalyse(ts2, ev, index, sims).cpu().numpy())
    status = np.concatenate(status)
    assert (status[size:] == NO_SLOT).all()
    want = np.where(before["total_visits"][:size] == 0, UNSEARCHED, REFRESHED)
    assert (status[:size] == want).all()
    assert tx.get().tobytes() == before.tobytes()
    ts2.close()
    tx.close()
    ts.close()


def test_duplicates_smallest_row_wins(xq, torch, O):
    """many rows on four slots, in three calls whose winners differ: only the first row of each slot writes, and the claim words are
    restored after each call (a word left at an earlier call's smaller winner would make a later winner a duplicate)"""
    te, ts, tx = fill_ring(xq, torch, harvest_positions(O, 40, 1, 6, seed=41), capacity=200, moves=3)
    size = tx.info()["size"]
    m = 64
    te2 = xq.TorchEnv(m)
    ts2 = xq.TorchSearch(te2, 8)
    ev = proj_eval(torch, 9)
    slots = np.array([3, 17, 50, size - 1])
    winners = []
    for call in range(3):
        rng = np.random.default_rng(call)
        index = rng.choice(slots, m).astype(np.int64)
        index[:call * 10] = -1                  # the first rows move on: the winners are later rows in later calls
        before = tx.get()
        status = tx.reanalyse(ts2, ev, torch.from_numpy(index).cuda(), 8).cpu().numpy()
        rec2 = recorded(xq, torch, ts2, False)
        first = {int(s): int(np.nonzero(index == s)[0][0]) for s in slots if (index == s).any()}
        want = np.full(m, DUPLICATE, np.uint8)
        want[index < 0] = NO_SLOT
        for s, t in first.items():
            want[t] = REFRESHED if rec2[t]["total_visits"] else UNSEARCHED
        assert (status == want).all(), call
        rows = np.array(sorted(t for t in first.values() if status[t] == REFRESHED), dtype=np.int64)
        check_refreshed(before, tx.get(), index, rows, rec2)
        winners.append(first)
    assert any(winners[2][s] > winners[0][s] for s in winners[2] if s in winners[0])
    ts2.close()
    tx.close()
    ts.close()


def test_ring_wraps_between_load_and_refresh(xq, torch, O):
    """a ring of 64 slots, loaded, searched, then overwritten by the next move's commit before the refresh: STALE, and the slots keep the
    new commit"""
    recs = harvest_positions(O, 64, 1, 6, seed=51)
    n, sims = len(recs), 8
    te = xq.TorchEnv(n)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    tx = xq.TorchExamples(te, n, 2)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(5)
    ones, zeros = torch.ones(n, dtype=torch.bool, device="cuda"), torch.zeros(n, device="cuda")
    search_move(torch, ts, sims, gen, True)
    tx.record(ts)
    tx.end_games(ones, zeros)
    first = tx.get()
    te2 = xq.TorchEnv(n)
    ts2 = xq.TorchSearch(te2, sims)
    index = torch.arange(n, dtype=torch.int64, device="cuda")
    tx.load(te2, index)
    ts2.run(proj_eval(torch, 3), sims)
    te.step(actions=ts.root().best, pick="given", auto_reset=True)
    search_move(torch, ts, sims, gen, True)
    tx.record(ts)
    tx.end_games(ones, zeros)
    second = tx.get()
    status = tx.refresh(ts2, index).cpu().numpy()
    after = tx.get()
    moved = np.array([first[i]["rec"].tobytes() != second[i]["rec"].tobytes() for i in range(n)])
    assert moved.sum() >= 50
    assert (status[moved] == STALE).all() and np.isin(status[~moved], (REFRESHED, UNSEARCHED)).all()
    assert after[moved].tobytes() == second[moved].tobytes()
    ts2.close()
    tx.close()
    ts.close()


def test_empty_ring_no_slot(xq, torch, O):
    m = 16
    te2 = xq.TorchEnv(m)
    te2.env.set_boards(harvest_positions(O, m, 1, 4, seed=61))
    ts2 = xq.TorchSearch(te2, 4)
    tx = xq.TorchExamples(te2, 32, 2)
    boards = te2.env.get_boards()
    index = torch.arange(m, dtype=torch.int64, device="cuda")
    status = tx.reanalyse(ts2, proj_eval(torch, 1), index, 4).cpu().numpy()
    assert te2.env.get_boards().tobytes() == boards.tobytes()
    assert (status == NO_SLOT).all()
    assert not tx.get().tobytes().strip(b"\0") and tx.info()["size"] == 0
    tx.close()
    ts2.close()


def test_no_legal_action_root_unsearched(xq, torch, O):
    """Black to move without a piece: the stored root has no edge, and its reanalysed root has none either"""
    recs = harvest_positions(O, 4, 1, 3, seed=2)
    codes = O.codes_of(recs[0])
    codes[codes >= 8] = 0
    recs[0]["sq"] = O.pack_codes(codes)
    recs[0]["player"] = 1
    te = xq.TorchEnv(4)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, 4)
    tx = xq.TorchExamples(te, 16, 2)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    search_move(torch, ts, 4, gen, True)
    tx.record(ts)
    tx.end_games(torch.ones(4, dtype=torch.bool, device="cuda"), torch.tensor([1.0, 0, 0, 0], device="cuda"))
    before = tx.get()
    assert before[0]["n_edges"] == 0 and before[0]["total_visits"] == 0
    te2 = xq.TorchEnv(4)
    ts2 = xq.TorchSearch(te2, 4)
    status = tx.reanalyse(ts2, proj_eval(torch, 2), torch.arange(4, dtype=torch.int64, device="cuda"), 4).cpu().numpy()
    assert status.tolist() == [UNSEARCHED, REFRESHED, REFRESHED, REFRESHED]
    assert tx.get()[0].tobytes() == before[0].tobytes()
    ts2.close()
    tx.close()
    ts.close()


@pytest.mark.parametrize("view", [0, 1])
def test_sample_after_refresh(xq, torch, O, view):
    te, ts, tx = fill_ring(xq, torch, harvest_positions(O, 48, 1, 8, seed=71 + view), capacity=300, moves=4)
    before, size = tx.get(), tx.info()["size"]
    m = 96
    te2 = xq.TorchEnv(m)
    ts2 = xq.TorchSearch(te2, 16)
    for first in range(0, size, m):
        st = tx.reanalyse(ts2, proj_eval(torch, 8), torch.arange(first, first + m, dtype=torch.int64, device="cuda"), 16)
        assert np.isin(st.cpu().numpy()[:size - first], (REFRESHED, UNSEARCHED)).all()
    ring = tx.get()
    assert (ring["visits"] != before["visits"]).any() and ring["rec"].tobytes() == before["rec"].tobytes()
    batch = 700
    s = tx.sample(batch, 77, 3, view=_vname(view), dtype=torch.float32)
    idx = s.index.cpu().numpy()
    pol, _ = targets_numpy(ring, idx, view)
    assert s.policy.cpu().numpy().view(np.uint32).tolist() == pol.view(np.uint32).tolist()
    assert s.q.cpu().numpy().view(np.uint32).tolist() == ring[idx]["q"].view(np.uint32).tolist()
    c = tx.sample(batch, 77, 3, view=_vname(view), dtype=torch.float32, compact=True)
    assert torch.equal(c.index, s.index) and torch.equal(c.q.view(torch.int32), s.q.view(torch.int32))
    pc = np.zeros((batch, 128), F32)
    for i, slot in enumerate(idx):
        x = ring[slot]
        ne, tot = int(x["n_edges"]), x["total_visits"]
        if tot:
            pc[i, :ne] = x["visits"][:ne].astype(F32) / F32(tot)
    assert c.policy.cpu().numpy().view(np.uint32).tolist() == pc.view(np.uint32).tolist()
    assert (c.counts.cpu().numpy() == ring[idx]["n_edges"]).all()
    ts2.close()
    tx.close()
    ts.close()


def test_scale_65536_rows_wrapped_ring(xq, torch):
    """65,536 rows against a ring of 2^21 slots that has wrapped, checked against record() as above"""
    n, cap, copies = 65536, 1 << 21, 33
    te = xq.TorchEnv(n, seed=3)
    te.env.rollout_random(6)
    ts = xq.TorchSearch(te, 4)
    ts.run(proj_eval(torch, 4), 4)
    tx = xq.TorchExamples(te, cap, copies)
    for _ in range(copies):
        tx.record(ts)
    tx.end_games(torch.ones(n, dtype=torch.bool, device="cuda"), torch.full((n,), 0.25, device="cuda"))
    info = tx.info()
    assert info["total_committed"] == n * copies > cap and info["size"] == cap
    ts.close()
    before = tx.get()
    index = np.random.default_rng(6).choice(cap, n, replace=False).astype(np.int64)
    te2 = xq.TorchEnv(n, env_id0=n)
    ts2 = xq.TorchSearch(te2, 4)
    status = tx.reanalyse(ts2, proj_eval(torch, 5), torch.from_numpy(index).cuda(), 4).cpu().numpy()
    rec2 = recorded(xq, torch, ts2, False)
    want = np.where(rec2["total_visits"] == 0, UNSEARCHED, REFRESHED)
    assert (status == want).all() and (status == REFRESHED).sum() > n * 0.99
    rows = np.nonzero(status == REFRESHED)[0]
    slots = index[rows]
    touched = np.zeros(cap, bool)
    touched[slots] = True
    step = 1 << 18
    for first in range(0, cap, step):           # the ring after the refresh, read in parts
        part = tx.get(first, step)
        keep = ~touched[first:first + step]
        assert part[keep].tobytes() == before[first:first + step][keep].tobytes(), first
        sel = np.nonzero(touched[first:first + step])[0]
        t = np.searchsorted(slots, first + sel, sorter=np.argsort(slots))
        r = rows[np.argsort(slots)[t]]
        for f in TARGETS:
            assert part[sel][f].tobytes() == rec2[r][f].tobytes(), (first, f)
        for f in KEEP:
            assert part[sel][f].tobytes() == before[first + sel][f].tobytes(), (first, f)
    ts2.close()
    tx.close()


def test_errors(xq, torch, O):
    from cn_chess_ai_b200 import XQError
    n = 16
    te, ts, tx = fill_ring(xq, torch, harvest_positions(O, n, 1, 4, seed=81), capacity=64, moves=2, sims=4)
    te2 = xq.TorchEnv(n)
    ts2 = xq.TorchSearch(te2, 4)
    tg = xq.TorchGumbel(ts2, 4)
    idx = torch.arange(n, dtype=torch.int64, device="cuda")
    with pytest.raises(XQError, match="error 5"):
        tx.refresh(ts2, idx)                                    # never reset
    ts2.reset()
    ts2.select()
    with pytest.raises(XQError, match="error 5"):
        tx.refresh(ts2, idx)                                    # a selection pending
    ts2.expand_backup(torch.zeros((n, 8100), device="cuda"), torch.zeros(n, device="cuda"))
    assert tx.refresh(ts2, idx).shape == (n,)
    with pytest.raises(XQError, match="error 5"):
        tx.refresh_gumbel(tg, idx)                              # no begin since the reset
    bad = [torch.arange(n - 1, dtype=torch.int64, device="cuda"), idx.to(torch.int32), idx.float(), idx.reshape(4, 4), idx.cpu(),
           torch.arange(2 * n, dtype=torch.int64, device="cuda")[::2]]
    for b in bad:
        with pytest.raises(ValueError):
            tx.refresh(ts2, b)
        with pytest.raises(ValueError):
            tx.refresh_gumbel(tg, b)
        with pytest.raises(ValueError):
            tx.load(te2, b)
    for call in (lambda: tx.examples.refresh_device(ts2.search, None), lambda: tx.examples.refresh_gumbel_device(tg.gumbel, None),
                 lambda: tx.examples.load_device(te2.env, None)):
        with pytest.raises(XQError, match="error 1"):
            call()
    tg.close()
    ts2.close()
    tx.close()
    ts.close()
