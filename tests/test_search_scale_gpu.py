"""GPU tests of the tree search at the sizes the benchmarks run: 65,536 trees of 200 and 300 simulations (slabs of 31.5 and 47 GB, edge
arrays past 2^31 elements), multi-leaf searches at 65,539 x 8 and 65,536 x 32 (compact rows), the Gumbel root search at 65,536 x 64,
play + advance + continuation on the benchmarked trees, and the advance kernel's opt-in shared memory at 65,536 simulations.

The inputs are drawn on the device from a seeded torch.Generator; only the rows of a sample of trees come back to the host, and the
numpy oracles (search_oracle, search_leaves_oracle, gumbel_oracle, test_search_reuse_gpu.advance_oracle) replay those trees leaf by
leaf and node by node, bit for bit.  The sample is derived from the layout (node j of tree t at g = t * cap + j, its 128 edge slots at
g * 128 .. g * 128 + 127): the trees at the CTA edges of the 4-warp and 32-board kernels, the last tree, the trees whose edge block holds
byte 2^31 or 2^32 of the 4-byte edge arrays (P, N, W, child), byte 2^31 of the int16 action array and element 2^31, and a seeded random
rest that carries boards near the move cap, boards with a capturable General, arbitrary piece sets (the generic kernels) and terminal
roots.  Each boundary tree is checked to hold expanded nodes on both sides of its boundary."""
import time

import numpy as np
import pytest

import gumbel_oracle as G
import policy_oracle as P
import search_oracle as S
import search_leaves_oracle as SL
import test_search_play_cpu as H
from conftest import harvest_positions, random_boards
from test_examples_gpu import _draw, targets_numpy
from test_gumbel_gpu import check_state
from test_search_gpu import _capture_next
from test_search_reuse_gpu import advance_oracle, assert_tree_equal, tree_from_device

pytestmark = pytest.mark.gpu

F32 = np.float32
FIELDS = ("status", "winner", "reward", "depth")
C_PUCT, FPU, TEMP, VL = 1.25, -0.1, 0.8, 1.0
EDGE_SLOTS = 128                   # edge slots per node (XQ_SEARCH_MAX_EDGES)
ENV_SEED = 31
GB = 1e9

# (what lies there, element index of the per-edge arrays)
BOUNDARIES = (("byte 2^31 of the 4-byte edge arrays (P, N, W, child)", 2 ** 31 // 4),
              ("byte 2^32 of the 4-byte edge arrays (P, N, W, child)", 2 ** 32 // 4),
              ("byte 2^31 of the int16 action array", 2 ** 31 // 2),
              ("element 2^31 of every edge array", 2 ** 31))


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


# ---- which trees are checked ----------------------------------------------------------------------------------------------------------
def boundary_trees(n, cap):
    """[(what, element, tree, node)]: the tree and node whose edge block starts at each boundary the layout reaches"""
    out = []
    for what, e in BOUNDARIES:
        if e < n * cap * EDGE_SLOTS:
            g = e // EDGE_SLOTS
            assert g * EDGE_SLOTS == e                       # every boundary starts an edge block
            out.append((what, e, g // cap, g % cap))
    return out


def sample_trees(n, cap, seed, total=48):
    """(sorted trees, boundary list, trees free for special boards): CTA edges, the last tree, the boundary trees and a seeded random rest"""
    fixed = {t for t in (0, 1, 3, 4, 31, 32, n - 1) if t < n}
    bnd = boundary_trees(n, cap)
    fixed |= {b[2] for b in bnd}
    rng = np.random.default_rng(seed)
    rest = []
    while len(fixed) + len(rest) < total:
        t = int(rng.integers(0, n))
        if t not in fixed and t not in rest:
            rest.append(t)
    return sorted(fixed | set(rest)), bnd, rest


def check_boundaries(bnd, dev, cap):
    """each boundary tree has an expanded node on both sides of its boundary; returns the report lines"""
    lines = []
    for what, e, t, j in bnd:
        nodes = dev[t][0]
        ex = nodes["expanded"].astype(bool)
        assert ex[:j].any() and ex[j:].any(), (what, t, j, len(nodes))
        lo, hi = int(np.nonzero(ex[:j])[0][-1]), j + int(np.nonzero(ex[j:])[0][0])
        lines.append(f"{what}: element {e} = tree {t} node {j} (cap {cap}); expanded nodes {lo} and {hi} of {len(nodes)}")
    return lines


# ---- boards ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def specials(O, oracle_lib):
    """boards for the sampled trees of the random rest: move_count 195..199, a capturable General, arbitrary piece sets, terminal roots
    (move_count 200, a General missing, no legal action)"""
    late = harvest_positions(O, 6, 1, 11, seed=905)
    late["move_count"] = 195 + np.arange(6) % 5
    late["move_count"][5] = 199
    cap = _capture_next(O, oracle_lib, 6, seed=906)
    arb = random_boards(O, 6, seed=907)
    term = harvest_positions(O, 6, 1, 9, seed=908)
    term["move_count"][:2] = 200
    for i in (2, 3):
        codes = O.codes_of(term[i])
        codes[codes == (1 if i == 2 else 8)] = 0
        term[i]["sq"] = O.pack_codes(codes)
    term["player"][4:] = 2
    out = []
    for k in range(6):
        out += [late[k], cap[k], arb[k], term[k]]
    return np.array(out, O.ENV_DTYPE)


def boards(O, n, seed, rest, specials):
    """n reachable positions of both colours to move; the first trees of `rest` get the special boards"""
    h = n // 2
    recs = np.concatenate([harvest_positions(O, h, 1, 7, seed=seed), harvest_positions(O, n - h, 1, 8, seed=seed + 1)])
    recs = recs[np.random.default_rng(seed).permutation(n)]
    for t, b in zip(rest, specials):
        recs[t] = b
    recs["ctr"] = np.arange(n, dtype=np.uint32) * 3 + 1
    return recs


# ---- memory ---------------------------------------------------------------------------------------------------------------------------
def need_memory(torch, nbytes, what):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"{what} needs {nbytes / GB:.1f} GB of device memory, {free / GB:.1f} GB are free")


class Peak:
    """the most device memory in use since creation, above what was in use then (cudaMemGetInfo, so the library's slabs count)"""

    def __init__(self, torch):
        self.torch = torch
        torch.cuda.synchronize()
        self.base = self.low = torch.cuda.mem_get_info()[0]

    def sample(self):
        self.low = min(self.low, self.torch.cuda.mem_get_info()[0])

    def gb(self):
        return (self.base - self.low) / GB


@pytest.fixture
def handles(torch):
    """a list the test appends its library handles to (env first): closed in reverse order and torch's cache emptied after the test,
    whether it passed or not, so that the suite's later tests keep their memory"""
    hs = []
    yield hs
    for h in reversed(hs):
        h.close()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def input_bytes(rows, width, elem):
    """device bytes Recorder.inputs holds at once for one call: the scores, the f16 draw and up to four bool temporaries over them"""
    return rows * width * (elem + 2 + 4) + rows * 16


def report(name, t0, peak, lines=()):
    print(f"\n[scale] {name}: {time.time() - t0:.1f} s, peak device memory {peak.gb():.1f} GB")
    for ln in lines:
        print(f"[scale]   {ln}")


# ---- seeded inputs on the device, recorded rows of the sampled trees ------------------------------------------------------------------
class Recorder:
    """drives a search (or a Gumbel search) on scores / values drawn on the device and keeps, per call, the leaf records, select outputs,
    scores and values of the sampled trees' rows only"""

    def __init__(self, torch, ts, which, seed, view=1, sdt=None, compact=False, tg=None, peak=None, vl=VL):
        self.torch, self.ts, self.tg, self.peak = torch, ts, tg, peak
        self.which = np.asarray(which, np.int64)
        self.w = torch.from_numpy(self.which).cuda()
        self.g = torch.Generator(device="cuda").manual_seed(seed)
        self.view, self.sdt, self.compact, self.vl = view, sdt, compact, vl
        self.log = []

    def inputs(self, rows):
        """scores [rows, 8100 or 128] (normal * 1.5 with 1 % NaN, 1 % -inf, 0.2 % +inf, 5 % rows all -inf) and values f32 [rows]
        (uniform in +-1.6, 5 % NaN)"""
        torch, g = self.torch, self.g
        width = 128 if self.compact else 8100
        x = torch.randn((rows, width), generator=g, device="cuda", dtype=self.sdt or torch.float32).mul_(1.5)
        u = torch.rand((rows, width), generator=g, device="cuda", dtype=torch.float16)
        x.masked_fill_(u < 0.01, float("nan"))
        x.masked_fill_((u >= 0.01) & (u < 0.02), float("-inf"))
        x.masked_fill_((u >= 0.02) & (u < 0.022), float("inf"))
        del u
        x.masked_fill_((torch.rand(rows, generator=g, device="cuda") < 0.05)[:, None], float("-inf"))
        v = torch.rand(rows, generator=g, device="cuda").mul_(3.2).sub_(1.6)
        v.masked_fill_(torch.rand(rows, generator=g, device="cuda") < 0.05, float("nan"))
        return x, v

    def rows(self, k):
        torch = self.torch
        return (self.w[:, None] * k + torch.arange(k, device="cuda")[None, :]).reshape(-1)

    def begin(self, n_sims, seed):
        """the Gumbel begin on the roots: records the root rows and all root values (check_state reads v0 by tree)"""
        sc, v = self.inputs(self.ts.n)
        self.tg.begin(sc, v, n_sims, seed=seed, temperature=TEMP, c_visit=50.0, c_scale=0.1, view=_vname(self.view))
        self.begin_rows = {"scores": sc[self.w].float().cpu().numpy(), "values": v[self.w].cpu().numpy()}
        self.v0 = v.cpu().numpy()

    def call(self, k):
        ts = self.ts
        if self.tg is not None:
            sel = self.tg.select(k, C_PUCT, FPU, self.vl)
        elif k == 1:
            sel = ts.select(C_PUCT, FPU)
        else:
            sel = ts.select_leaves(k, C_PUCT, FPU, self.vl)
        r = self.rows(k)
        rec = {f: getattr(sel, f).reshape(-1)[r].cpu().numpy() for f in FIELDS}
        rec["leaves"] = ts.leaves()[r].cpu().numpy()
        sc, v = self.inputs(ts.n * k)
        if self.peak:
            self.peak.sample()
        rec["scores"], rec["values"], rec["k"] = sc[r].float().cpu().numpy(), v[r].cpu().numpy(), k
        if self.compact:
            ts.expand_backup_compact(sc, v, temperature=TEMP)
        else:
            ts.expand_backup(sc, v, temperature=TEMP, view=_vname(self.view))
        self.log.append(rec)
        del sc, v

    def run(self, plan):
        for k in plan:
            self.call(k)
        self.torch.cuda.synchronize()


def replay(L, trees, rec, dev, gumbel=False, calls=None):
    """the oracle trees (dict tree -> tree, in the recorder's order) through the recorded calls (all, or the range `calls`), compared
    slot by slot; the device's priors are taken at each expansion.  Returns {(tree, node): (call, row)} of the rows that expanded nodes."""
    which = list(trees)
    assert which == rec.which.tolist()
    raw_at = {}
    for s in (range(len(rec.log)) if calls is None else calls):
        c = rec.log[s]
        k = c["k"]
        for p, i in enumerate(which):
            T = trees[i]
            if gumbel:
                slots = T.select_gumbel(k, C_PUCT, FPU, rec.vl)
            elif k == 1:
                j = T.select(C_PUCT, FPU)
                slots = [(j, T.status[j])]
            else:
                slots = T.select_leaves(k, C_PUCT, FPU, rec.vl)
            for kk, (j, st) in enumerate(slots):
                r = p * k + kk
                assert c["leaves"][r].tobytes() == T.rec[j].tobytes(), (s, i, kk, j)
                got = {f: int(c[f][r]) for f in FIELDS}
                assert got == {"status": st, "winner": T.winner[j], "reward": T.reward[j], "depth": T.depth[j]}, (s, i, kk, j)
                if st == 0:
                    raw_at[(i, j)] = (s, r)
            SL.LeavesTree.expand_backup_slots(T, slots, lambda j: dev[i][1][j]["prior"], c["values"][p * k:(p + 1) * k])
    return raw_at


def check_trees(trees, dev, rec, raw_at):
    """every node and edge field of get_tree bit for bit; the priors of the nodes expanded in the recorded calls against float64"""
    n_nodes = 0
    for i, T in trees.items():
        assert_tree_equal(dev[i], T, i)
        n_nodes += len(T.rec)
    for (i, j), (s, r) in raw_at.items():
        T = trees[i]
        c = len(T.act[j])
        if c == 0:
            continue
        row = rec.log[s]["scores"][r] if s != "begin" else rec.begin_rows["scores"][r]
        if rec.compact:
            raw = row[:c]
        else:
            flip = rec.view == 1 and T.rec[j]["player"] == 1
            raw = row[np.where(flip, 8099 - T.act[j], T.act[j])]
        want = S.priors64(raw, TEMP)
        l = P.clean(raw)
        with np.errstate(invalid="ignore"):
            arg = np.where(np.isfinite(l) & np.isfinite(l.max()), np.abs(l - l.max()) / TEMP, 0.0)
        tol = 1e-6 + 2.0 ** -23 * arg                       # as test_search_gpu._replay: 1e-6 plus the f32 rounding of (l - m) / T
        got = dev[i][1][j]["prior"][:c].astype(np.float64)
        big = want > 1e-30
        assert (np.abs(got - want)[big] <= tol[big] * want[big]).all() and (got[~big] < 1e-30).all(), (i, j)
    return n_nodes


def check_root(torch, ts, trees, view):
    """root(): visits, q and best of the sampled trees against the oracle"""
    w = torch.tensor(list(trees), device="cuda")
    vis, q, best = (x[w].cpu().numpy() for x in ts.root(_vname(view)))
    for p, (i, T) in enumerate(trees.items()):
        wv, wq, wb = T.root(view)
        assert np.array_equal(vis[p], wv) and int(best[p]) == wb, i
        assert (np.isnan(q[p]) and np.isnan(wq)) or q[p].view(np.uint32) == wq.view(np.uint32), i


def statuses(rec):
    return set(np.concatenate([c["status"] for c in rec.log]).tolist())


def puct_search(xq, torch, O, L, specials, n, max_sims, plan, view, sdt, seed, max_leaves=1, compact=False, peak=None, total=48,
                mid=None, handles=None):
    """a search of n trees on seeded device inputs, recorded on the sampled trees and replayed by the oracle: (te, ts, rec, trees, dev,
    boundary report, boards).  mid = (k, on_device(te, ts, which), on_oracle(trees)): called after the first k calls of the plan, on the
    device and on the oracle trees.  The handles are appended to `handles` as they are made."""
    cap = max_sims + 1
    which, bnd, rest = sample_trees(n, cap, seed, total)
    recs = boards(O, n, seed, rest, specials)
    te = xq.TorchEnv(n, seed=ENV_SEED)
    handles.append(te)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, max_sims, max_leaves)
    handles.append(ts)
    ts.reset()
    rec = Recorder(torch, ts, which, seed, view=view, sdt=sdt, compact=compact, peak=peak)
    k = len(plan) if mid is None else mid[0]
    rec.run(plan[:k])
    if mid is not None:
        mid[1](te, ts, which)
        rec.run(plan[k:])
    dev = {i: ts.search.get_tree(i) for i in which}
    lines = check_boundaries(bnd, dev, cap)
    trees = {i: SL.LeavesTree(L, recs[i]) for i in which}
    raw_at = replay(L, trees, rec, dev, calls=range(k))
    if mid is not None:
        mid[2](trees)
        raw_at.update(replay(L, trees, rec, dev, calls=range(k, len(plan))))
    check_trees(trees, dev, rec, raw_at)
    check_root(torch, ts, trees, view)
    assert {0, 1, 2, 3}.issubset(statuses(rec))         # captures, move caps and boards without a legal action were reached
    return te, ts, rec, trees, dev, lines, recs


def _plan(n_sims, L):
    """the selection sizes of TorchSearch.run(leaves=L): one leaf first (it expands the roots), then L-leaf calls, the last one smaller"""
    out = [1]
    while sum(out) < n_sims:
        out.append(min(L, n_sims - sum(out)))
    return out




# ---- the example ring fed from the searches ----------------------------------------------------------------------------------------------
RING, COPIES, RESULT = 1 << 21, 33, 0.25          # 65,536 envs x 33 examples = 2,162,688 commits: the 2^21-slot ring wraps


def example_of(dt, T, e, ply, z, weights=None):
    """the example record() (record_gumbel() with the Gumbel weights) stores from oracle tree T of env e at ply `ply`, committed with
    result z from Red's side in the env's first game"""
    x = np.zeros((), dt)
    x["rec"] = T.rec[0]
    x["env"], x["ply"], x["game"] = e, ply, 0
    ne = len(T.act[0]) if T.expanded[0] else 0
    N = T.N[0] if ne else np.zeros(0, np.int64)
    x["n_edges"] = ne
    x["action"][:] = -1
    x["action"][:ne] = T.act[0][:ne] if ne else []
    x["visits"][:ne] = N if weights is None else weights
    x["total_visits"] = int(x["visits"].sum())
    sw = F32(0)
    for w in (T.W[0] if ne else []):
        sw = F32(sw + w)
    sn = int(N.sum())
    x["q"] = F32(sw / F32(sn)) if sn else F32(np.nan)
    x["z"] = F32(z) if T.rec[0]["player"] == 0 else -F32(z)
    return x


def fill_ring(xq, torch, te, runner, gumbel, handles):
    """a 2^21-slot ring holding COPIES examples of every root of `runner`, all committed at once (it wraps): the buffer"""
    tx = xq.TorchExamples(te, RING, COPIES)
    handles.append(tx)
    for _ in range(COPIES):
        tx.record_gumbel(runner) if gumbel else tx.record(runner)
    tx.end_games(torch.ones(te.n, dtype=torch.bool, device="cuda"), torch.full((te.n,), RESULT, device="cuda"))
    info = tx.info()
    assert info["total_committed"] == te.n * COPIES > RING and info["size"] == RING and info["stale"] == 0
    return tx


def ring_slots(n, e):
    """{slot: ply} of env e's examples still in the ring: commit number e * COPIES + ply, the last RING commits survive"""
    total = n * COPIES
    return {(e * COPIES + c) % RING: c for c in range(COPIES) if e * COPIES + c >= total - RING}


def same_example(a, b, tag, weights=False):
    """a == b bit for bit (q: both NaN or the same bits); weights: the Gumbel weights round(pi' 2^24) may differ by one unit, since the
    oracle's pi' is within rtol 4e-6 of the device's, not bit for bit; total_visits is then the sum of a's weights"""
    fa, fb = a.copy(), b.copy()
    qa, qb = F32(fa["q"]), F32(fb["q"])
    assert (np.isnan(qa) and np.isnan(qb)) or qa.view(np.uint32) == qb.view(np.uint32), tag
    fa["q"] = fb["q"] = 0
    if weights:
        va, vb = fa["visits"].astype(np.int64), fb["visits"].astype(np.int64)
        assert (np.abs(va - vb) <= 1).all() and int(fa["total_visits"]) == int(va.sum()), tag
        fa["visits"] = fb["visits"] = 0
        fa["total_visits"] = fb["total_visits"] = 0
    assert fa.tobytes() == fb.tobytes(), tag


def check_ring(xq, torch, tx, want, view, weights=False):
    """want {slot: example}: the ring's slots bit for bit (same_example), then sample / sample_compact rows that land on them against
    the slots, and load"""
    for s, x in list(want.items()):
        got = tx.get(s, 1)[0]
        same_example(got, x, s, weights)
        want[s] = got
    batch, seed, counter = 65536, 7, 3
    sm = tx.sample(batch, seed, counter, view=_vname(view))
    sc = tx.sample(batch, seed, counter, view=_vname(view), compact=True)
    idx = sm.index.cpu().numpy()
    draw = (_draw(seed, batch, counter) % np.uint64(RING)).astype(np.int64)
    assert (idx == draw).all() and (sc.index.cpu().numpy() == idx).all()
    hits = np.nonzero(np.isin(idx, list(want)))[0]
    assert len(hits) >= 10, len(hits)
    h = torch.from_numpy(hits).cuda()
    pol, val, q = (t[h].cpu().numpy() for t in (sm.policy, sm.value, sm.q))
    ca, cp, cc = (t[h].cpu().numpy() for t in (sc.actions, sc.policy, sc.counts))
    xs = np.array([want[int(idx[r])] for r in hits], xq.EXAMPLE_DTYPE)
    wpol, _ = targets_numpy(xs, np.arange(len(xs)), view)
    for k, x in enumerate(xs):
        ne, tot = int(x["n_edges"]), int(x["total_visits"])
        assert pol[k].tobytes() == wpol[k].tobytes() and F32(val[k]) == F32(x["z"]), k
        assert (np.isnan(q[k]) and np.isnan(x["q"])) or F32(q[k]).view(np.uint32) == F32(x["q"]).view(np.uint32), k
        a = x["action"][:ne].astype(np.int64)
        if view == 1 and x["rec"]["player"] == 1:
            a = 8099 - a
        assert int(cc[k]) == ne and (ca[k, :ne] == a).all() and (ca[k, ne:] == -1).all(), k
        wp = x["visits"][:ne].astype(F32) / F32(tot) if tot else np.zeros(ne, F32)
        assert cp[k, :ne].tobytes() == wp.tobytes() and (cp[k, ne:] == 0).all(), k
    slots = np.array(sorted(want), np.int64)
    te2 = xq.TorchEnv(len(slots))
    tx.load(te2, torch.from_numpy(slots).cuda())
    got = te2.env.get_boards()
    te2.close()
    for r, s in enumerate(slots):
        assert got[r].tobytes() == want[s]["rec"].tobytes(), s
    return len(hits)


def expected_ring(xq, trees, n, weights=None):
    """{slot: example} of the sampled trees' surviving examples, and how many of them sit in slots the ring wrapped onto"""
    want, wrapped = {}, 0
    for i, T in trees.items():
        for s, c in ring_slots(n, int(i)).items():
            want[s] = example_of(xq.EXAMPLE_DTYPE, T, int(i), c, RESULT, None if weights is None else weights[i])
            wrapped += int(i) * COPIES + c >= RING
    return want, wrapped


# ---- (a) + (f) + (h): the benchmarked configuration, the example ring, then play, advance and 50 more simulations ------------------------
def test_puct_65536_trees_200_simulations_play_advance(xq, torch, O, oracle_lib, specials, handles):
    """PUCT, one leaf, 65,536 trees x 200 simulations (31.5 GB slab), dense bf16 scores, side view.  After 120 simulations every root
    is recorded 33 times into a 2^21-slot example ring that wraps; its slots, sample / sample_compact rows and load are checked against
    examples built from the oracle trees at that point, and after the 200th simulation refresh() against the oracle's final roots.
    Then play with temperature 1 and a sample_plies schedule (roots at move_count 7 are sampled, the rest greedy), advance(min_free = 50)
    and 50 more simulations."""
    L = oracle_lib
    n, max_sims, view, min_free, mid_k = 65536, 200, 1, 50, 120
    slab = n * xq.search_bytes_per_tree(max_sims)
    need_memory(torch, slab + xq.examples_bytes(n, RING, COPIES) + input_bytes(n, 8100, 2) + 4 * GB, "65,536 trees x 200 simulations")
    t0, peak = time.time(), Peak(torch)
    box = {}

    def on_device(te, ts, which):
        box["tx"] = fill_ring(xq, torch, te, ts, False, handles)
        peak.sample()

    def on_oracle(trees):
        box["want"], box["wrapped"] = expected_ring(xq, trees, n)

    te, ts, rec, trees, dev, lines, recs = puct_search(xq, torch, O, L, specials, n, max_sims, [1] * max_sims, view, torch.bfloat16, 11,
                                                       peak=peak, mid=(mid_k, on_device, on_oracle), handles=handles)
    assert len(lines) == 3                              # 65,536 x 201 x 128 edge slots < 2^31: every boundary but element 2^31
    lines.append(f"slab {slab / GB:.1f} GB")
    report("PUCT 65,536 x 200, bf16, side", t0, peak, lines)
    # the ring recorded after 120 simulations
    t1 = time.time()
    tx, want = box["tx"], box["want"]
    assert box["wrapped"] >= COPIES                     # the last tree's examples lie in slots the ring wrapped onto
    hits = check_ring(xq, torch, tx, want, view)
    # refresh: each sampled tree rewrites its last surviving slot from its final root
    which = rec.which
    index = np.full(n, -1, np.int64)
    last = {}
    for i in which:
        sl = ring_slots(n, int(i))
        if sl:
            index[i] = last[i] = max(sl, key=sl.get)
    before = {s: tx.get(s, 1)[0] for s in last.values()}
    status = tx.refresh(ts, torch.from_numpy(index).cuda()).cpu().numpy()
    assert (status[index < 0] == 1).all()               # NO_SLOT
    refreshed = 0
    for i, s in last.items():
        x = example_of(xq.EXAMPLE_DTYPE, trees[i], int(i), 0, RESULT)
        got = tx.get(s, 1)[0]
        if x["total_visits"] == 0:
            assert status[i] == 4 and got.tobytes() == before[s].tobytes(), i          # UNSEARCHED: the slot is left alone
            continue
        assert status[i] == 0, (i, status[i])
        refreshed += 1
        for f in ("rec", "env", "game", "ply", "z"):
            assert got[f].tobytes() == before[s][f].tobytes(), (i, f)
        for f in ("rec", "env", "game", "ply", "z"):
            x[f] = got[f]
        same_example(got, x, ("refresh", i))
    assert refreshed >= 30
    report("example ring of 2^21 slots", t1, peak, [f"{len(want)} slots checked ({box['wrapped']} wrapped), {hits} sampled rows, "
                                                    f"{refreshed} refreshed"])
    # play: temperature 1 below sample_plies = 8, greedy from there
    t1 = time.time()
    ctr = te.env.get_boards()["ctr"]
    res = ts.play(temperature=1.0, sample_plies=8, view="side", auto_reset=True)
    acts, valid = res.actions[rec.w].cpu().numpy(), res.valid[rec.w].cpu().numpy()
    lib = xq.lib()
    kinds = set()
    for p, i in enumerate(which):
        T = trees[i]
        n0 = T.N[0] if T.expanded[0] and T.act[0] is not None and len(T.act[0]) else np.zeros(0, np.int64)
        if n0.sum() == 0:
            assert acts[p] == -1 and valid[p] == 0, i
            kinds.add("none")
            continue
        flip = view == 1 and T.rec[0]["player"] == 1
        if T.rec[0]["move_count"] < 8:
            u = F32(lib.xq_rng(ENV_SEED, int(i), int(ctr[i])) >> 40) * F32(2.0 ** -24)
            k = H.sample_numpy(n0.astype(np.int32), 1.0, u)[0]
            kinds.add("sampled")
        else:
            k = int(np.argmax(n0))
            kinds.add("greedy")
        assert acts[p] == (8099 - T.act[0][k] if flip else T.act[0][k]) and valid[p] == 1, i
    assert kinds == {"none", "sampled", "greedy"}, kinds
    envs = te.env.get_boards()
    kept = ts.advance(min_free, view="side").cpu().numpy()
    after = {}
    for i in which:
        after[i], k = advance_oracle(L, tree_from_device(L, *dev[i]), envs[i], min_free, max_sims + 1)
        assert kept[i] == k, i
        assert_tree_equal(ts.search.get_tree(int(i)), after[i], ("advance", i))
    assert (kept[which] > 1).sum() >= 10 and (kept[which] == 0).any(), kept[which]     # kept subtrees and rebuilt trees
    rec2 = Recorder(torch, ts, which, 12, view=view, sdt=torch.bfloat16, peak=peak)
    rec2.run([1] * min_free)
    with pytest.raises(xq.XQError):
        ts.select()
    dev2 = {i: ts.search.get_tree(int(i)) for i in which}
    raw_at = replay(L, after, rec2, dev2)
    check_trees(after, dev2, rec2, raw_at)
    check_root(torch, ts, after, view)
    report("play + advance(50) + 50 simulations", t1, peak, [f"kept subtrees on the sampled trees: {int((kept[which] > 1).sum())}"])


# ---- (b): past 2^31 edge elements ------------------------------------------------------------------------------------------------------
def test_puct_65536_trees_300_simulations_past_2_31_edges(xq, torch, O, oracle_lib, specials, handles):
    """PUCT, one leaf, 65,536 trees x 300 simulations (47 GB slab, 2.52e9 edge slots): element 2^31 is the edge block of node 78 of
    tree 55,738; dense f32 scores, absolute view"""
    n, max_sims = 65536, 300
    slab = n * xq.search_bytes_per_tree(max_sims)
    need_memory(torch, slab + input_bytes(n, 8100, 4) + 4 * GB, "65,536 trees x 300 simulations")
    t0, peak = time.time(), Peak(torch)
    assert boundary_trees(n, max_sims + 1)[-1][2:] == (55738, 78)
    *_, lines, _ = puct_search(xq, torch, O, oracle_lib, specials, n, max_sims, [1] * max_sims, 0, None, 21, peak=peak, handles=handles)
    assert len(lines) == 4
    lines.append(f"slab {slab / GB:.1f} GB")
    report("PUCT 65,536 x 300, f32, absolute", t0, peak, lines)


# ---- (c) / (d): multi-leaf ---------------------------------------------------------------------------------------------------------------
def test_leaves_8_on_65539_trees(xq, torch, O, oracle_lib, specials, handles):
    """8 leaves per call, virtual loss 1, dense f32 scores, side view, 65,539 trees x 64 simulations: a partial last CTA in every kernel
    at the benchmark size"""
    n, max_sims, L = 65539, 64, 8
    slab = n * xq.search_bytes_per_tree(max_sims, L)
    need_memory(torch, slab + input_bytes(n * L, 8100, 4) + 4 * GB, "65,539 trees x 8 leaves")
    t0, peak = time.time(), Peak(torch)
    plan = _plan(max_sims, L)
    _, _, rec, trees, _, lines, _ = puct_search(xq, torch, O, oracle_lib, specials, n, max_sims, plan, 1, None, 31, max_leaves=L, peak=peak,
                                                handles=handles)
    assert 4 in statuses(rec) and n - 1 in trees
    report("8 leaves, 65,539 x 64, f32, side", t0, peak, lines)


def test_leaves_32_compact_deep(xq, torch, O, oracle_lib, specials, handles):
    """32 leaves per call, compact f32 rows, 65,536 trees x 96 simulations: one leaf, then three 32-leaf calls (31 in the last)"""
    n, max_sims, L = 65536, 96, 32
    slab = n * xq.search_bytes_per_tree(max_sims, L)
    need_memory(torch, slab + input_bytes(n * L, 128, 4) + 4 * GB, "65,536 trees x 32 compact leaves")
    t0, peak = time.time(), Peak(torch)
    plan = _plan(max_sims, L)
    assert plan == [1, 32, 32, 31]
    _, _, rec, trees, dev, lines, _ = puct_search(xq, torch, O, oracle_lib, specials, n, max_sims, plan, 0, None, 41, max_leaves=L,
                                                  compact=True, peak=peak, handles=handles)
    assert 4 in statuses(rec)
    assert max(int(dev[i][0]["depth"].max()) for i in trees) >= 3
    report("32 compact leaves, 65,536 x 96", t0, peak, lines)


# ---- (e) + (h): Gumbel, the improved policy against float64, the Gumbel weights in the example ring --------------------------------------
def fp64_roots(ts, tg, pol, trees, view, c_visit=50.0, c_scale=0.1):
    """every listed root's improved policy (pol: the device's dense rows of those trees, in order) against improved_policy64 and its
    bound: the worst |pi_f32 - pi_64| / bound, and per root (n_edges, span of the completed q, span of the finite logits)"""
    worst, seen = 0.0, []
    for p, i in enumerate(trees):
        nodes, edges = ts.search.get_tree(int(i))
        st = tg.gumbel.get(int(i))
        if st["m"] == 0:
            assert not pol[p].any(), i
            continue
        ne = int(nodes[0]["n_edges"])
        e = edges[0][:ne]
        pi, bnd = G.improved_policy64(e["visits"], e["value_sum"], e["prior"], st["logit"][:ne], st["root_value"], c_visit, c_scale)
        a = e["action"].astype(np.int64)
        got = pol[p][np.where(view == 1 and nodes[0]["rec"]["player"] == 1, 8099 - a, a)].astype(np.float64)
        err = np.abs(got - pi)
        assert (err <= bnd).all(), (i, float((err / np.maximum(bnd, 1e-300)).max()))
        live = bnd > 0
        if live.any():
            worst = max(worst, float((err[live] / bnd[live]).max()))
        q, _ = G.completed_q(e["visits"], e["value_sum"], e["prior"], st["root_value"])
        lg = st["logit"][:ne][np.isfinite(st["logit"][:ne])]
        seen.append((ne, float(q.max()) - float(q.min()), float(lg.max() - lg.min()) if len(lg) else 0.0))
    return worst, seen


def test_gumbel_65536_trees(xq, torch, O, oracle_lib, specials, handles):
    """Gumbel root search, max_considered 16, 8 leaves per call, 65,536 trees x 64 simulations, bf16 scores, side view: the begin state,
    every selection and the trees bit for bit, the action exactly, the improved policy as test_gumbel_gpu checks it and, at every root,
    within the float64 bound of gumbel_oracle.improved_policy64; then every root is recorded 33 times with record_gumbel into a wrapping
    2^21-slot ring, checked against the oracle's Gumbel weights"""
    L = oracle_lib
    n, max_sims, leaves, m, view, seed = 65536, 64, 8, 16, 1, 51
    slab = n * xq.search_bytes_per_tree(max_sims, leaves)
    need_memory(torch, slab + input_bytes(n * leaves, 8100, 2) + n * 8100 * 4 + 4 * GB, "Gumbel 65,536 trees x 8 leaves")
    t0, peak = time.time(), Peak(torch)
    which, bnd, rest = sample_trees(n, max_sims + 1, seed)
    recs = boards(O, n, seed, rest, specials)
    te = xq.TorchEnv(n, seed=ENV_SEED)
    handles.append(te)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, max_sims, leaves)
    handles.append(ts)
    tg = xq.TorchGumbel(ts, m)
    handles.append(tg)
    ts.reset()
    rec = Recorder(torch, ts, which, seed, view=view, sdt=torch.bfloat16, tg=tg, peak=peak)
    rec.begin(max_sims, seed)
    plan = [leaves] * (max_sims // leaves)
    rec.run(plan)
    dev = {i: ts.search.get_tree(int(i)) for i in which}
    lines = check_boundaries(bnd, dev, max_sims + 1)
    trees = {}
    for p, i in enumerate(which):
        Tr = G.GumbelTree(L, recs[i])
        if Tr.status[0] == 0:          # begin expands and backs up the root
            Tr.expand(0, dev[i][1][0]["prior"])
            Tr.backup(0, rec.begin_rows["values"][p])
        Tr.begin(check_state(recs, tg, dev[i], int(i), m, rec.v0, seed), max_sims, 50.0, 0.1)
        trees[i] = Tr
    raw_at = replay(L, trees, rec, dev, gumbel=True)
    raw_at.update({(i, 0): ("begin", p) for p, i in enumerate(which) if trees[i].expanded[0]})
    check_trees(trees, dev, rec, raw_at)
    pol_all, act = tg.root(_vname(view))
    peak.sample()
    pol, act = pol_all[rec.w].cpu().numpy(), act[rec.w].cpu().numpy()
    live, weights = 0, {}
    for p, (i, Tr) in enumerate(trees.items()):
        wp, wa, _ = Tr.gumbel_root(view)
        assert int(act[p]) == wa, i
        assert np.allclose(pol[p], wp, rtol=4e-6, atol=1e-12), i
        if Tr.gs["m"]:
            live += 1
            assert abs(float(pol[p].astype(np.float64).sum()) - 1.0) < 1e-5, i
            z, _, _, _ = Tr.root_stats()
            weights[i] = G.improved_policy(z)[1]
        else:
            weights[i] = np.zeros(len(Tr.act[0]) if Tr.expanded[0] else 0, np.int64)
    assert live >= 30
    # every root against float64
    t1 = time.time()
    pol_host = pol_all.cpu().numpy()
    del pol_all
    worst, seen = fp64_roots(ts, tg, pol_host, range(n), view)
    del pol_host
    lines.append(f"improved policy of all {len(seen)} roots with an edge within the float64 bound: worst error / bound {worst:.3g} "
                 f"({time.time() - t1:.0f} s)")
    # the Gumbel weights in the example ring
    tx = fill_ring(xq, torch, te, tg, True, handles)
    peak.sample()
    want, wrapped = expected_ring(xq, trees, n, weights)
    assert wrapped >= COPIES
    hits = check_ring(xq, torch, tx, want, view, weights=True)
    lines.append(f"example ring: {len(want)} slots checked ({wrapped} wrapped), {hits} sampled rows")
    report("Gumbel m = 16, 8 leaves, 65,536 x 64, bf16", t0, peak, lines)


def _one_and_most_edges(O, L):
    """boards with exactly one legal action, and the boards with the most legal actions among 20,000 arbitrary ones"""
    b = random_boards(O, 20000, seed=71)
    b = b[[not S.generals_missing(r) for r in b]]
    counts, _ = P.oracle_lists(L, b)
    one = b[counts == 1][:8]
    most = b[np.argsort(-counts.astype(np.int64), kind="stable")[:8]]
    return one, most, int(counts.max())


def test_gumbel_improved_policy_fp64_edges(xq, torch, O, oracle_lib, handles):
    """the improved policy against float64 at its edges, 8 trees each: a single edge; the most edges the rules give (the list holds
    up to 128; no board of 20,000 arbitrary ones has more than about 100 legal actions); every completed q equal (every leaf value 0.5
    and root value -0.5, every visited root edge visited once); max q - min q below, at and just above the 1e-8 floor; root scores spread by
    1e3 (logits from -inf to the f32 range); ordinary roots.  max_considered 128, 16 simulations of one leaf."""
    L = oracle_lib
    t0, peak = time.time(), Peak(torch)
    one, most, maxc = _one_and_most_edges(O, L)
    reach = harvest_positions(O, 32, 1, 8, seed=72)
    recs = np.concatenate([one, most, reach])
    n, sims, m, view = len(recs), 16, 128, 1
    assert n == 48 and len(one) == 8
    group = np.repeat(np.arange(6), 8)          # 0 one edge, 1 most edges, 2 equal q, 3 floor, 4 logits spread 1e3, 5 ordinary
    floor = F32(1e-8)
    spans = np.array([5e-9, floor, 1.0000001e-8, 2e-8] * 2, F32)
    te = xq.TorchEnv(n, seed=ENV_SEED)
    handles.append(te)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, sims)
    handles.append(ts)
    tg = xq.TorchGumbel(ts, m)
    handles.append(tg)
    rng = np.random.default_rng(73)

    def scores():
        x = (rng.standard_normal((n, 8100)) * 1.5).astype(F32)
        x[group == 4] = rng.uniform(-1e3, 0.0, (8, 8100)).astype(F32)
        return torch.from_numpy(x).cuda()

    def values(root):
        v = rng.uniform(-1.0, 1.0, n).astype(F32)
        v[group == 2] = F32(-0.5) if root else F32(0.5)         # q = -0.5 on every visited edge, and v_mix is -0.5 exactly
        v[group == 3] = F32(0.0) if root else rng.integers(0, 2, 8) * spans       # q is 0 or -span
        return torch.from_numpy(v).cuda()

    ts.reset()
    tg.begin(scores(), values(True), sims, seed=5, temperature=TEMP, view=_vname(view))
    for _ in range(sims):
        tg.select(1, C_PUCT, FPU, VL)
        ts.expand_backup(scores(), values(False), temperature=TEMP, view=_vname(view))
    pol = tg.root(_vname(view)).policy.cpu().numpy()
    worst, seen = fp64_roots(ts, tg, pol, range(n), view)
    assert len(seen) == n
    ne, span, lspan = (np.array(x) for x in zip(*seen))
    assert (ne[group == 0] == 1).all() and ne[group == 1].max() == maxc >= 90
    assert (span[group == 2] == 0).all()
    f = span[group == 3]
    assert (f < floor).sum() == 2 and (f == floor).sum() == 2 and ((f > floor) & (f < 3e-8)).sum() == 4, f
    assert lspan[group == 4].max() > 50 and lspan[group == 5].max() < 50
    peak.sample()
    report("Gumbel improved policy against float64 at its edges", t0, peak,
           [f"worst error / bound {worst:.3g}; most edges {maxc}; floor spans {np.round(f / 1e-8, 3).tolist()} x 1e-8"])


# ---- (g): the advance kernel's opt-in shared memory --------------------------------------------------------------------------------------
def test_advance_at_65536_simulations(xq, torch, O, oracle_lib, handles):
    """5 trees of max_simulations 65,536 (the advance kernel's bitmap takes 4 x 8 x 2,049 bytes, above 48 KB: the opt-in shared-memory
    path) filled by 32-leaf compact calls until a tree holds more than 49,152 nodes (membership words above 1,536); after a move every
    tree is compared with the advance oracle on its get_tree"""
    L = oracle_lib
    n, max_sims, leaves = 5, xq.SEARCH_ADVANCE_MAX_SIMULATIONS, 32
    need_memory(torch, n * xq.search_bytes_per_tree(max_sims, leaves) + 2 * GB, "5 trees x 65,536 simulations")
    t0, peak = time.time(), Peak(torch)
    recs = harvest_positions(O, n, 1, 6, seed=61)
    te = xq.TorchEnv(n, seed=ENV_SEED)
    handles.append(te)
    te.env.set_boards(recs)
    ts = xq.TorchSearch(te, max_sims, leaves)
    handles.append(ts)
    ts.reset()
    g = torch.Generator(device="cuda").manual_seed(61)
    used = 0
    while used < max_sims:
        k = min(leaves, max_sims - used)
        ts.select_leaves(k, C_PUCT, FPU, 3.0)
        sc = torch.randn((n * k, 128), generator=g, device="cuda")
        v = torch.rand(n * k, generator=g, device="cuda").mul_(2).sub_(1)
        ts.expand_backup_compact(sc, v, temperature=TEMP)
        used += k
    peak.sample()
    pre = {i: tree_from_device(L, *ts.search.get_tree(i)) for i in range(n)}
    sizes = [len(T.rec) for T in pre.values()]
    assert max(sizes) > 49152, sizes
    te.step(actions=ts.root("side").best, pick="given", view="side", auto_reset=False)
    envs = te.env.get_boards()
    kept = ts.advance(1).cpu().numpy()
    deep = 0
    for i in range(n):
        want, k = advance_oracle(L, pre[i], envs[i], 1, max_sims + 1)
        assert kept[i] == k, (i, kept[i], k)
        assert_tree_equal(ts.search.get_tree(i), want, ("advance", i))
        if k > 1 and sizes[i] > 49152:
            deep += 1
    assert deep >= 1, (sizes, kept)
    report("advance at 65,536 simulations", t0, peak, [f"tree sizes {sizes}, kept {kept.tolist()}"])
