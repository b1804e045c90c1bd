"""numpy restatement of the batched tree search (include/xq.h: xq_search_*), shared by test_search_cpu.py and test_search_gpu.py.

Lists come from the oracle (xqo_batch_all_actions), child boards from xqo_batch_step.  PUCT, Q, the value cleaning and the backup are
spelled out in np.float32 in the stated operation order, so that they match the device bit for bit.  The replay takes each node's priors
from the device tree (xq_search_get_tree); priors64 checks those priors separately against a float64 softmax and the noise mix."""
import numpy as np

import policy_oracle as P

F32 = np.float32


def puct(p, n, w, c_puct, fpu, n_node):
    """Q + U per edge: Q = N > 0 ? W / N : fpu, U = ((c_puct * P) * sqrt(N_node)) / (1 + N), every operation rounded to f32"""
    p, w = np.asarray(p, F32), np.asarray(w, F32)
    n = np.asarray(n, np.int64)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(n > 0, w / n.astype(F32), F32(fpu)).astype(F32)
    sq = np.sqrt(F32(n_node))
    u = ((F32(c_puct) * p) * sq) / (1 + n).astype(F32)
    return (q + u).astype(F32)


def select_edge(p, n, w, c_puct, fpu, n_node):
    """the largest score, first in list order on ties (np.argmax returns the first maximum)"""
    return int(np.argmax(puct(p, n, w, c_puct, fpu, n_node)))


def clean_value(v):
    v = np.asarray(v, F32)
    return np.clip(np.where(np.isnan(v), F32(0), v), F32(-1), F32(1)).astype(F32)


def priors64(raw, t, noise=None, eps=0.0):
    """float64 priors of one node from its raw listed scores: softmax(clean / t), uniform when every score is -inf; noise mixed in"""
    l = P.clean(raw)
    n = len(l)
    if n == 0:
        return np.zeros(0)
    m = l.max()
    if m == -np.inf:
        p = np.full(n, 1.0 / n)
    else:
        with np.errstate(invalid="ignore", over="ignore"):
            e = np.where(np.isfinite(l), np.exp((l - m) / t), 0.0)
        p = e / e.sum()
    if noise is not None:
        p = (1.0 - eps) * p + eps * np.asarray(noise, np.float64)
    return p


def generals_missing(rec):
    sq = np.asarray(rec["sq"], np.uint32)
    codes = [(int(sq[s >> 3]) >> ((s & 7) * 4)) & 15 for s in range(90)]
    return 1 not in codes or 8 not in codes


class Tree:
    """one search tree as lists of node fields and per-node edge arrays (list order)"""

    def __init__(self, L, root):
        self.L = L
        self.rec = [root.copy()]
        self.parent, self.pedge, self.visits, self.reward, self.depth = [-1], [0], [0], [0], [0]
        r = root[None].copy()
        self.winner = [int(L.xqo_winner(r.ctypes.data))]
        self.status = [1 if generals_missing(root) else (2 if root["move_count"] >= 200 else 0)]
        self.expanded = [False]
        self.act, self.P, self.N, self.W, self.child = [None], [None], [None], [None], [None]

    def lists(self, j):
        c, a = P.oracle_lists(self.L, self.rec[j][None])
        a = a[0, :c[0]]
        return ((a >> 7).astype(np.int64) * 90 + (a & 127)).astype(np.int64)

    def select(self, c_puct, fpu):
        j = 0
        while self.expanded[j] and not self.status[j]:
            k = select_edge(self.P[j], self.N[j], self.W[j], c_puct, fpu, self.visits[j])
            if self.child[j][k] >= 0:
                j = int(self.child[j][k])
                continue
            return self._make_child(j, k)
        return j

    def _make_child(self, j, k):
        r = self.rec[j][None].copy()
        a = int(self.act[j][k])
        act = np.array([(a // 90) << 7 | (a % 90)], np.uint16)
        rew = np.zeros(1, np.int32)
        done, win, cap, valid = (np.zeros(1, np.uint8) for _ in range(4))
        self.L.xqo_batch_step(r.ctypes.data, 1, act, rew, done, win, cap, valid)
        assert valid[0] == 1
        nj = len(self.rec)
        self.rec.append(r[0])
        self.parent.append(j); self.pedge.append(k); self.visits.append(0); self.reward.append(int(rew[0]))
        self.depth.append(self.depth[j] + 1); self.winner.append(int(win[0]))
        self.status.append(1 if generals_missing(r[0]) else (2 if done[0] else 0))
        self.expanded.append(False)
        self.act.append(None); self.P.append(None); self.N.append(None); self.W.append(None); self.child.append(None)
        self.child[j][k] = nj
        return nj

    def expand(self, j, priors):
        acts = self.lists(j)
        self.act[j] = acts
        self.P[j] = np.asarray(priors, F32)[:len(acts)].copy()
        self.N[j] = np.zeros(len(acts), np.int64)
        self.W[j] = np.zeros(len(acts), F32)
        self.child[j] = np.full(len(acts), -1, np.int64)
        self.expanded[j] = True
        if len(acts) == 0:
            self.status[j] = 3

    def backup(self, j, value):
        v = clean_value(value)
        self.visits[j] += 1
        while j > 0:
            p = self.parent[j]
            v = F32(-v)
            e = self.pedge[j]
            self.N[p][e] += 1
            self.W[p][e] = F32(self.W[p][e] + v)
            self.visits[p] += 1
            j = p

    def root(self, view):
        """(visits [8100] in the frame of view, q, best)"""
        vis = np.zeros(8100, np.int32)
        flip = view == 1 and self.rec[0]["player"] == 1
        if not self.expanded[0] or len(self.act[0]) == 0:
            return vis, np.float32(np.nan), -1
        idx = np.where(flip, 8099 - self.act[0], self.act[0])
        vis[idx] = self.N[0]
        sw = F32(0)
        for x in self.W[0]:
            sw = F32(sw + x)
        sn = int(self.N[0].sum())
        q = F32(sw / F32(sn)) if sn > 0 else F32(np.nan)
        best = int(idx[int(np.argmax(self.N[0]))]) if sn > 0 else -1
        return vis, q, best

