"""numpy restatement of the multi-leaf selection (include/xq.h: xq_search_select_leaves_device) on search_oracle.Tree: L descents per
call in order, the virtual-loss score with the in-flight counts of the earlier descents, duplicate slots, and the expansion + backup
in slot order.  Every score is spelled out in np.float32 in the stated operation order, so that it matches the device bit for bit."""
import numpy as np

import search_oracle as S

F32 = np.float32
DUPLICATE = 4


def puct_vl(p, n, w, c, vl, c_puct, fpu, n_node, c_node):
    """Q + U per edge with virtual loss: N' = N + c, W' = c > 0 ? W - vl * c : W, Q = N' > 0 ? W' / N' : fpu,
    U = ((c_puct * P) * sqrt(N_node + c_node)) / (1 + N'), every operation rounded to f32"""
    p, w = np.asarray(p, F32), np.asarray(w, F32)
    c = np.asarray(c, np.int64)
    nv = np.asarray(n, np.int64) + c
    wv = np.where(c > 0, (w + -(F32(vl) * c.astype(F32))).astype(F32), w).astype(F32)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(nv > 0, wv / nv.astype(F32), F32(fpu)).astype(F32)
    sq = np.sqrt(F32(int(n_node) + int(c_node)))
    u = ((F32(c_puct) * p) * sq) / (1 + nv).astype(F32)
    return (q + u).astype(F32)


def inflight_counts(paths, node_path):
    """the definition of the in-flight counts at a node: paths = the node lists (root first) of the earlier descents, node_path = the
    node list from the root to the node.  {edge child node: count}; a path went through edge (j -> c) if it contains j followed by c"""
    d = len(node_path) - 1
    out = {}
    for p in paths:
        if len(p) > d + 1 and list(p[:d + 1]) == list(node_path):
            out[p[d + 1]] = out.get(p[d + 1], 0) + 1
    return out


class LeavesTree(S.Tree):
    """a search_oracle.Tree with the multi-leaf selection"""

    def select_leaves(self, L, c_puct, fpu, vl):
        """the L descents of one call: [(leaf node, status)], status 4 for a duplicate"""
        inflight = {}                     # (node, edge) -> descents of this call through it
        ended = set()
        out = []
        for _ in range(L):
            j, path = 0, []
            while self.expanded[j] and not self.status[j]:
                ne = len(self.act[j])
                c = np.array([inflight.get((j, e), 0) for e in range(ne)], np.int64)
                k = int(np.argmax(puct_vl(self.P[j], self.N[j], self.W[j], c, vl, c_puct, fpu, self.visits[j], int(c.sum()))))
                path.append((j, k))
                if self.child[j][k] >= 0:
                    j = int(self.child[j][k])
                    continue
                j = self._make_child(j, k)
                break
            for key in path:
                inflight[key] = inflight.get(key, 0) + 1
            dup = not self.expanded[j] and self.status[j] == 0 and j in ended
            ended.add(j)
            out.append((j, DUPLICATE if dup else self.status[j]))
        return out

    def expand_backup_slots(self, slots, priors_of, values):
        """expand every status-0 slot (priors_of(node) -> priors), then back up every slot but duplicates in slot order"""
        for j, st in slots:
            if st == 0:
                self.expand(j, priors_of(j))
        for (j, st), v in zip(slots, values):
            if st != DUPLICATE:
                self.backup(j, v)
