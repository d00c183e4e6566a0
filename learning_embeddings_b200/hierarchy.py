"""Hierarchies the hot path is exercised on: the 723-node ETHEC label tree and synthetic random trees.

The ETHEC parent array in data/ethec_hierarchy.npz was extracted from the reference's hard-coded
taxonomy (data/db.py:3480-3510, ETHECLabelMapMerged) by tests/golden/make_golden.py; it is data, not
code.  Closure / non-edge queries use Euler-tour intervals, so nothing here needs the reference's dense
n x n adjacency (order_embeddings.py:417-423), which does not exist at 82 K nodes (SURVEY F7).
"""
import os

import numpy as np

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


class Hierarchy:
    """Forest given by a parent array (-1 = root).  Node ids are level-major like the reference's."""

    def __init__(self, parents, levels=None):
        self.parents = np.asarray(parents, dtype=np.int64)
        self.n = len(self.parents)
        self.levels = None if levels is None else [int(v) for v in levels]
        if self.levels is not None:
            stops = np.cumsum(self.levels)
            self.level_start = [int(v) for v in stops - np.asarray(self.levels)]
            self.level_stop = [int(v) for v in stops]
        order = np.argsort(self.parents, kind="stable")
        self.children_ptr = np.searchsorted(self.parents[order], np.arange(-1, self.n + 1))
        self.children_idx = order
        # iterative Euler tour
        self.tin = np.zeros(self.n, dtype=np.int64)
        self.tout = np.zeros(self.n, dtype=np.int64)
        self.depth = np.zeros(self.n, dtype=np.int64)
        clock = 0
        roots = self._children(-1)
        stack = [(int(r), 0) for r in roots[::-1]]
        while stack:
            node, state = stack.pop()
            if state == 0:
                self.tin[node] = clock
                clock += 1
                stack.append((node, 1))
                for c in self._children(node)[::-1]:
                    self.depth[c] = self.depth[node] + 1
                    stack.append((int(c), 0))
            else:
                self.tout[node] = clock - 1

    @classmethod
    def from_closure_edges(cls, n, edges):
        """The forest whose transitive closure is `edges`, (ancestor, descendant) pairs -- the reference's G_tc edge
        list (order_embeddings.py:371).  A node's parent is its ancestor with the most ancestors.  Raises ValueError
        when the edges are not the closure of a forest on n nodes (a diamond, a cycle, a missing transitive edge)."""
        e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
        if len(e) and (e.min() < 0 or e.max() >= n):
            raise ValueError("closure edge endpoint outside [0, %d)" % n)
        if np.any(e[:, 0] == e[:, 1]):
            raise ValueError("closure edge from a node to itself")
        if len(e) == 0:
            return cls(np.full(n, -1, dtype=np.int64))
        e = np.unique(e, axis=0)
        n_anc = np.bincount(e[:, 1], minlength=n)
        o = np.lexsort((n_anc[e[:, 0]], e[:, 1]))          # per descendant, ancestors by their own ancestor count
        u, v = e[o, 0], e[o, 1]
        last = np.r_[v[1:] != v[:-1], True]
        parents = np.full(n, -1, dtype=np.int64)
        parents[v[last]] = u[last]
        has = parents >= 0
        # in a forest the parent has exactly one ancestor fewer; this also rules out cycles
        if np.any(n_anc[parents[has]] != n_anc[has] - 1):
            raise ValueError("the edges are not the transitive closure of a forest")
        h = cls(parents)
        if not np.array_equal(h.closure_edges(), e):
            raise ValueError("the edges are not the transitive closure of a forest")
        return h

    def _children(self, node):
        lo, hi = self.children_ptr[node + 1], self.children_ptr[node + 2]
        return self.children_idx[lo:hi]

    def is_descendant(self, u, v):
        """v is a strict descendant of u (vectorised)."""
        return (self.tin[v] > self.tin[u]) & (self.tin[v] <= self.tout[u])

    def closure_edges(self):
        """All (ancestor, descendant) pairs = edges of the transitive closure (order_embeddings.py:371)."""
        us, vs = [], []
        cur = np.arange(self.n)
        anc = self.parents.copy()
        while True:
            m = anc >= 0
            if not m.any():
                break
            us.append(anc[m])
            vs.append(cur[m])
            nxt = np.full(self.n, -1, dtype=np.int64)
            nxt[m] = self.parents[anc[m]]
            anc = nxt
        u, v = np.concatenate(us), np.concatenate(vs)
        o = np.lexsort((v, u))
        return np.stack([u[o], v[o]], axis=1)

    def negative_adjacency(self):
        """Dense bool matrix of the reference (ones - closure - diagonal); only sensible for small n."""
        A = np.ones((self.n, self.n), dtype=bool)
        e = self.closure_edges()
        A[e[:, 0], e[:, 1]] = False
        np.fill_diagonal(A, False)
        return A

    def sample_negatives(self, u, v, n_neg, rng):
        """Uniform draws from the reference's candidate sets, vectorised (rejection on Euler intervals).

        neg_to[i, p]   uniform over {x : x != u_i, x not a descendant of u_i}   (corrupt the child)
        neg_from[i, p] uniform over {x : x != v_i, x not an ancestor of v_i}    (corrupt the parent)
        Same distribution as random.choice(np.where(negative_G[u])) but NOT the same stream: used for
        synthetic benchmark batches; the bit-exact sampler is criterion.sample_negative_edge."""
        u = np.asarray(u)
        v = np.asarray(v)
        B = len(u)
        uu = np.repeat(u[:, None], n_neg, 1)
        vv = np.repeat(v[:, None], n_neg, 1)
        # a node whose subtree is everything else has no "corrupted child" candidate: the reference's
        # random.choice raises IndexError on the empty list (order_embeddings.py:1007)
        if len(u) and int((self.tout[u] - self.tin[u]).max()) >= self.n - 1:
            raise IndexError("a positive's parent is an ancestor of every other node: no negative candidate")
        neg_to = rng.integers(0, self.n, size=(B, n_neg))
        neg_from = rng.integers(0, self.n, size=(B, n_neg))
        while True:
            bad = (neg_to == uu) | self.is_descendant(uu, neg_to)
            k = int(bad.sum())
            if k == 0:
                break
            neg_to[bad] = rng.integers(0, self.n, size=k)
        while True:
            bad = (neg_from == vv) | self.is_descendant(neg_from, vv)
            k = int(bad.sum())
            if k == 0:
                break
            neg_from[bad] = rng.integers(0, self.n, size=k)
        return neg_to, neg_from


def ethec():
    with np.load(os.path.join(_DATA, "ethec_hierarchy.npz")) as z:
        return Hierarchy(z["parents"], z["levels"])


def random_tree(n, gamma, seed=0, roots=8):
    """SURVEY 8(d) cfg4: parent(i) = floor(i * r**gamma), r ~ U[0,1); nodes 0..roots-1 are roots.  A forest,
    not a single tree: under a single root the reference's candidate list for "corrupt the child of the
    root" is empty (order_embeddings.py:993, random.choice raises IndexError), so such a graph cannot be
    trained by the reference either.  random_tree(82115, 1.0831) has 741 845 closure edges (SURVEY target 743 K +- 1 %)."""
    rng = np.random.default_rng(seed)
    r = rng.random(n)
    parents = np.floor(np.arange(n) * r ** gamma).astype(np.int64)
    parents[1:] = np.minimum(parents[1:], np.arange(1, n) - 1)
    parents[:roots] = -1
    return Hierarchy(parents)
