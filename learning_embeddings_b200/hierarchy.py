"""Hierarchies the hot path is exercised on: the 723-node ETHEC label tree and synthetic random trees.

The ETHEC parent array in data/ethec_hierarchy.npz was extracted from the reference's hard-coded
taxonomy (data/db.py:3480-3510, ETHECLabelMapMerged) by tests/golden/make_golden.py; it is data, not
code.  Closure / non-edge queries use Euler-tour intervals (a forest) or an interval cover (DagHierarchy, a node with
several parents), so nothing here needs the reference's dense n x n adjacency (order_embeddings.py:417-423), which does
not exist at 82 K nodes (SURVEY F7).
"""
import os

import numpy as np

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


class _Closure:
    """Queries shared by Hierarchy and DagHierarchy, written in terms of is_descendant(u, v), closure_edges() and
    the per-node counts n_desc (strict descendants) and n_anc (strict ancestors)."""

    def _set_levels(self, levels):
        self.levels = None if levels is None else [int(v) for v in levels]
        if self.levels is not None:
            stops = np.cumsum(self.levels)
            self.level_start = [int(v) for v in stops - np.asarray(self.levels)]
            self.level_stop = [int(v) for v in stops]

    def rank_slots(self):
        """(pos_ptr, slot_of_edge) of the reconstruction ranks (metrics.reconstruction_ranks), computed once.  Apex u's
        positives own the slots [pos_ptr[u], pos_ptr[u+1]) (pos_ptr: int64 [n+1], the prefix of n_desc); v's slot
        under u is tin[v] - tin[u] - 1 inside u's primary interval, then u's extra intervals follow in order.
        slot_of_edge[i] (int64 [n_edges]) is the slot of closure_edges()[i]: a permutation of [0, n_edges)."""
        if getattr(self, "_rank_slots", None) is None:
            pos_ptr = np.r_[0, np.cumsum(np.asarray(self.n_desc, dtype=np.int64))].astype(np.int64)
            self._rank_xcum = None if getattr(self, "extra_lo", None) is None else np.zeros(0, dtype=np.int32)
            if pos_ptr[-1] == 0:   # no edge (Hierarchy.closure_edges needs one)
                self._rank_slots = (pos_ptr, np.zeros(0, dtype=np.int64))
                return self._rank_slots
            e = self.closure_edges()
            u, v = e[:, 0], e[:, 1]
            tin, tout = np.asarray(self.tin, dtype=np.int64), np.asarray(self.tout, dtype=np.int64)
            tv = tin[v]
            s = tv - tin[u] - 1
            lo = getattr(self, "extra_lo", None)
            if lo is not None and len(lo):
                lo = lo.astype(np.int64)
                size = self.extra_hi.astype(np.int64) - lo + 1
                first = self.extra_ptr[:-1].astype(np.int64)
                owner = np.repeat(np.arange(self.n), np.diff(self.extra_ptr))
                before = np.cumsum(size) - size                              # sizes of all earlier extra intervals
                xcum = (tout - tin)[owner] + before - before[first[owner]]   # slots of owner's cover before interval i
                out = ~((tv > tin[u]) & (tv <= tout[u]))
                i = np.searchsorted(self._extra_key, u[out] * self.n + tv[out], side="right") - 1
                s[out] = xcum[i] + tv[out] - lo[i]
                self._rank_xcum = xcum.astype(np.int32)
            self._rank_slots = (pos_ptr, pos_ptr[u] + s)
        return self._rank_slots

    def heldout_slots(self, edges):
        """(eval_ptr, slot_map, order, xcum) of link prediction on the held-out closure edges `edges` [m, 2]
        (metrics.link_prediction_ranks / link_prediction_f1): the held-out pairs keep rank_slots()' order, so apex u's own
        the held-out slots [eval_ptr[u], eval_ptr[u+1]) (eval_ptr: int64 [n+1]).  slot_map (int32 [n_closure]) is the
        held-out slot of each closure slot, -1 for a pair that is not held out; order (int64 [m]) the held-out slot of
        edges[i]; xcum (int32, one per extra interval) the closure slots of an apex before each of its extra intervals,
        None for a Hierarchy.  Raises ValueError for an endpoint outside [0, n), a pair that is not a closure edge or a
        repeated pair."""
        pos_ptr, slot_of_edge = self.rank_slots()
        e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
        if len(e) and (e.min() < 0 or e.max() >= self.n):
            raise ValueError("held-out edge endpoint outside [0, %d)" % self.n)
        keys = _edge_keys(e, self.n)
        if len(np.unique(keys)) != len(keys):
            raise ValueError("a held-out edge is given twice")
        ck = _edge_keys(self.closure_edges(), self.n) if len(slot_of_edge) else np.zeros(0, dtype=np.int64)
        if not np.all(_in_sorted(keys, ck)):
            raise ValueError("a held-out pair is not a closure edge")
        cslot = slot_of_edge[np.searchsorted(ck, keys)] if len(keys) else np.zeros(0, dtype=np.int64)
        held = np.zeros(len(slot_of_edge), dtype=bool)
        held[cslot] = True
        before = np.r_[0, np.cumsum(held)].astype(np.int64)   # held-out slots before each closure slot
        slot_map = np.where(held, before[:-1], -1).astype(np.int32)
        return before[pos_ptr], slot_map, before[cslot], self._rank_xcum

    def negative_adjacency(self):
        """Dense bool matrix of the reference (ones - closure - diagonal); only sensible for small n."""
        A = np.ones((self.n, self.n), dtype=bool)
        e = self.closure_edges()
        A[e[:, 0], e[:, 1]] = False
        np.fill_diagonal(A, False)
        return A

    def sample_negatives(self, u, v, n_neg, rng):
        """Uniform draws from the reference's candidate sets, vectorised (rejection on is_descendant).

        neg_to[i, p]   uniform over {x : x != u_i, x not a descendant of u_i}   (corrupt the child)
        neg_from[i, p] uniform over {x : x != v_i, x not an ancestor of v_i}    (corrupt the parent)
        Same distribution as random.choice(np.where(negative_G[u])) but NOT the same stream: used for
        synthetic benchmark batches; the bit-exact sampler is criterion.sample_negative_edge.
        Raises IndexError, before any draw, when a candidate set is empty: u_i above every other node, or v_i below
        every other node (a Hierarchy that is a chain, where the rejection loop could never end)."""
        u = np.asarray(u)
        v = np.asarray(v)
        B = len(u)
        uu = np.repeat(u[:, None], n_neg, 1)
        vv = np.repeat(v[:, None], n_neg, 1)
        # a node whose subtree is everything else has no "corrupted child" candidate: the reference's
        # random.choice raises IndexError on the empty list (order_embeddings.py:1007); likewise a child below
        # every other node has no "corrupted parent" candidate
        if len(u) and int(self.n_desc[u].max()) >= self.n - 1:
            raise IndexError("a positive's parent is an ancestor of every other node: no negative candidate")
        if len(v) and int(self.n_anc[v].max()) >= self.n - 1:
            raise IndexError("a positive's child is a descendant of every other node: no negative candidate")
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


class Hierarchy(_Closure):
    """Forest given by a parent array (-1 = root).  Node ids are level-major like the reference's."""

    def __init__(self, parents, levels=None):
        self.parents = np.asarray(parents, dtype=np.int64)
        self.n = len(self.parents)
        self._set_levels(levels)
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
        self.n_desc = self.tout - self.tin
        self.n_anc = self.depth

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


def _edge_keys(e, n):
    return e[:, 0] * n + e[:, 1]


def _compose(first, second, n):
    """Keys a * n + c of the pairs (a, c) with (a, b) in `first` and (b, c) in `second`, with repeats."""
    o = np.argsort(second[:, 0], kind="stable")
    src, dst = second[o, 0], second[o, 1]
    ptr = np.searchsorted(src, np.arange(n + 1))
    b = first[:, 1]
    cnt = ptr[b + 1] - ptr[b]
    total = int(cnt.sum())
    at = np.arange(total) - np.repeat(np.cumsum(cnt) - cnt, cnt) + np.repeat(ptr[b], cnt)
    return np.repeat(first[:, 0], cnt) * n + dst[at]


def _in_sorted(keys, sorted_keys):
    if len(sorted_keys) == 0:
        return np.zeros(len(keys), dtype=bool)
    i = np.minimum(np.searchsorted(sorted_keys, keys), len(sorted_keys) - 1)
    return sorted_keys[i] == keys


def _edge_array(n, edges, what):
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    if len(e) and (e.min() < 0 or e.max() >= n):
        raise ValueError("%s endpoint outside [0, %d)" % (what, n))
    if np.any(e[:, 0] == e[:, 1]):
        raise ValueError("%s from a node to itself" % what)
    k = np.unique(_edge_keys(e, n))
    return np.stack([k // n, k % n], axis=1), k


class DagHierarchy(_Closure):
    """Transitive closure of a DAG: a node may have several parents (the WordNet noun hierarchy is one).  Descendant
    queries use an interval cover instead of the dense n x n closure: the preorder numbers `tin` of a spanning
    forest, a primary interval [tin[u], tout[u]] of numbers that are all u or below u, and the maximal runs of u's
    other descendants' numbers as extra intervals [extra_lo[i], extra_hi[i]], i in [extra_ptr[u], extra_ptr[u+1]),
    sorted and disjoint.  The closure of a forest has Hierarchy's tin / tout and no extra interval."""

    def __init__(self, n, edges, levels=None):
        """`edges`: the closure's (ancestor, descendant) pairs, unique, sorted and checked; build one with
        from_closure_edges or from_parents."""
        self.n = int(n)
        self._set_levels(levels)
        e = self._edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
        self.n_anc = np.bincount(e[:, 1], minlength=n)
        self.n_desc = np.bincount(e[:, 0], minlength=n)
        # spanning forest: a node's tree parent is its ancestor with the most ancestors (always a direct parent),
        # ties to the larger id as in Hierarchy.from_closure_edges
        o = np.lexsort((self.n_anc[e[:, 0]], e[:, 1]))
        u, v = e[o, 0], e[o, 1]
        last = np.r_[v[1:] != v[:-1], True] if len(v) else np.zeros(0, dtype=bool)
        parents = np.full(n, -1, dtype=np.int64)
        parents[v[last]] = u[last]
        self.parents = parents
        self.tin = Hierarchy(parents).tin
        # every node's own number and its descendants' numbers, in order per node, cut into maximal runs; a run is
        # also cut before tin[u], so the run that starts there is the primary interval and the rest are extra
        a = np.concatenate([e[:, 0], np.arange(n)])
        t = np.concatenate([self.tin[e[:, 1]], self.tin])
        o = np.lexsort((t, a))
        a, t = a[o], t[o]
        first = np.r_[True, (a[1:] != a[:-1]) | (t[1:] != t[:-1] + 1)] | (t == self.tin[a])
        s = np.flatnonzero(first)
        owner, lo, hi = a[s], t[s], t[np.r_[s[1:] - 1, len(t) - 1]]
        primary = lo == self.tin[owner]
        self.tout = np.empty(n, dtype=np.int64)
        self.tout[owner[primary]] = hi[primary]
        x = ~primary
        self.extra_ptr = np.r_[0, np.cumsum(np.bincount(owner[x], minlength=n))].astype(np.int32)
        self.extra_lo = lo[x].astype(np.int32)
        self.extra_hi = hi[x].astype(np.int32)
        self._extra_key = owner[x] * self.n + lo[x]   # sorted: owner, then lo

    @classmethod
    def from_closure_edges(cls, n, edges, levels=None):
        """From (ancestor, descendant) pairs in any order -- the reference's G_tc edge list (order_embeddings.py:371).
        Raises ValueError for an endpoint outside [0, n), a self edge or a set that is not transitively closed (in a
        closed set a cycle implies a self edge)."""
        e, k = _edge_array(n, edges, "closure edge")
        if len(e) and not np.all(_in_sorted(_compose(e, e, n), k)):
            raise ValueError("the edges are not transitively closed")
        return cls(n, e, levels)

    @classmethod
    def from_parents(cls, n, edges, levels=None):
        """From direct (parent, child) edges; the closure is computed here.  Raises ValueError for an endpoint outside
        [0, n), a self edge or a cycle."""
        direct, known = _edge_array(n, edges, "parent edge")
        frontier = direct
        while len(frontier):   # pairs joined by a path of one more edge; a cycle shows up as a pair (u, u)
            k = np.unique(_compose(frontier, direct, n))
            if np.any(k // n == k % n):
                raise ValueError("the parent edges contain a cycle")
            k = k[~_in_sorted(k, known)]
            known = np.union1d(known, k)
            frontier = np.stack([k // n, k % n], axis=1)
        return cls(n, np.stack([known // n, known % n], axis=1), levels)

    def is_descendant(self, u, v):
        """v is a strict descendant of u (vectorised, broadcasting)."""
        u, v = np.broadcast_arrays(np.asarray(u, dtype=np.int64), np.asarray(v, dtype=np.int64))
        tv = self.tin[v]
        below = (tv > self.tin[u]) & (tv <= self.tout[u])
        if len(self.extra_lo):
            i = np.searchsorted(self._extra_key, u * self.n + tv, side="right") - 1   # last extra run starting <= tv
            below |= (i >= self.extra_ptr[u]) & (tv <= self.extra_hi[np.maximum(i, 0)])
        return below

    def closure_edges(self):
        """All (ancestor, descendant) pairs, sorted like Hierarchy.closure_edges."""
        return self._edges.copy()


def split_edges(h, val=0.05, test=0.05, train_nonbasic=1.0, seed=0):
    """Link-prediction split of the closure of h (the protocol of create_splits, order_embeddings.py:397-497): the
    basic edges -- the transitive reduction, pairs (u, v) with no w such that u > w > v; a Hierarchy's parent edges --
    always train; of the n_nb other closure edges int(val n_nb) go to "val", int(test n_nb) to "test" and
    int(train_nonbasic n_nb) of the rest to "train".  The draw is np.random.default_rng(seed)'s (not the reference's
    random.sample order).  Returns {"train", "val", "test"}, each int64 [m, 2] (ancestor, descendant), sorted."""
    e = h.closure_edges() if h.rank_slots()[0][-1] else np.zeros((0, 2), dtype=np.int64)
    n = h.n
    keys = _edge_keys(e, n)
    nonbasic = _in_sorted(keys, np.unique(_compose(e, e, n))) if len(e) else np.zeros(0, dtype=bool)
    basic, nb = keys[~nonbasic], keys[nonbasic]
    n_nb = len(nb)
    n_val, n_test = int(val * n_nb), int(test * n_nb)
    if n_val + n_test > n_nb:
        raise ValueError("val + test exceed the %d non-basic edges" % n_nb)
    perm = np.random.default_rng(seed).permutation(n_nb)
    n_train = min(int(train_nonbasic * n_nb), n_nb - n_val - n_test)
    parts = {"train": np.r_[basic, nb[perm[n_val + n_test:n_val + n_test + n_train]]],
             "val": nb[perm[:n_val]], "test": nb[perm[n_val:n_val + n_test]]}
    out = {}
    for name, k in parts.items():
        k = np.sort(k)
        out[name] = np.stack([k // n, k % n], axis=1).astype(np.int64)
    return out


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


def random_dag(n, gamma, frac, seed=0, roots=8):
    """random_tree(n, gamma, seed, roots) plus, for each non-root node with probability frac, a second parent drawn
    uniformly from the lower ids that are not already its ancestors (WordNet-like multiple inheritance; edges still
    point from lower to higher ids, so the graph is acyclic).  frac = 0 gives random_tree's closure."""
    par = random_tree(n, gamma, seed, roots).parents
    rng = np.random.default_rng([seed, 1])
    second = {}
    for i in np.flatnonzero(rng.random(n) < frac):
        i = int(i)
        if i < roots:
            continue
        anc, stack = set(), [int(par[i])]   # lower ids only: their parents are final
        while stack:
            a = stack.pop()
            if a < 0 or a in anc:
                continue
            anc.add(a)
            stack.append(int(par[a]))
            stack.append(second.get(a, -1))
        if len(anc) >= i:
            continue
        while True:
            j = int(rng.integers(0, i))
            if j not in anc:
                break
        second[i] = j
    has = np.flatnonzero(par >= 0)
    edges = np.concatenate([np.stack([par[has], has], axis=1),
                            np.array(sorted((p, c) for c, p in second.items()), dtype=np.int64).reshape(-1, 2)])
    return DagHierarchy.from_parents(n, edges)
