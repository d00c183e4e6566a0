"""Reconstruction F1 on DAG hierarchies without a GPU: DagHierarchy's interval cover, its constructors and negatives,
random_dag, and the argument checks of lec_recon_pass_dag."""
import ctypes

import numpy as np
import pytest

from learning_embeddings_b200 import _native, hierarchy
import test_reconstruction_cpu as forest
from test_reconstruction_cpu import FAKE, recon

DIAMOND = [(0, 1), (0, 2), (1, 3), (2, 3), (0, 3)]
# 0 -> {1, 2}; 1 -> {3, 4}; 2 -> {4, 5}; 3 -> 6; 4 -> {6, 7}; 8 is a root with child 5 and 7; closed below
SMALL_DAG_PARENTS = [(0, 1), (0, 2), (1, 3), (1, 4), (2, 4), (2, 5), (3, 6), (4, 6), (4, 7), (8, 5), (8, 7)]


def dense_closure(n, parent_edges):
    C = np.zeros((n, n), dtype=bool)
    for a, b in parent_edges:
        C[a, b] = True
    for k in range(n):   # Warshall
        C |= C[:, k:k + 1] & C[k:k + 1, :]
    return C


def descendant_sets_from_cover(d):
    """each node's descendants as the union of its primary (minus itself) and extra intervals of preorder numbers"""
    by_tin = np.argsort(d.tin)
    out = []
    for u in range(d.n):
        ts = list(range(int(d.tin[u]) + 1, int(d.tout[u]) + 1))
        for i in range(d.extra_ptr[u], d.extra_ptr[u + 1]):
            ts += range(int(d.extra_lo[i]), int(d.extra_hi[i]) + 1)
        out.append(set(by_tin[ts].tolist()))
    return out


@pytest.mark.parametrize("make", [hierarchy.ethec, lambda: hierarchy.random_tree(2000, 1.0831)], ids=["ethec", "random_tree"])
def test_forest_closure_gives_euler_intervals(make):
    h = make()
    e = h.closure_edges()
    d = hierarchy.DagHierarchy.from_closure_edges(h.n, e[np.random.default_rng(0).permutation(len(e))])
    assert np.array_equal(d.tin, h.tin) and np.array_equal(d.tout, h.tout)
    assert int(d.extra_ptr[-1]) == 0 and len(d.extra_lo) == 0 and len(d.extra_ptr) == h.n + 1
    assert np.array_equal(d.closure_edges(), e)
    assert np.array_equal(d.n_desc, h.n_desc) and np.array_equal(d.n_anc, h.n_anc)


@pytest.mark.parametrize("n, parent_edges", [(4, [(0, 1), (0, 2), (1, 3), (2, 3)]), (9, SMALL_DAG_PARENTS)],
                         ids=["diamond", "small_dag"])
def test_diamonds_are_accepted(n, parent_edges):
    C = dense_closure(n, parent_edges)
    want = np.argwhere(C)
    rng = np.random.default_rng(1)
    d = hierarchy.DagHierarchy.from_closure_edges(n, want[rng.permutation(len(want))])
    assert np.array_equal(d.closure_edges(), want)
    u, v = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    assert np.array_equal(d.is_descendant(u, v), C)
    assert np.array_equal(d.negative_adjacency(), ~C & ~np.eye(n, dtype=bool))
    p = hierarchy.DagHierarchy.from_parents(n, parent_edges)
    assert np.array_equal(p.closure_edges(), want)
    assert np.array_equal(p.tin, d.tin) and np.array_equal(p.tout, d.tout)
    assert np.array_equal(p.extra_ptr, d.extra_ptr) and np.array_equal(p.extra_lo, d.extra_lo)
    # round trip through the edge list
    e = hierarchy.DagHierarchy.from_closure_edges(n, d.closure_edges())
    assert np.array_equal(e.closure_edges(), want) and np.array_equal(e.extra_hi, d.extra_hi)


def test_diamond_cover():
    # node 3's ancestors 1 and 2 tie for its tree parent and the larger id wins: spanning forest 0 -> {1, 2}, 2 -> 3
    d = hierarchy.DagHierarchy.from_closure_edges(4, DIAMOND)
    assert d.parents.tolist() == [-1, 0, 0, 2]
    assert d.tin.tolist() == [0, 1, 2, 3] and d.tout.tolist() == [3, 1, 3, 3]
    assert d.extra_ptr.tolist() == [0, 0, 1, 1, 1]    # node 1 reaches 3 (preorder 3) outside [1, 1]
    assert d.extra_lo.tolist() == [3] and d.extra_hi.tolist() == [3]


@pytest.mark.parametrize("n, edges", [
    (3, [(0, 1), (1, 1), (0, 2)]),           # self edge
    (3, [(0, 1), (0, 3)]),                   # endpoint past n
    (3, [(-1, 1)]),                          # negative endpoint
    (3, [(0, 1), (1, 2)]),                   # transitive edge (0, 2) missing
    (4, DIAMOND[:-1]),                       # diamond without (0, 3)
    (2, [(0, 1), (1, 0)]),                   # cycle (its closure would need (0, 0))
    (3, [(0, 1), (1, 2), (2, 0), (0, 2), (1, 0), (2, 1)]),   # closed apart from the self edges: a cycle
])
def test_from_closure_edges_rejects(n, edges):
    with pytest.raises(ValueError):
        hierarchy.DagHierarchy.from_closure_edges(n, edges)


def test_from_parents_rejects():
    for n, edges in [(3, [(0, 1), (1, 2), (2, 0)]), (2, [(1, 1)]), (2, [(0, 2)])]:
        with pytest.raises(ValueError):
            hierarchy.DagHierarchy.from_parents(n, edges)


def test_no_edges_and_levels():
    d = hierarchy.DagHierarchy.from_closure_edges(5, np.zeros((0, 2), dtype=np.int64), levels=[2, 3])
    assert d.tin.tolist() == [0, 1, 2, 3, 4] and d.tout.tolist() == [0, 1, 2, 3, 4]
    assert d.level_start == [0, 2] and d.level_stop == [2, 5]
    assert not d.is_descendant(np.arange(5), np.arange(5)[::-1]).any()


def test_interval_cover_invariants():
    d = hierarchy.random_dag(4000, 1.0831, 0.05)
    assert int(d.extra_ptr[-1]) > 0
    e = d.closure_edges()
    desc = [set() for _ in range(d.n)]
    for a, b in e.tolist():
        desc[a].add(b)
    for u in range(d.n):
        lo, hi = d.extra_lo[d.extra_ptr[u]:d.extra_ptr[u + 1]], d.extra_hi[d.extra_ptr[u]:d.extra_ptr[u + 1]]
        assert np.all(lo <= hi)
        assert np.all(lo[1:] > hi[:-1])                                          # sorted and disjoint
        assert not np.any((lo <= d.tout[u]) & (hi >= d.tin[u]))                  # outside the primary interval
    assert descendant_sets_from_cover(d) == desc                                 # union = descendant set
    assert np.array_equal(d.n_desc, [len(s) for s in desc])
    # the vectorised query against the sets
    rng = np.random.default_rng(2)
    u, v = rng.integers(0, d.n, 200000), rng.integers(0, d.n, 200000)
    u = np.concatenate([u, e[:, 0]])
    v = np.concatenate([v, e[:, 1]])
    assert np.array_equal(d.is_descendant(u, v), np.array([b in desc[a] for a, b in zip(u.tolist(), v.tolist())]))


def test_random_dag_without_extra_parents_is_random_tree():
    for n, seed in [(2000, 0), (5000, 3)]:
        d = hierarchy.random_dag(n, 1.0831, 0.0, seed=seed)
        t = hierarchy.random_tree(n, 1.0831, seed=seed)
        assert np.array_equal(d.closure_edges(), t.closure_edges())
        assert np.array_equal(d.tin, t.tin) and np.array_equal(d.tout, t.tout) and int(d.extra_ptr[-1]) == 0


def test_random_dag_is_a_dag_with_second_parents():
    d = hierarchy.random_dag(3000, 1.0831, 0.05, seed=4)
    t = hierarchy.random_tree(3000, 1.0831, seed=4)
    e = d.closure_edges()
    assert np.all(e[:, 0] < e[:, 1])
    te = t.closure_edges()
    assert len(e) > len(te)
    assert np.all(np.isin(te[:, 0] * 3000 + te[:, 1], e[:, 0] * 3000 + e[:, 1]))   # the tree's edges stay
    assert np.array_equal(d.n_anc[:8], np.zeros(8))                                # roots stay roots


def test_dag_negatives_exclude_the_closure():
    d = hierarchy.random_dag(4000, 1.0831, 0.05)
    e = d.closure_edges()
    rng = np.random.default_rng(5)
    sel = rng.integers(0, len(e), 5000)
    u, v = e[sel, 0], e[sel, 1]
    nt, nf = d.sample_negatives(u, v, 5, rng)
    keys = set((e[:, 0] * d.n + e[:, 1]).tolist())
    assert not np.any(nt == u[:, None]) and not np.any(nf == v[:, None])
    assert not any(a * d.n + b in keys for a, b in zip(np.repeat(u, 5).tolist(), nt.reshape(-1).tolist()))
    assert not any(a * d.n + b in keys for a, b in zip(nf.reshape(-1).tolist(), np.repeat(v, 5).tolist()))
    # the SamplerGraph route of training only reads the closure edges and the level bounds
    from learning_embeddings_b200.sampler import SamplerGraph
    SamplerGraph.from_hierarchy(d)


def test_dag_negatives_raise_when_there_is_no_candidate():
    # 0 -> {1, 2} -> 3: node 3 is below every other node, node 0 above every other node
    d = hierarchy.DagHierarchy.from_closure_edges(4, DIAMOND)
    rng = np.random.default_rng(0)
    with pytest.raises(IndexError):
        d.sample_negatives([1], [3], 2, rng)
    with pytest.raises(IndexError):
        d.sample_negatives([0], [1], 2, rng)


def parent_sample_negatives(h, u, v, n_neg, rng):
    """Hierarchy.sample_negatives as it was before the base class: rejection on the Euler intervals"""
    u, v = np.asarray(u), np.asarray(v)
    B = len(u)
    uu, vv = np.repeat(u[:, None], n_neg, 1), np.repeat(v[:, None], n_neg, 1)
    if len(u) and int((h.tout[u] - h.tin[u]).max()) >= h.n - 1:
        raise IndexError("no negative candidate")
    neg_to = rng.integers(0, h.n, size=(B, n_neg))
    neg_from = rng.integers(0, h.n, size=(B, n_neg))
    below = lambda a, b: (h.tin[b] > h.tin[a]) & (h.tin[b] <= h.tout[a])   # noqa: E731
    while True:
        bad = (neg_to == uu) | below(uu, neg_to)
        k = int(bad.sum())
        if k == 0:
            break
        neg_to[bad] = rng.integers(0, h.n, size=k)
    while True:
        bad = (neg_from == vv) | below(neg_from, vv)
        k = int(bad.sum())
        if k == 0:
            break
        neg_from[bad] = rng.integers(0, h.n, size=k)
    return neg_to, neg_from


@pytest.mark.parametrize("make", [hierarchy.ethec, lambda: hierarchy.random_tree(4000, 1.0831, seed=1)], ids=["ethec", "tree"])
def test_hierarchy_negatives_unchanged(make):
    h = make()
    e = h.closure_edges()
    sel = np.random.default_rng(6).integers(0, len(e), 3000)
    got = h.sample_negatives(e[sel, 0], e[sel, 1], 5, np.random.default_rng(7))
    want = parent_sample_negatives(h, e[sel, 0], e[sel, 1], 5, np.random.default_rng(7))
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    star = hierarchy.Hierarchy([-1, 0, 0, 0])
    with pytest.raises(IndexError):
        star.sample_negatives([0], [1], 2, np.random.default_rng(0))
    # a chain: node 2 is below every other node, so "corrupt the parent" has no candidate (this used to loop forever)
    chain = hierarchy.Hierarchy([-1, 0, 1])
    with pytest.raises(IndexError):
        chain.sample_negatives([1], [2], 2, np.random.default_rng(0))


def extra(**kw):
    x = _native.LecReconExtra(FAKE, FAKE, FAKE, 10)
    for k, v in kw.items():
        setattr(x, k, v)
    return x


@pytest.mark.parametrize("fields, code", [
    (dict(ptr=0), -1), (dict(lo=0), -1), (dict(hi=0), -1),
    (dict(count=-1), -4), (dict(count=1 << 31), -4), (dict(count=-1, ptr=0), -4),
])
def test_dag_pass_validation_codes(fields, code):
    lib = _native.lib()
    assert "lec_recon_pass_dag" in _native.EXPORTS
    assert lib.lec_recon_pass_dag(ctypes.byref(recon()), ctypes.byref(extra(**fields)), ctypes.c_void_p(0)) == code


@pytest.mark.parametrize("fields, code", forest.test_argument_validation_codes.pytestmark[0].args[1])
def test_dag_pass_without_extra_is_recon_pass(fields, code):
    lib = _native.lib()
    null = ctypes.c_void_p(0)
    r = recon(**fields)
    assert lib.lec_recon_pass_dag(ctypes.byref(r), None, null) == lib.lec_recon_pass(ctypes.byref(r), null) == code
    assert lib.lec_recon_pass_dag(ctypes.byref(r), ctypes.byref(extra(count=0, ptr=0)), null) == code
    # an invalid lec_recon_t is reported before the extra intervals are looked at
    assert lib.lec_recon_pass_dag(ctypes.byref(r), ctypes.byref(extra(ptr=0)), null) == code


def test_dag_pass_edges():
    lib = _native.lib()
    null = ctypes.c_void_p(0)
    assert lib.lec_recon_pass_dag(None, None, null) == -1
    assert lib.lec_recon_pass_dag(ctypes.byref(recon(u_begin=40, u_end=40)), ctypes.byref(extra()), null) == 0
