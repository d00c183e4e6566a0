"""Reconstruction F1 on DAG hierarchies on the GPU (metrics.reconstruction_f1 with a DagHierarchy / lec_recon_pass_dag):
bit-equal to the materialised path -- the SIMT score matrix split by the dense DAG closure, then best_f1_sweep -- on
drawn and trained rows, an apex with over a thousand extra intervals, ties, a zero row, small workspaces, hand-summed
apex shards and padded engine rows; a forest given as a DagHierarchy; and the cfg4-sized DAG."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from learning_embeddings_b200 import _native, hierarchy, metrics
from learning_embeddings_b200.engine import ConeStep, pack_index_block
from learning_embeddings_b200.sampler import SamplerGraph
from oracle import cones
from test_reconstruction_gpu import KS, drawn_rows, drawn_table

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def wide_apex_dag(n=6000, apex=3, seed=2):
    """random_tree plus `apex` as an extra parent of every other leaf that is not already below it"""
    t = hierarchy.random_tree(n, 1.0831, seed=seed)
    leaves = np.setdiff1d(np.arange(n), t.parents)
    leaves = leaves[~t.is_descendant(apex, leaves) & (leaves != apex)][::2]
    has = np.flatnonzero(t.parents >= 0)
    edges = np.concatenate([np.stack([t.parents[has], has], 1), np.stack([np.full(len(leaves), apex), leaves], 1)])
    return hierarchy.DagHierarchy.from_parents(n, edges)


@functools.lru_cache(maxsize=None)
def dag(name):
    if name == "dag4000":
        return hierarchy.random_dag(4000, 1.0831, 0.05)
    if name == "diamonds":   # 600 nodes, a second parent for half of them
        return hierarchy.random_dag(600, 1.0831, 0.5, seed=3)
    if name == "wide_apex":
        return wide_apex_dag()
    raise KeyError(name)


def split_matrix(rows, h, geom):
    """materialised path: the lec_score_topk_ex matrix (S[u, v] = E(x = u, y = v)) split by the dense closure"""
    from learning_embeddings_b200 import ops
    n = rows.shape[0]
    S = torch.empty((n, n), device=DEV, dtype=torch.float32)
    ops.score_topk_into(rows, rows, geom, KS[geom], [], [], 1, None, None, S, 1, engine="simt")
    e = torch.as_tensor(h.closure_edges(), device=DEV)
    pos = torch.zeros((n, n), dtype=torch.bool, device=DEV)
    pos[e[:, 0], e[:, 1]] = True
    off = ~torch.eye(n, dtype=torch.bool, device=DEV)
    return S[pos], S[off & ~pos]


def check_equal(rows, h, geom, D=None, cpu_oracle=True, **kw):
    stats = kw.setdefault("stats", {})
    got = metrics.reconstruction_f1(rows, h, geom, KS[geom], D=D, **kw)
    contig = rows if D is None else rows[:, :D].contiguous()
    ep, en = split_matrix(contig, h, geom)
    assert stats["n_pos"] == ep.numel() and stats["n_neg"] == en.numel()
    assert stats["extra_intervals"] == int(h.extra_ptr[-1])
    want = metrics.best_f1_sweep(ep, en)
    assert np.array_equal(got, want, equal_nan=True), (got, want)
    if cpu_oracle:
        ref = np.array(cones.best_f1_sweep(ep.cpu(), en.cpu()))
        assert np.array_equal(got, ref), (got, ref)
    return got


@functools.lru_cache(maxsize=None)
def trained_rows(name, geom, D, steps=200):
    """the engine's padded rows after `steps` ConeStep steps on the DAG, negatives from the device sampler"""
    h = dag(name)
    B, Nn = 1024, 5
    eng = ConeStep(drawn_table(h.n, D, geom).to(DEV), geom, Nn, B, K=KS[geom], alpha=0.05, lr=0.01)
    edges = h.closure_edges()
    graph = SamplerGraph.from_hierarchy(h)
    rng = np.random.default_rng(0)
    for step in range(steps):
        sel = rng.integers(0, len(edges), size=B)
        u, v = edges[sel, 0], edges[sel, 1]
        nt, nf = graph.draw_philox(torch.from_numpy(u).to(DEV), torch.from_numpy(v).to(DEV), Nn, seed=11, step=step)
        eng.step_device(*eng._split(pack_index_block(u, v, nt.cpu().numpy(), nf.cpu().numpy()).to(DEV), B))
    torch.cuda.synchronize()
    return eng.rows.clone(), eng.D


def test_workloads_have_extra_intervals():
    assert int(dag("dag4000").extra_ptr[-1]) > 0 and int(dag("diamonds").extra_ptr[-1]) > 0
    assert int(np.diff(dag("wide_apex").extra_ptr).max()) > 1000


@pytest.mark.parametrize("name", ["dag4000", "diamonds"])
@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_exact_drawn_rows(geom, D, name):
    check_equal(drawn_rows(dag(name), geom, D), dag(name), geom)


@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_exact_trained_rows(geom, D):
    rows, D = trained_rows("dag4000", geom, D)
    check_equal(rows, dag("dag4000"), geom, D=D)


@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_apex_with_many_extra_intervals(geom, D):
    check_equal(drawn_rows(dag("wide_apex"), geom, D), dag("wide_apex"), geom)


@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_quantised_rows_ties_and_zero_row(geom):
    h = dag("diamonds")
    base = drawn_rows(h, geom, 10)
    pick = torch.as_tensor(np.random.default_rng(3).integers(0, 6, size=h.n), device=DEV)
    rows = base[pick].contiguous()
    check_equal(rows, h, geom)
    rows = drawn_rows(h, geom, 10)
    rows[int(np.argmax(np.diff(h.extra_ptr)))] = 0.0   # the apex with the most extra intervals
    check_equal(rows, h, geom)


def test_small_workspace_takes_rounds():
    small = int(_native.lib().lec_recon_workspace_bytes(1))
    h = dag("dag4000")
    opened = []
    for geom in ("euc", "hyp", "oe"):
        rows = drawn_rows(h, geom, 10, seed=7)
        big_stats, small_stats = {}, {}
        big = metrics.reconstruction_f1(rows, h, geom, KS[geom], stats=big_stats)
        got = check_equal(rows, h, geom, cpu_oracle=False, workspace_bytes=small, stats=small_stats)
        assert np.array_equal(got, big)
        assert small_stats["rounds"] == 1 + small_stats["open_bins"] == 1 + big_stats["open_bins"]
        opened.append(small_stats["open_bins"])
    assert max(opened) > 1, opened


def dag_sharded(rows, h, geom, D, cuts, workspace_bytes):
    """three apex shards on one GPU through lec_recon_pass_dag, their counters summed by hand after every pass"""
    lib = _native.lib()
    tin = torch.as_tensor(h.tin, dtype=torch.int32, device=DEV)
    tout = torch.as_tensor(h.tout, dtype=torch.int32, device=DEV)
    xptr, xlo, xhi = (torch.as_tensor(a, dtype=torch.int32, device=DEV) for a in (h.extra_ptr, h.extra_lo, h.extra_hi))
    x = _native.LecReconExtra(xptr.data_ptr(), xlo.data_ptr(), xhi.data_ptr(), int(h.extra_ptr[-1]))
    cb = int(lib.lec_recon_counter_bytes(workspace_bytes))
    ws = [torch.zeros(workspace_bytes, device=DEV, dtype=torch.uint8) for _ in cuts[:-1]]
    args = [metrics.recon_args(rows, tin, tout, geom, KS[geom], D, a, b, w) for a, b, w in zip(cuts[:-1], cuts[1:], ws)]
    outs = [torch.empty(7, device=DEV, dtype=torch.float64) for _ in ws]
    status = [torch.zeros(4, device=DEV, dtype=torch.int64) for _ in ws]
    stream = _native.stream_ptr(DEV)
    for _ in range(10000):
        for r in args:
            _native.check(lib.lec_recon_pass_dag(ctypes.byref(r), ctypes.byref(x), stream), "lec_recon_pass_dag")
        total = sum(w[:cb].view(torch.int64) for w in ws)
        for w in ws:
            w[:cb].view(torch.int64).copy_(total)
        for r, o, s in zip(args, outs, status):
            _native.check(lib.lec_recon_finish(ctypes.byref(r), _native._p(o), _native._p(s), stream), "lec_recon_finish")
        st = [s.cpu().tolist() for s in status]
        assert all(v == st[0] for v in st)
        if st[0][0] == 0:
            break
    rows_out = [o.cpu().numpy() for o in outs]
    assert all(np.array_equal(v, rows_out[0]) for v in rows_out)
    return rows_out[0]


@pytest.mark.parametrize("geom,D", [("hyp", 10), ("euc", 50), ("oe", 2)])
def test_sharded_and_padded_rows(geom, D):
    h = dag("dag4000")
    rows, D = trained_rows("dag4000", geom, D)
    assert rows.shape[1] > D or D % 4 == 0
    ref = metrics.reconstruction_f1(rows[:, :D].contiguous(), h, geom, KS[geom])
    assert np.array_equal(metrics.reconstruction_f1(rows, h, geom, KS[geom], D=D), ref)   # padded engine rows
    # a shard boundary inside a run of consecutive apexes with extra intervals
    has = np.diff(h.extra_ptr) > 0
    run = int(np.flatnonzero(has[:-1] & has[1:])[0]) + 1
    for nb in (int(_native.lib().lec_recon_workspace_bytes(1)), int(_native.lib().lec_recon_workspace_bytes(64))):
        got = dag_sharded(rows, h, geom, D, [0, run, 2900, h.n], nb)
        assert np.array_equal(got, ref), (got, ref)


@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_forest_as_dag_hierarchy_is_bit_equal(geom):
    t = hierarchy.random_tree(4000, 1.0831, seed=1)
    d = hierarchy.DagHierarchy.from_closure_edges(t.n, t.closure_edges())
    rows = drawn_rows(t, geom, 10)
    stats = {}
    got = metrics.reconstruction_f1(rows, d, geom, KS[geom], stats=stats)
    assert stats["extra_intervals"] == 0
    assert np.array_equal(got, metrics.reconstruction_f1(rows, t, geom, KS[geom]), equal_nan=True)


def test_cfg4_scale():
    h = hierarchy.random_dag(82115, 1.0831, 0.02)
    n_pos = len(h.closure_edges())
    rows = drawn_rows(h, "hyp", 50)
    stats = {}
    got = metrics.reconstruction_f1(rows, h, "hyp", KS["hyp"], stats=stats)
    assert stats["extra_intervals"] > 0
    assert stats["n_pos"] == n_pos
    assert stats["n_neg"] == 82115 * 82114 - n_pos
    assert 0.0 <= got[0] <= 1.0
    assert got[5] <= n_pos and got[6] <= stats["n_neg"]
    assert stats["workspace_bytes"] < 256 << 20
