"""Reconstruction F1 on the GPU (metrics.reconstruction_f1 / lec_recon_*): bit-equal to the materialised path -- the SIMT
score matrix split by the Euler intervals, then best_f1_sweep -- on drawn and trained rows, adversarial inputs, small
workspaces (several rounds), hand-summed apex shards and padded engine rows; plus the cfg4-sized tree."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from learning_embeddings_b200 import _native, hierarchy, metrics, ops
from learning_embeddings_b200.engine import ConeStep, pack_index_block
from oracle import cones
from test_reconstruction_cpu import reconstruction_pairs

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
KS = {"euc": 3.0, "hyp": 0.1, "oe": 0.0}
ROW_MODE = {"euc": _native.ROWS_EUC_SOFTCLIP, "hyp": _native.ROWS_HYP_SHELL, "oe": _native.ROWS_NONE}


@functools.lru_cache(maxsize=None)
def tree(name):
    return hierarchy.ethec() if name == "ethec" else hierarchy.random_tree(4000, 1.0831, seed=1)


def drawn_table(n, D, geom, seed=0):
    """raw rows drawn like test_doc_training_iteration_equals_engine (shell of the inner radius for hyp)"""
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(n, D, generator=g)
    if geom == "hyp":
        r_in = cones.inner_radius(KS["hyp"])
        return (r_in + 0.05 * torch.rand(n, 1, generator=g)) * w / w.norm(dim=1, keepdim=True)
    return w


def drawn_rows(h, geom, D, seed=0):
    rows, _ = ops.rows_forward(drawn_table(h.n, D, geom, seed).to(DEV), ROW_MODE[geom], KS[geom], geom)
    return rows[:, :D].contiguous()


@functools.lru_cache(maxsize=None)
def trained_rows(name, geom, D, steps=200):
    """the engine's padded rows [n, ld] after `steps` ConeStep steps (E == 0 inside trained cones)"""
    h = tree(name)
    B, Nn = 1024, 5
    eng = ConeStep(drawn_table(h.n, D, geom).to(DEV), geom, Nn, B, K=KS[geom], alpha=0.05, lr=0.01)
    edges = h.closure_edges()
    rng = np.random.default_rng(0)
    for _ in range(steps):
        sel = rng.integers(0, len(edges), size=B)
        u, v = edges[sel, 0], edges[sel, 1]
        nt, nf = h.sample_negatives(u, v, Nn, rng)
        eng.step_device(*eng._split(pack_index_block(u, v, nt, nf).to(DEV), B))
    torch.cuda.synchronize()
    return eng.rows.clone(), eng.D


def split_matrix(rows, h, geom):
    """materialised path: the lec_score_topk_ex matrix (S[u, v] = E(x = u, y = v)) split by the Euler intervals"""
    n = rows.shape[0]
    S = torch.empty((n, n), device=DEV, dtype=torch.float32)
    ops.score_topk_into(rows, rows, geom, KS[geom], [], [], 1, None, None, S, 1, engine="simt")
    tin = torch.as_tensor(h.tin, device=DEV)
    tout = torch.as_tensor(h.tout, device=DEV)
    pos = (tin[:, None] < tin[None, :]) & (tin[None, :] <= tout[:, None])
    off = ~torch.eye(n, dtype=torch.bool, device=DEV)
    return S[pos], S[off & ~pos]


def check_equal(rows, h, geom, D=None, cpu_oracle=True, **kw):
    got = metrics.reconstruction_f1(rows, h, geom, KS[geom], D=D, **kw)
    contig = rows if D is None else rows[:, :D].contiguous()
    ep, en = split_matrix(contig, h, geom)
    want = metrics.best_f1_sweep(ep, en)
    assert np.array_equal(got, want, equal_nan=True), (got, want)
    if cpu_oracle:
        ref = np.array(cones.best_f1_sweep(ep.cpu(), en.cpu()))
        assert np.array_equal(got, ref), (got, ref)
    return got


@pytest.mark.parametrize("name", ["ethec", "tree4000"])
@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_exact_drawn_rows(geom, D, name):
    check_equal(drawn_rows(tree(name), geom, D), tree(name), geom)


@pytest.mark.parametrize("name", ["ethec", "tree4000"])
@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_exact_trained_rows(geom, D, name):
    rows, D = trained_rows(name, geom, D)
    check_equal(rows, tree(name), geom, D=D)


@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_quantised_rows_ties(geom):
    # six distinct rows shared by all nodes: fewer than 50 distinct energies, each carried by many pairs of both signs
    h = tree("ethec")
    base = drawn_rows(h, geom, 10)
    pick = torch.as_tensor(np.random.default_rng(3).integers(0, 6, size=h.n), device=DEV)
    rows = base[pick].contiguous()
    ep, en = split_matrix(rows, h, geom)
    e = torch.cat([ep, en])
    assert torch.unique(e[~torch.isnan(e)]).numel() < 50     # pairs of one row are NaN in hyp
    check_equal(rows, h, geom)


def test_zero_row_and_identical_rows():
    h = tree("ethec")
    rows = drawn_rows(h, "hyp", 10)
    rows[5] = 0.0                  # NaN apex row (the reference's zero label row)
    rows[100] = rows[200]          # two distinct nodes with one row: their pair is NaN and counts
    ep, en = split_matrix(rows, h, "hyp")
    assert bool(torch.isnan(ep).any()) and bool(torch.isnan(en).any())
    check_equal(rows, h, "hyp")
    rows_euc = drawn_rows(h, "euc", 10)
    rows_euc[100] = rows_euc[200]
    check_equal(rows_euc, h, "euc")


@pytest.mark.parametrize("geom", ["hyp", "oe"])
def test_forest_without_edges(geom):
    h = hierarchy.Hierarchy(np.full(500, -1))
    stats = {}
    got = check_equal(drawn_rows(h, geom, 10), h, geom, cpu_oracle=False, stats=stats)
    assert stats["n_pos"] == 0 and stats["n_neg"] == 500 * 499
    assert np.isnan(got[0])


def test_small_workspace_takes_rounds():
    # random rows: a flat F1 curve opens several coarse bins; one bin per round must give the same row
    small = int(_native.lib().lec_recon_workspace_bytes(1))
    opened = []
    for geom in ("euc", "hyp", "oe"):
        h = tree("tree4000")
        rows = drawn_rows(h, geom, 10, seed=7)
        big_stats, small_stats = {}, {}
        big = metrics.reconstruction_f1(rows, h, geom, KS[geom], stats=big_stats)
        got = metrics.reconstruction_f1(rows, h, geom, KS[geom], workspace_bytes=small, stats=small_stats)
        assert np.array_equal(got, big)
        assert small_stats["open_bins"] == big_stats["open_bins"]
        assert small_stats["rounds"] == 1 + small_stats["open_bins"]
        assert big_stats["rounds"] == 1 + -(-big_stats["open_bins"] // metrics.RECON_OPEN_BINS)
        opened.append(small_stats["open_bins"])
    assert max(opened) > 1, opened


def sharded(rows, h, geom, D, cuts, workspace_bytes):
    """three apex shards on one GPU, their counters summed by hand after every pass"""
    lib = _native.lib()
    tin = torch.as_tensor(h.tin, dtype=torch.int32, device=DEV)
    tout = torch.as_tensor(h.tout, dtype=torch.int32, device=DEV)
    cb = int(lib.lec_recon_counter_bytes(workspace_bytes))
    ws = [torch.zeros(workspace_bytes, device=DEV, dtype=torch.uint8) for _ in cuts[:-1]]
    args = [metrics.recon_args(rows, tin, tout, geom, KS[geom], D, a, b, w) for a, b, w in zip(cuts[:-1], cuts[1:], ws)]
    outs = [torch.empty(7, device=DEV, dtype=torch.float64) for _ in ws]
    status = [torch.zeros(4, device=DEV, dtype=torch.int64) for _ in ws]
    stream = _native.stream_ptr(DEV)
    for _ in range(10000):
        for r in args:
            _native.check(lib.lec_recon_pass(ctypes.byref(r), stream), "lec_recon_pass")
        total = sum(w[:cb].view(torch.int64) for w in ws)
        for w in ws:
            w[:cb].view(torch.int64).copy_(total)
        for r, o, s in zip(args, outs, status):
            _native.check(lib.lec_recon_finish(ctypes.byref(r), _native._p(o), _native._p(s), stream), "lec_recon_finish")
        st = [s.cpu().tolist() for s in status]
        assert all(x == st[0] for x in st)
        if st[0][0] == 0:
            break
    rows_out = [o.cpu().numpy() for o in outs]
    assert all(np.array_equal(x, rows_out[0]) for x in rows_out)
    return rows_out[0]


@pytest.mark.parametrize("geom,D", [("hyp", 10), ("euc", 50), ("oe", 2)])
def test_sharded_and_padded_rows(geom, D):
    h = tree("tree4000")
    rows, D = trained_rows("tree4000", geom, D)
    assert rows.shape[1] > D or D % 4 == 0
    ref = metrics.reconstruction_f1(rows[:, :D].contiguous(), h, geom, KS[geom])
    assert np.array_equal(metrics.reconstruction_f1(rows, h, geom, KS[geom], D=D), ref)   # padded engine rows
    n = h.n
    for nb in (int(_native.lib().lec_recon_workspace_bytes(1)), int(_native.lib().lec_recon_workspace_bytes(64))):
        got = sharded(rows, h, geom, D, [0, 17, 2900, n], nb)
        assert np.array_equal(got, ref), (got, ref)


def test_cfg4_scale():
    h = hierarchy.random_tree(82115, 1.0831)
    rows = drawn_rows(h, "hyp", 50)
    stats = {}
    got = metrics.reconstruction_f1(rows, h, "hyp", KS["hyp"], stats=stats)
    assert stats["n_pos"] == 741845
    assert stats["n_neg"] == 82115 * 82114 - 741845
    assert 0.0 <= got[0] <= 1.0
    assert got[5] <= 741845 and got[6] <= stats["n_neg"]
    assert stats["workspace_bytes"] < 256 << 20


def test_fp64_threshold_sanity():
    # the oracle's fp64 energies at the returned threshold give nearly the returned F1
    h = tree("ethec")
    rows, D = trained_rows("ethec", "hyp", 10)
    got = metrics.reconstruction_f1(rows, h, "hyp", KS["hyp"], D=D)
    u, v, pos = reconstruction_pairs(h)
    emb = rows[:, :D].double().cpu()
    E = cones.energy("hyp", emb[u], emb[v], KS["hyp"])
    ref = cones.metrics_at_threshold(E[pos], E[~pos], got[1])
    assert abs(ref[0] - got[0]) <= 1e-3, (ref, got)
