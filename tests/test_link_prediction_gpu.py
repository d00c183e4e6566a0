"""Link prediction on held-out closure edges on the GPU (metrics.link_prediction_ranks / link_prediction_f1): with every
closure edge held out, bit-identical to reconstruction_ranks / reconstruction_f1; on split_edges held-out sets, equal to
the materialised SIMT matrix plus the dense reference (ranks as integers, AP within 1e-12 relative, F1 rows bit for
bit against best_f1_sweep and EmbeddingMetrics(..., 'test'))."""
import ctypes
import functools
import math

import numpy as np
import pytest
import torch

from learning_embeddings_b200 import _native, hierarchy, metrics, ops
from learning_embeddings_b200.engine import ConeStep, pack_index_block
from test_link_prediction_cpu import link_prediction_oracle
from test_reconstruction_dag_gpu import dag
from test_reconstruction_gpu import KS, drawn_rows, drawn_table, trained_rows, tree

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@functools.lru_cache(maxsize=None)
def graph(name):
    return dag(name) if name == "dag4000" else tree(name)


@functools.lru_cache(maxsize=None)
def trained_dag_rows(geom, D, steps=200):
    """the engine's padded rows after ConeStep steps on dag4000's closure"""
    h = graph("dag4000")
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


def matrix(rows, h, geom, D=None, sample=None):
    x = rows if D is None else rows[:, :D].contiguous()
    sample = np.arange(h.n) if sample is None else sample
    S = torch.empty((len(sample), h.n), device=DEV, dtype=torch.float32)
    ops.score_topk_into(x[torch.as_tensor(sample, device=DEV)].contiguous(), x, geom, KS[geom], [], [], 1, None, None, S,
                        1, engine="simt")
    return S


def masks(h, edges, sample):
    below = h.is_descendant(sample[:, None], np.arange(h.n)[None, :])
    row = np.full(h.n, -1)
    row[sample] = np.arange(len(sample))
    e = np.asarray(edges).reshape(-1, 2)
    e = e[row[e[:, 0]] >= 0]
    held = np.zeros_like(below)
    held[row[e[:, 0]], e[:, 1]] = True
    return below, held


def check_ranks(rows, h, geom, edges, D=None, sample=None, got=None):
    """link_prediction_ranks against the score matrix rows of `sample` (every apex by default) and the oracle"""
    edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    if got is None:
        got = metrics.link_prediction_ranks(rows, h, edges, geom, KS[geom], D=D, return_ranks=True)
    sample = np.arange(h.n) if sample is None else np.unique(sample)
    S = matrix(rows, h, geom, D, sample)
    below, held = masks(h, edges, sample)
    ranks, ap = link_prediction_oracle(S.cpu().numpy(), below, held, apex=sample)
    assert got["n_edges"] == len(edges) and got["n_apexes"] == len(np.unique(edges[:, 0]))
    sel = np.flatnonzero(np.isin(edges[:, 0], sample))
    sel = sel[np.lexsort((edges[sel, 1], edges[sel, 0]))]     # the oracle's row-major order
    assert np.array_equal(got["ranks"].cpu().numpy()[sel], ranks)
    has = held.any(1)
    assert np.all(np.isnan(got["ap"][sample][~has]))
    np.testing.assert_allclose(got["ap"][sample][has], ap[has], rtol=1e-12, atol=0)
    if len(sample) == h.n and len(edges):
        assert got["mean_rank"] == ranks[:, 1].sum() / len(edges)
        assert got["mean_rank_optimistic"] == ranks[:, 0].sum() / len(edges)
        want = math.fsum(ap[has].tolist()) / int(has.sum())
        assert abs(got["map"] - want) <= 1e-12 * want, (got["map"], want)
    return got


def split_energies(rows, h, geom, edges, D=None):
    S = matrix(rows, h, geom, D)
    below, held = masks(h, edges, np.arange(h.n))
    neg = ~below
    np.fill_diagonal(neg, False)
    return S[torch.as_tensor(held, device=DEV)], S[torch.as_tensor(neg, device=DEV)]


def em_row(ep, en, t):
    return np.array(metrics.EmbeddingMetrics(ep, en, t, "test").calculate_metrics(), dtype=np.float64)


def same(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64), equal_nan=True)


def check_full_closure(rows, h, geom, D=None):
    e = h.closure_edges()
    got = metrics.link_prediction_ranks(rows, h, e, geom, KS[geom], D=D, return_ranks=True)
    want = metrics.reconstruction_ranks(rows, h, geom, KS[geom], D=D, return_ranks=True)
    assert torch.equal(got["ranks"], want["ranks"])
    assert np.array_equal(got["ap"], want["ap"], equal_nan=True)
    for k in ("mean_rank", "mean_rank_optimistic", "map", "n_edges", "n_apexes"):
        assert got[k] == want[k], k
    f1 = metrics.link_prediction_f1(rows, h, e, geom, KS[geom], D=D)
    assert same(f1, metrics.reconstruction_f1(rows, h, geom, KS[geom], D=D))


@pytest.mark.parametrize("name", ["ethec", "tree4000", "dag4000"])
@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_full_closure_is_reconstruction(geom, D, name):
    check_full_closure(drawn_rows(graph(name), geom, D), graph(name), geom)


@pytest.mark.parametrize("name", ["tree4000", "dag4000"])
@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_full_closure_is_reconstruction_padded_rows(geom, D, name):
    rows, D = trained_rows(name, geom, D) if name == "tree4000" else trained_dag_rows(geom, D)
    check_full_closure(rows, graph(name), geom, D=D)


@pytest.mark.parametrize("frac", [0.05, 0.25, 0.5])
@pytest.mark.parametrize("name", ["ethec", "tree4000", "dag4000"])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_split_exact(geom, name, frac):
    h = graph(name)
    rows = drawn_rows(h, geom, 10)
    test = hierarchy.split_edges(h, val=frac, test=frac, seed=1)["test"]
    check_ranks(rows, h, geom, test)
    ep, en = split_energies(rows, h, geom, test)
    stats = {}
    best = metrics.link_prediction_f1(rows, h, test, geom, KS[geom], stats=stats)
    assert same(best, metrics.best_f1_sweep(ep, en))
    assert stats["n_pos"] == len(test) and stats["skipped_pairs"] == len(h.closure_edges()) - len(test)
    # the counts of the best row come back at its own threshold
    at = metrics.link_prediction_f1(rows, h, test, geom, KS[geom], threshold=float(best[1]))
    assert at[5] == best[5] and at[6] == best[6] and at[1] == best[1]


@pytest.mark.parametrize("name", ["tree4000", "dag4000"])
@pytest.mark.parametrize("geom", ["euc", "hyp"])
def test_threshold_rows(geom, name):
    h = graph(name)
    rows = drawn_rows(h, geom, 10)
    rows[7] = 0.0                      # a zero row: NaN energies for hyp
    rows[100] = rows[200]
    s = hierarchy.split_edges(h, val=0.25, test=0.25, seed=2)
    t_val = float(metrics.link_prediction_f1(rows, h, s["val"], geom, KS[geom])[1])
    ep, en = split_energies(rows, h, geom, s["test"])
    occurs = float(ep[len(ep) // 2])   # an energy that occurs: a tie at the threshold
    for t in (t_val, 0.0, -0.0, math.inf, occurs, float(en[0]), -0.5, math.nan):
        stats = {}
        got = metrics.link_prediction_f1(rows, h, s["test"], geom, KS[geom], threshold=t, stats=stats)
        want = em_row(ep, en, t)
        assert same(got, want), (t, got, want)
        assert stats["rounds"] <= 2
    if geom == "hyp":
        assert bool(torch.isnan(en).any())


def test_empty_heldout_set():
    h = graph("tree4000")
    rows = drawn_rows(h, "hyp", 10)
    got = metrics.link_prediction_ranks(rows, h, np.zeros((0, 2), dtype=np.int64), "hyp", KS["hyp"], return_ranks=True)
    assert got["n_edges"] == 0 and got["n_apexes"] == 0 and got["ranks"].shape == (0, 2)
    assert all(math.isnan(got[k]) for k in ("mean_rank", "mean_rank_optimistic", "map"))
    assert np.all(np.isnan(got["ap"]))
    stats = {}
    row = metrics.link_prediction_f1(rows, h, np.zeros((0, 2), dtype=np.int64), "hyp", KS["hyp"], stats=stats)
    assert stats["n_pos"] == 0 and math.isnan(row[4])
    _, en = split_energies(rows, h, "hyp", np.zeros((0, 2), dtype=np.int64))
    assert stats["n_neg"] == en.numel()
    at = metrics.link_prediction_f1(rows, h, np.zeros((0, 2), dtype=np.int64), "hyp", KS["hyp"], threshold=0.5)
    assert at[5] == 0 and at[6] == int((en > 0.5).sum()) and at[3] == 0.0


@pytest.mark.parametrize("name", ["tree4000", "dag4000"])
def test_apexes_with_all_or_none_held_out(name):
    h = graph(name)
    rows = drawn_rows(h, "hyp", 10)
    e = h.closure_edges()
    big = np.argsort(h.n_desc)[-6:]
    rng = np.random.default_rng(5)
    keep = (rng.random(len(e)) < 0.3) | np.isin(e[:, 0], big[:3])   # all of three large apexes' pairs
    keep &= ~np.isin(e[:, 0], big[3:])                              # none of three others'
    got = check_ranks(rows, h, "hyp", e[keep])
    assert np.all(np.isnan(got["ap"][big[3:]])) and not np.any(np.isnan(got["ap"][big[:3]]))
    ep, en = split_energies(rows, h, "hyp", e[keep])
    assert same(metrics.link_prediction_f1(rows, h, e[keep], "hyp", KS["hyp"]), metrics.best_f1_sweep(ep, en))


def test_apex_shards_add_up_and_calls_are_bit_identical():
    lib = _native.lib()
    for name, geom in (("tree4000", "hyp"), ("dag4000", "euc")):
        h = graph(name)
        rows = drawn_rows(h, geom, 10)
        test = hierarchy.split_edges(h, val=0.1, test=0.1, seed=3)["test"]
        one = metrics.link_prediction_ranks(rows, h, test, geom, KS[geom], return_ranks=True)
        two = metrics.link_prediction_ranks(rows, h, test, geom, KS[geom], return_ranks=True)
        assert np.array_equal(one["ap"], two["ap"], equal_nan=True) and torch.equal(one["ranks"], two["ranks"])
        assert one["map"] == two["map"] and one["mean_rank"] == two["mean_rank"]
        f_one = metrics.link_prediction_f1(rows, h, test, geom, KS[geom])
        assert same(f_one, metrics.link_prediction_f1(rows, h, test, geom, KS[geom]))
        t = float(f_one[1]) * 1.5
        f_at = metrics.link_prediction_f1(rows, h, test, geom, KS[geom], threshold=t)
        assert same(f_at, metrics.link_prediction_f1(rows, h, test, geom, KS[geom], threshold=t))

        held = metrics._Heldout(h, test, DEV)
        cov = metrics._Cover(h, DEV)
        n_pos = len(test)
        cuts = [0, 17, 2900, h.n]
        # ranks: one lec_rank_run_heldout per shard
        nb = int(lib.lec_rank_workspace_bytes(h.n, n_pos))
        total = torch.zeros(3, dtype=torch.int64, device=DEV)
        ap = torch.zeros(h.n, dtype=torch.float64, device=DEV)
        ranks = torch.zeros((n_pos, 2), dtype=torch.int32, device=DEV)
        for a, b in zip(cuts[:-1], cuts[1:]):
            ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
            r = metrics.rank_args(rows, cov.tin, cov.tout, cov.x, held.eval_ptr, n_pos, geom, KS[geom], 10, a, b, ws)
            sums = torch.empty(3, dtype=torch.int64, device=DEV)
            part = torch.zeros(h.n, dtype=torch.float64, device=DEV)
            _native.check(lib.lec_rank_run_heldout(ctypes.byref(r), ctypes.byref(held.h), _native._p(sums),
                                                   _native._p(part), _native._p(ranks), _native.stream_ptr(DEV)),
                          "lec_rank_run_heldout")
            total += sums
            ap += part
        assert int(total[1]) == round(one["mean_rank"] * n_pos)
        assert int(total[0]) == round(one["mean_rank_optimistic"] * n_pos)
        has = np.diff(held.eval_ptr_h) > 0
        assert np.array_equal(ap.cpu().numpy()[has], one["ap"][has])
        assert torch.equal(ranks[torch.as_tensor(held.order, device=DEV)], one["ranks"])
        # F1: every shard's pass adds to the same counters before each finish
        for threshold, want in ((None, f_one), (t, f_at)):
            ws = torch.zeros(int(lib.lec_recon_workspace_bytes(metrics.RECON_OPEN_BINS)), dtype=torch.uint8, device=DEV)
            out = torch.empty(7, dtype=torch.float64, device=DEV)
            status = torch.zeros(4, dtype=torch.int64, device=DEV)
            rs = [metrics.recon_args(rows, cov.tin, cov.tout, geom, KS[geom], 10, a, b, ws)
                  for a, b in zip(cuts[:-1], cuts[1:])]
            for _ in range(64):
                for r in rs:
                    _native.check(lib.lec_recon_pass_heldout(ctypes.byref(r), None if cov.x is None else ctypes.byref(cov.x),
                                                             ctypes.byref(held.h), _native.stream_ptr(DEV)), "pass")
                if threshold is None:
                    _native.check(lib.lec_recon_finish(ctypes.byref(rs[0]), _native._p(out), _native._p(status),
                                                       _native.stream_ptr(DEV)), "finish")
                else:
                    _native.check(lib.lec_recon_finish_at(ctypes.byref(rs[0]), threshold, _native._p(out),
                                                          _native._p(status), _native.stream_ptr(DEV)), "finish_at")
                if int(status[0]) == 0:
                    break
            got = out.cpu().numpy()
            if threshold is not None:
                got[1] = threshold
            assert same(got, want), (got, want)


@pytest.mark.parametrize("kind", ["tree", "dag"])
def test_cfg4_scale(kind):
    h = hierarchy.random_tree(82115, 1.0831) if kind == "tree" else hierarchy.random_dag(82115, 1.0831, 0.02)
    rows = drawn_rows(h, "hyp", 50)
    s = hierarchy.split_edges(h, val=0.05, test=0.05)
    test = s["test"]
    got = metrics.link_prediction_ranks(rows, h, test, "hyp", KS["hyp"], return_ranks=True)
    r = got["ranks"].cpu().numpy()
    assert np.all(r[:, 0] >= 1) and np.all(r[:, 0] <= r[:, 1]) and np.all(r[:, 1] <= h.n - h.n_desc[test[:, 0]])
    assert 0.0 <= got["map"] <= 1.0 and 1.0 <= got["mean_rank_optimistic"] <= got["mean_rank"]
    has = np.unique(test[:, 0])
    sample = np.r_[has[np.argsort(h.n_desc[has])[-8:]], np.random.default_rng(1).choice(has, 248, replace=False)]
    check_ranks(rows, h, "hyp", test, sample=sample, got=got)
    stats = {}
    best = metrics.link_prediction_f1(rows, h, test, "hyp", KS["hyp"], stats=stats)
    assert stats["n_pos"] == len(test) and stats["n_neg"] == h.n * (h.n - 1) - len(h.closure_edges())
    at = metrics.link_prediction_f1(rows, h, test, "hyp", KS["hyp"], threshold=float(best[1]))
    assert at[5] == best[5] and at[6] == best[6]
