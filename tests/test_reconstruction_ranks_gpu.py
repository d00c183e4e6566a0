"""Reconstruction mean rank and MAP on the GPU (metrics.reconstruction_ranks / lec_rank_run) against the materialised
path: the SIMT score matrix (or its rows for sampled apexes) and the dense reference of the contract.  Exact means ranks
equal as integers and AP per apex and MAP within 1e-12 relative."""
import ctypes
import functools
import math

import numpy as np
import pytest
import torch

from learning_embeddings_b200 import _native, hierarchy, metrics, ops
from test_reconstruction_dag_gpu import dag
from test_reconstruction_gpu import KS, drawn_rows, trained_rows, tree
from test_reconstruction_ranks_cpu import reconstruction_ranks_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@functools.lru_cache(maxsize=None)
def graph(name):
    return dag(name) if name in ("dag4000", "wide_apex") else tree(name)


def check_exact(rows, h, geom, D=None, sample=None, got=None):
    """rows of the score matrix for `sample` (every apex by default) and the oracle against reconstruction_ranks"""
    if got is None:
        got = metrics.reconstruction_ranks(rows, h, geom, KS[geom], D=D, return_ranks=True)
    x = rows if D is None else rows[:, :D].contiguous()
    n = h.n
    sample = np.arange(n) if sample is None else np.unique(sample)
    S = torch.empty((len(sample), n), device=DEV, dtype=torch.float32)
    ops.score_topk_into(x[torch.as_tensor(sample, device=DEV)].contiguous(), x, geom, KS[geom], [], [], 1, None, None, S,
                        1, engine="simt")
    pos = h.is_descendant(sample[:, None], np.arange(n)[None, :])
    ranks, ap = reconstruction_ranks_oracle(S.cpu().numpy(), pos, apex=sample)
    e = h.closure_edges()
    sel = np.isin(e[:, 0], sample)
    assert got["n_edges"] == len(e) and got["n_apexes"] == int(np.count_nonzero(h.n_desc))
    assert np.array_equal(got["ranks"].cpu().numpy()[sel], ranks)
    has = h.n_desc[sample] > 0
    assert np.all(np.isnan(got["ap"][sample][~has]))
    np.testing.assert_allclose(got["ap"][sample][has], ap[has], rtol=1e-12, atol=0)
    if len(sample) == n:
        assert got["mean_rank"] == ranks[:, 1].sum() / len(e)
        assert got["mean_rank_optimistic"] == ranks[:, 0].sum() / len(e)
        want = math.fsum(ap[has].tolist()) / int(has.sum())
        assert abs(got["map"] - want) <= 1e-12 * want, (got["map"], want)
    return got


@pytest.mark.parametrize("name", ["ethec", "tree4000", "dag4000"])
@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_exact_drawn_rows(geom, D, name):
    check_exact(drawn_rows(graph(name), geom, D), graph(name), geom)


@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_exact_trained_padded_rows(geom, D):
    # the engine's padded rows after training: E == 0 ties everywhere
    rows, D = trained_rows("tree4000", geom, D)
    assert rows.shape[1] > D or D % 4 == 0
    got = check_exact(rows, tree("tree4000"), geom, D=D)
    plain = metrics.reconstruction_ranks(rows[:, :D].contiguous(), tree("tree4000"), geom, KS[geom], return_ranks=True)
    assert torch.equal(plain["ranks"], got["ranks"])


@pytest.mark.parametrize("D", [2, 10, 50])
@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_apex_with_many_extra_intervals(geom, D):
    h = graph("wide_apex")
    assert int(np.diff(h.extra_ptr).max()) > 1000
    check_exact(drawn_rows(h, geom, D), h, geom)


@pytest.mark.parametrize("geom", ["euc", "hyp", "oe"])
def test_quantised_rows(geom):
    h = tree("ethec")
    base = drawn_rows(h, geom, 10)
    pick = torch.as_tensor(np.random.default_rng(3).integers(0, 6, size=h.n), device=DEV)
    got = check_exact(base[pick].contiguous(), h, geom)
    assert np.any(got["ranks"][:, 0].cpu().numpy() != got["ranks"][:, 1].cpu().numpy())   # ties with negatives


def test_zero_row_and_identical_rows():
    h = tree("ethec")
    rows = drawn_rows(h, "hyp", 10)
    rows[5] = 0.0                  # NaN apex row
    rows[100] = rows[200]          # their pair is NaN
    check_exact(rows, h, "hyp")


def test_forest_without_edges():
    h = hierarchy.Hierarchy(np.full(500, -1))
    got = metrics.reconstruction_ranks(drawn_rows(h, "hyp", 10), h, "hyp", KS["hyp"], return_ranks=True)
    assert got["n_edges"] == 0 and got["n_apexes"] == 0 and got["ranks"].shape == (0, 2)
    assert all(math.isnan(got[k]) for k in ("mean_rank", "mean_rank_optimistic", "map"))
    assert np.all(np.isnan(got["ap"]))


def test_apex_above_every_other_node():
    h = hierarchy.random_tree(3000, 1.0831, seed=4, roots=1)
    assert h.n_desc[0] == h.n - 1
    got = check_exact(drawn_rows(h, "hyp", 10), h, "hyp")
    e = h.closure_edges()
    assert got["ap"][0] == 1.0 and bool((got["ranks"][torch.as_tensor(e[:, 0] == 0, device=DEV)] == 1).all())


def test_global_counters_of_a_large_apex():
    # node 0 is above 19 000 others: more buckets than one tile's shared memory holds, so it counts in global memory
    big = hierarchy.random_tree(19001, 1.0831, seed=5, roots=1)
    h = hierarchy.Hierarchy(np.r_[big.parents, np.full(999, -1)])
    assert h.n_desc[0] == 19000 > metrics.RANK_SHARED_BUCKETS
    for geom in ("hyp", "euc"):
        rows = drawn_rows(h, geom, 10)
        sample = np.r_[0, np.argsort(h.n_desc)[-8:], np.random.default_rng(0).choice(h.n, 120, replace=False)]
        got = metrics.reconstruction_ranks(rows, h, geom, KS[geom], return_ranks=True)
        check_exact(rows, h, geom, sample=sample, got=got)


def test_apex_shards_add_up_and_calls_are_bit_identical():
    lib = _native.lib()
    for name, geom in (("tree4000", "hyp"), ("dag4000", "euc")):
        h = graph(name)
        rows = drawn_rows(h, geom, 10)
        one = metrics.reconstruction_ranks(rows, h, geom, KS[geom], return_ranks=True)
        two = metrics.reconstruction_ranks(rows, h, geom, KS[geom], return_ranks=True)
        assert np.array_equal(one["ap"], two["ap"], equal_nan=True) and torch.equal(one["ranks"], two["ranks"])
        assert one["map"] == two["map"] and one["mean_rank"] == two["mean_rank"]
        pos_ptr_h, slot = h.rank_slots()
        pos_ptr = torch.as_tensor(pos_ptr_h, device=DEV)
        tin = torch.as_tensor(h.tin, dtype=torch.int32, device=DEV)
        tout = torch.as_tensor(h.tout, dtype=torch.int32, device=DEV)
        x = None
        if hasattr(h, "extra_ptr"):
            xs = [torch.as_tensor(a, dtype=torch.int32, device=DEV) for a in (h.extra_ptr, h.extra_lo, h.extra_hi)]
            x = _native.LecReconExtra(xs[0].data_ptr(), xs[1].data_ptr(), xs[2].data_ptr(), int(h.extra_ptr[-1]))
        n_pos = int(pos_ptr_h[-1])
        nb = int(lib.lec_rank_workspace_bytes(h.n, n_pos))
        total = torch.zeros(3, dtype=torch.int64, device=DEV)
        ap = torch.zeros(h.n, dtype=torch.float64, device=DEV)
        ranks = torch.zeros((n_pos, 2), dtype=torch.int32, device=DEV)
        cuts = [0, 17, 2900, h.n]
        for a, b in zip(cuts[:-1], cuts[1:]):
            ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
            r = metrics.rank_args(rows, tin, tout, x, pos_ptr, n_pos, geom, KS[geom], 10, a, b, ws)
            sums = torch.empty(3, dtype=torch.int64, device=DEV)
            part = torch.zeros(h.n, dtype=torch.float64, device=DEV)
            _native.check(lib.lec_rank_run(ctypes.byref(r), _native._p(sums), _native._p(part), _native._p(ranks),
                                           _native.stream_ptr(DEV)), "lec_rank_run")
            total += sums
            ap += part
        assert int(total[1]) == round(one["mean_rank"] * n_pos) and int(total[0]) == round(one["mean_rank_optimistic"] * n_pos)
        ap = ap.cpu().numpy()
        has = h.n_desc > 0
        assert np.array_equal(ap[has], one["ap"][has])
        assert torch.equal(ranks[torch.as_tensor(slot, device=DEV)], one["ranks"])


@pytest.mark.parametrize("kind", ["tree", "dag"])
def test_cfg4_scale(kind):
    h = hierarchy.random_tree(82115, 1.0831) if kind == "tree" else hierarchy.random_dag(82115, 1.0831, 0.02)
    rows = drawn_rows(h, "hyp", 50)
    stats = {}
    got = metrics.reconstruction_ranks(rows, h, "hyp", KS["hyp"], return_ranks=True, stats=stats)
    assert got["n_edges"] == (741845 if kind == "tree" else 836664)
    e = h.closure_edges()
    r = got["ranks"].cpu().numpy()
    assert np.all(r[:, 0] >= 1) and np.all(r[:, 0] <= r[:, 1]) and np.all(r[:, 1] <= h.n - h.n_desc[e[:, 0]])
    assert 0.0 <= got["map"] <= 1.0
    assert 1.0 <= got["mean_rank_optimistic"] <= got["mean_rank"]
    sample = np.r_[np.argsort(h.n_desc)[-8:], np.random.default_rng(1).choice(np.flatnonzero(h.n_desc), 248, replace=False)]
    check_exact(rows, h, "hyp", sample=sample, got=got)
