"""Reconstruction mean rank and MAP without a device: the dense reference of lec_rank_run's contract
(reconstruction_ranks_oracle, which the GPU tests compare against) checked against brute-force counting and sklearn,
its key rules (NaN, -0), the positive-slot layout of Hierarchy and DagHierarchy, and the C ABI's argument codes."""
import ctypes

import numpy as np
import pytest

from learning_embeddings_b200 import _native, hierarchy
from test_reconstruction_dag_gpu import wide_apex_dag


def rank_keys(S):
    """key of an fp32 energy: its bits, -0 as 0, every NaN one value after +inf (energies are >= 0 or NaN)"""
    S = np.asarray(S, dtype=np.float32)
    b = S.view(np.uint32).astype(np.int64)
    return np.where(np.isnan(S), 0x7FC00000, np.where(b == 0x80000000, 0, b))


def reconstruction_ranks_oracle(S, pos_mask, apex=None):
    """Dense restatement of the contract.  S [m, n] fp32: S[i, v] = E(x = rows[apex[i]], y = rows[v]); pos_mask [m, n]
    bool: v strictly below apex[i]; apex: the node of each row (default 0..m-1), whose own pair is skipped.
    Returns ranks int64 [n_edges, 2] (rank_opt, rank_pess) of the positives in row-major order and ap fp64 [m] (NaN for a
    row without positives): per apex, the negatives are every other v that is not positive."""
    S = np.asarray(S, dtype=np.float32)
    m, n = S.shape
    apex = np.arange(m) if apex is None else np.asarray(apex)
    key = rank_keys(S)
    ranks, ap = [], np.full(m, np.nan)
    for i in range(m):
        neg = ~pos_mask[i]
        neg[apex[i]] = False
        pk = key[i, pos_mask[i]]
        if len(pk) == 0:
            continue
        nk = np.sort(key[i, neg])
        ranks.append(np.stack([1 + np.searchsorted(nk, pk, "left"), 1 + np.searchsorted(nk, pk, "right")], 1))
        ps = np.sort(pk)
        t, c = np.unique(ps, return_counts=True)
        tp = np.searchsorted(ps, t, "right")
        fp = np.searchsorted(nk, t, "right")
        ap[i] = float(np.sum(c * (tp / (tp + fp)))) / len(pk)
    return (np.concatenate(ranks) if ranks else np.zeros((0, 2), dtype=np.int64)), ap


def brute_force(S, pos_mask):
    n = S.shape[0]
    key = rank_keys(S)
    out = []
    for u in range(n):
        for v in range(n):
            if not pos_mask[u, v]:
                continue
            neg = [key[u, w] for w in range(n) if w != u and not pos_mask[u, w]]
            out.append((1 + sum(k < key[u, v] for k in neg), 1 + sum(k <= key[u, v] for k in neg)))
    return np.array(out, dtype=np.int64).reshape(-1, 2)


def tied_case(seed, n=24):
    rng = np.random.default_rng(seed)
    S = rng.integers(0, 5, size=(n, n)).astype(np.float32) * np.float32(0.25)   # five values: ties of both signs
    pos = rng.random((n, n)) < 0.3
    np.fill_diagonal(pos, False)
    pos[0] = True                         # apex 0: every other node is a positive, so it has no negative
    pos[0, 0] = False
    pos[1] = False                        # a node without positives
    return S, pos


@pytest.mark.parametrize("seed", range(5))
def test_oracle_ranks_match_brute_force(seed):
    S, pos = tied_case(seed)
    ranks, ap = reconstruction_ranks_oracle(S, pos)
    assert np.array_equal(ranks, brute_force(S, pos))
    assert np.all(ranks[:, 0] <= ranks[:, 1])
    assert np.isnan(ap[1])
    assert ap[0] == 1.0 and np.all(ranks[: pos[0].sum()] == 1)   # no negatives: AP 1, every rank 1


@pytest.mark.parametrize("seed", range(5))
def test_oracle_ap_matches_sklearn(seed):
    sk = pytest.importorskip("sklearn.metrics")
    S, pos = tied_case(seed)
    _, ap = reconstruction_ranks_oracle(S, pos)
    n = S.shape[0]
    for u in range(n):
        if not pos[u].any():
            continue
        keep = np.arange(n) != u
        want = sk.average_precision_score(pos[u, keep], -S[u, keep].astype(np.float64))
        assert abs(ap[u] - want) <= 1e-12 * max(1.0, want), (u, ap[u], want)


def test_nan_and_negative_zero_keys():
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    # apex 0: positives {1: -0, 2: NaN}; negatives {3: +0, 4: inf, 5: NaN (another bit pattern), 6: 1}
    S = np.zeros((7, 7), dtype=np.float32)
    S[0, 1:] = [-0.0, nan, 0.0, inf, np.float32(-nan), 1.0]
    pos = np.zeros((7, 7), dtype=bool)
    pos[0, [1, 2]] = True
    k = rank_keys(S[0])
    assert k[1] == k[3] == 0 and k[2] == k[5] == 0x7FC00000 > k[4]
    ranks, ap = reconstruction_ranks_oracle(S, pos)
    # -0 ties +0: opt 1, pess 2.  NaN is above 0, 1 and inf and ties the negative NaN: opt 4, pess 5
    assert ranks.tolist() == [[1, 2], [4, 5]]
    # AP: t = 0: TP 1, FP 1 -> 1/2 * 1/2;  t = NaN: TP 2, FP 4 -> 1/2 * 2/6
    assert abs(ap[0] - (0.25 + 1.0 / 6.0)) < 1e-15


def cover_order(h, u):
    """v's in slot order under u, from the cover directly"""
    tin = np.asarray(h.tin)
    node_at = np.argsort(tin)
    runs = [(tin[u] + 1, h.tout[u])]
    if hasattr(h, "extra_ptr"):
        runs += list(zip(h.extra_lo[h.extra_ptr[u]:h.extra_ptr[u + 1]], h.extra_hi[h.extra_ptr[u]:h.extra_ptr[u + 1]]))
    return np.concatenate([node_at[lo:hi + 1] for lo, hi in runs]) if runs else np.zeros(0, dtype=np.int64)


@pytest.mark.parametrize("name", ["ethec", "tree4000", "dag4000", "wide_apex"])
def test_slot_layout(name):
    h = {"ethec": hierarchy.ethec, "tree4000": lambda: hierarchy.random_tree(4000, 1.0831),
         "dag4000": lambda: hierarchy.random_dag(4000, 1.0831, 0.05), "wide_apex": wide_apex_dag}[name]()
    pos_ptr, slot = h.rank_slots()
    e = h.closure_edges()
    assert pos_ptr.dtype == np.int64 and pos_ptr[0] == 0 and pos_ptr[-1] == len(e)
    assert np.array_equal(np.diff(pos_ptr), h.n_desc)
    assert np.array_equal(np.sort(slot), np.arange(len(e)))        # a permutation
    assert np.all((slot >= pos_ptr[e[:, 0]]) & (slot < pos_ptr[e[:, 0] + 1]))
    inside = (h.tin[e[:, 1]] > h.tin[e[:, 0]]) & (h.tin[e[:, 1]] <= h.tout[e[:, 0]])
    assert np.array_equal(slot[inside], pos_ptr[e[inside, 0]] + h.tin[e[inside, 1]] - h.tin[e[inside, 0]] - 1)
    v_at = np.empty(len(e), dtype=np.int64)
    v_at[slot] = e[:, 1]
    apexes = np.flatnonzero(h.n_desc)
    if hasattr(h, "extra_ptr"):   # every apex with extra intervals, plus the largest ones
        apexes = np.union1d(np.flatnonzero(np.diff(h.extra_ptr)), np.argsort(h.n_desc)[-8:])
    for u in apexes[:400]:
        assert np.array_equal(v_at[pos_ptr[u]:pos_ptr[u + 1]], cover_order(h, u)), u
    if name == "wide_apex":
        assert int(np.diff(h.extra_ptr).max()) > 1000


def test_argument_validation_codes():
    lib = _native.lib()
    assert lib.lec_rank_workspace_bytes(-1, 0) == -4
    assert lib.lec_rank_workspace_bytes(10, 1 << 31) == -4
    fake = 0x1000
    sums, ap = ctypes.c_void_p(fake), ctypes.c_void_p(fake)
    null = ctypes.c_void_p(0)

    def args(**kw):
        r = _native.LecRank()
        r.geom, r.K, r.rows, r.n, r.D, r.ld = 1, 0.1, fake, 10, 4, 4
        r.tin, r.tout, r.pos_ptr, r.n_pos, r.u_begin, r.u_end = fake, fake, fake, 9, 0, 10
        r.workspace, r.workspace_bytes = fake, 1 << 20
        for k, v in kw.items():
            setattr(r, k, v)
        return r

    def run(r, s=sums, a=ap):
        return lib.lec_rank_run(ctypes.byref(r), s, a, null, null)

    assert lib.lec_rank_run(None, sums, ap, null, null) == -1
    assert run(args(rows=0)) == -1
    assert run(args(pos_ptr=0)) == -1
    assert run(args(workspace=0)) == -1
    assert run(args(), s=null) == -1
    assert run(args(), a=null) == -1
    assert run(args(D=0)) == -2
    assert run(args(D=65, ld=68)) == -2
    assert run(args(ld=6)) == -2
    assert run(args(geom=7)) == -3
    assert run(args(u_end=11)) == -4
    assert run(args(u_begin=5, u_end=4)) == -4
    assert run(args(n_pos=-1)) == -4
    assert run(args(n_pos=1 << 31)) == -4
    x = _native.LecReconExtra(0, fake, fake, 3)
    assert run(args(extra=ctypes.pointer(x))) == -1
    x = _native.LecReconExtra(fake, fake, fake, 10)
    assert run(args(extra=ctypes.pointer(x))) == -4                # more extra intervals than positives
    assert run(args(rows=0x1004)) == -5
    assert run(args(workspace=0x1008)) == -5


def test_slot_layout_without_edges():
    pos_ptr, slot = hierarchy.Hierarchy(np.full(50, -1)).rank_slots()
    assert np.array_equal(pos_ptr, np.zeros(51)) and slot.shape == (0,)
