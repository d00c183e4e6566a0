"""Link prediction on held-out closure edges without a device: Hierarchy / DagHierarchy.heldout_slots against
rank_slots, hierarchy.split_edges, the dense reference of the contract (link_prediction_oracle, which the GPU tests
compare against) checked against brute-force counting and sklearn, and the argument codes of the new C entry points."""
import ctypes

import numpy as np
import pytest

from learning_embeddings_b200 import _native, hierarchy
from test_reconstruction_ranks_cpu import rank_keys, reconstruction_ranks_oracle, tied_case


def link_prediction_oracle(S, below, held, apex=None):
    """Dense restatement of the contract.  S [m, n] fp32: S[i, v] = E(x = rows[apex[i]], y = rows[v]); below [m, n]
    bool: v strictly below apex[i] in the full closure; held [m, n] bool (a subset of below): the held-out pairs.
    Positives are the held-out pairs, negatives every other v != apex[i] that is not below apex[i]; the other pairs
    below are skipped.  Returns reconstruction_ranks_oracle's (ranks of the held-out pairs in row-major order, ap)."""
    S = np.asarray(S, dtype=np.float32)
    m, n = S.shape
    apex = np.arange(m) if apex is None else np.asarray(apex)
    assert not np.any(held & ~below)
    key = rank_keys(S)
    ranks, ap = [], np.full(m, np.nan)
    for i in range(m):
        neg = ~below[i]
        neg[apex[i]] = False
        pk = key[i, held[i]]
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


def brute_force(S, below, held):
    n = S.shape[0]
    key = rank_keys(S)
    out = []
    for u in range(n):
        for v in range(n):
            if not held[u, v]:
                continue
            neg = [key[u, w] for w in range(n) if w != u and not below[u, w]]
            out.append((1 + sum(k < key[u, v] for k in neg), 1 + sum(k <= key[u, v] for k in neg)))
    return np.array(out, dtype=np.int64).reshape(-1, 2)


def held_case(seed):
    S, below = tied_case(seed)
    rng = np.random.default_rng(seed + 100)
    held = below & (rng.random(below.shape) < 0.5)
    held[2] = below[2]                 # an apex with every pair below it held out
    held[3] = False                    # and one with none
    return S, below, held


@pytest.mark.parametrize("seed", range(5))
def test_oracle_matches_brute_force(seed):
    S, below, held = held_case(seed)
    ranks, ap = link_prediction_oracle(S, below, held)
    assert np.array_equal(ranks, brute_force(S, below, held))
    assert np.isnan(ap[3]) and np.isnan(ap[1])
    # every pair below held out: the reconstruction contract
    r_all, ap_all = link_prediction_oracle(S, below, below)
    r_rec, ap_rec = reconstruction_ranks_oracle(S, below)
    assert np.array_equal(r_all, r_rec) and np.array_equal(ap_all, ap_rec, equal_nan=True)


@pytest.mark.parametrize("seed", range(5))
def test_oracle_ap_matches_sklearn_without_skipped_pairs(seed):
    sk = pytest.importorskip("sklearn.metrics")
    S, below, held = held_case(seed)
    _, ap = link_prediction_oracle(S, below, held)
    n = S.shape[0]
    for u in range(n):
        if not held[u].any():
            continue
        keep = (np.arange(n) != u) & (held[u] | ~below[u])      # skipped pairs removed
        want = sk.average_precision_score(held[u, keep], -S[u, keep].astype(np.float64))
        assert abs(ap[u] - want) <= 1e-12 * max(1.0, want), (u, ap[u], want)


GRAPHS = {"ethec": hierarchy.ethec, "tree4000": lambda: hierarchy.random_tree(4000, 1.0831),
          "dag4000": lambda: hierarchy.random_dag(4000, 1.0831, 0.05)}


@pytest.mark.parametrize("name", list(GRAPHS))
def test_heldout_slots_against_rank_slots(name):
    h = GRAPHS[name]()
    pos_ptr, slot = h.rank_slots()
    e = h.closure_edges()
    # the full closure: the closure layout itself
    eval_ptr, slot_map, order, xcum = h.heldout_slots(e)
    assert eval_ptr.dtype == np.int64 and slot_map.dtype == np.int32 and order.dtype == np.int64
    assert np.array_equal(eval_ptr, pos_ptr) and np.array_equal(slot_map, np.arange(len(e)))
    assert np.array_equal(order, slot)
    # a shuffled subset
    rng = np.random.default_rng(0)
    pick = rng.permutation(len(e))[: len(e) // 4]
    eval_ptr, slot_map, order, xcum = h.heldout_slots(e[pick])
    assert eval_ptr[0] == 0 and eval_ptr[-1] == len(pick)
    assert np.array_equal(np.diff(eval_ptr), np.bincount(e[pick, 0], minlength=h.n))
    assert np.array_equal(np.sort(order), np.arange(len(pick)))
    assert np.array_equal(slot_map[slot[pick]], order)
    assert np.count_nonzero(slot_map >= 0) == len(pick)
    kept = np.flatnonzero(slot_map >= 0)
    assert np.array_equal(slot_map[kept], np.arange(len(pick)))     # closure-slot order is kept
    assert np.all((order >= eval_ptr[e[pick, 0]]) & (order < eval_ptr[e[pick, 0] + 1]))
    if name == "dag4000":   # xcum: the closure slots of the apex before each extra interval
        assert xcum.dtype == np.int32 and len(xcum) == h.extra_ptr[-1]
        for u in np.flatnonzero(np.diff(h.extra_ptr))[:200]:
            size = h.extra_hi[h.extra_ptr[u]:h.extra_ptr[u + 1]] - h.extra_lo[h.extra_ptr[u]:h.extra_ptr[u + 1]] + 1
            want = h.tout[u] - h.tin[u] + np.r_[0, np.cumsum(size)[:-1]]
            assert np.array_equal(xcum[h.extra_ptr[u]:h.extra_ptr[u + 1]], want)
    else:
        assert xcum is None


def test_heldout_slots_rejects_bad_edges():
    h = hierarchy.ethec()
    e = h.closure_edges()
    with pytest.raises(ValueError, match="outside"):
        h.heldout_slots(np.r_[e[:3], [[0, h.n]]])
    with pytest.raises(ValueError, match="outside"):
        h.heldout_slots([[-1, 5]])
    with pytest.raises(ValueError, match="not a closure edge"):
        h.heldout_slots(np.r_[e[:3], e[:1, ::-1]])
    with pytest.raises(ValueError, match="twice"):
        h.heldout_slots(np.r_[e[:3], e[1:2]])
    d = hierarchy.random_dag(500, 1.0831, 0.1)
    with pytest.raises(ValueError, match="not a closure edge"):
        d.heldout_slots([[1, 0]])
    eval_ptr, slot_map, order, _ = h.heldout_slots(np.zeros((0, 2), dtype=np.int64))
    assert eval_ptr[-1] == 0 and np.all(slot_map == -1) and order.shape == (0,)


def transitive_reduction(h):
    e = h.closure_edges()
    A = np.zeros((h.n, h.n), dtype=bool)
    A[e[:, 0], e[:, 1]] = True
    two = (A.astype(np.int32) @ A.astype(np.int32)) > 0
    return e[~two[e[:, 0], e[:, 1]]]


def keys(e, n):
    return set((np.asarray(e)[:, 0] * n + np.asarray(e)[:, 1]).tolist())


@pytest.mark.parametrize("name", ["ethec", "tree600", "dag600"])
def test_split_edges(name):
    h = {"ethec": hierarchy.ethec, "tree600": lambda: hierarchy.random_tree(600, 1.0831, seed=2),
         "dag600": lambda: hierarchy.random_dag(600, 1.0831, 0.1, seed=2)}[name]()
    n = h.n
    closure = keys(h.closure_edges(), n)
    basic = keys(transitive_reduction(h), n)
    if isinstance(h, hierarchy.Hierarchy):
        par = np.flatnonzero(h.parents >= 0)
        assert basic == keys(np.stack([h.parents[par], par], 1), n)
    n_nb = len(closure) - len(basic)
    for frac in (0.05, 0.25):
        s = hierarchy.split_edges(h, val=frac, test=frac, train_nonbasic=0.5, seed=3)
        tr, va, te = (keys(s[k], n) for k in ("train", "val", "test"))
        assert all(s[k].dtype == np.int64 and s[k].shape[1] == 2 for k in s)
        assert len(tr) == len(s["train"]) and len(va) == len(s["val"]) and len(te) == len(s["test"])
        assert basic <= tr and not (tr & va) and not (tr & te) and not (va & te)
        assert (tr | va | te) <= closure
        assert len(va) == int(frac * n_nb) and len(te) == int(frac * n_nb)
        assert len(tr) == len(basic) + min(int(0.5 * n_nb), n_nb - 2 * int(frac * n_nb))
        again = hierarchy.split_edges(h, val=frac, test=frac, train_nonbasic=0.5, seed=3)
        assert all(np.array_equal(s[k], again[k]) for k in s)
        other = hierarchy.split_edges(h, val=frac, test=frac, train_nonbasic=0.5, seed=4)
        assert not np.array_equal(s["test"], other["test"])
    full = hierarchy.split_edges(h)
    assert keys(full["train"], n) | keys(full["val"], n) | keys(full["test"], n) == closure


def test_split_edges_ethec_counts():
    s = hierarchy.split_edges(hierarchy.ethec(), train_nonbasic=0.9)
    assert (len(s["train"]), len(s["val"]), len(s["test"])) == (1848, 62, 62)


def test_argument_validation_codes():
    lib = _native.lib()
    fake = 0x1000
    null = ctypes.c_void_p(0)
    out = ctypes.c_void_p(fake)

    def held(**kw):
        h = _native.LecHeldout(fake, fake, fake, 100)
        for k, v in kw.items():
            setattr(h, k, v)
        return h

    # lec_rank_run_heldout
    def rank_args(**kw):
        r = _native.LecRank()
        r.geom, r.K, r.rows, r.n, r.D, r.ld = 1, 0.1, fake, 10, 4, 4
        r.tin, r.tout, r.pos_ptr, r.n_pos, r.u_begin, r.u_end = fake, fake, fake, 9, 0, 10
        r.workspace, r.workspace_bytes = fake, 1 << 20
        for k, v in kw.items():
            setattr(r, k, v)
        return r

    def rank(r, h):
        return lib.lec_rank_run_heldout(ctypes.byref(r), None if h is None else ctypes.byref(h), out, out, null, null)

    assert lib.lec_rank_run_heldout(None, ctypes.byref(held()), out, out, null, null) == -1
    assert rank(rank_args(rows=0), held()) == -1
    assert rank(rank_args(D=0), held()) == -2
    assert rank(rank_args(geom=7), held()) == -3
    assert rank(rank_args(u_end=11), held()) == -4
    assert rank(rank_args(rows=0x1004), held()) == -5
    assert rank(rank_args(), held(closure_ptr=0)) == -1
    assert rank(rank_args(), held(slot_map=0)) == -1
    assert rank(rank_args(), held(n_closure=-1)) == -4
    assert rank(rank_args(), held(n_closure=1 << 31)) == -4
    assert rank(rank_args(n_pos=101), held()) == -4                     # more held-out pairs than closure pairs
    x = _native.LecReconExtra(fake, fake, fake, 3)
    assert rank(rank_args(extra=ctypes.pointer(x)), held(xcum=0)) == -1
    x = _native.LecReconExtra(fake, fake, fake, 50)   # more extra intervals than held-out pairs is fine, so the
    assert rank(rank_args(extra=ctypes.pointer(x), u_end=11), held()) == -4    # range is what fails here
    assert rank(rank_args(extra=ctypes.pointer(x), u_end=11), None) == -4
    x = _native.LecReconExtra(fake, fake, fake, 101)
    assert rank(rank_args(extra=ctypes.pointer(x)), held()) == -4
    x = _native.LecReconExtra(fake, fake, fake, 10)
    assert rank(rank_args(extra=ctypes.pointer(x)), None) == -4                  # without h the bound is n_pos

    # lec_recon_pass_heldout and lec_recon_finish_at
    nb = int(lib.lec_recon_workspace_bytes(1))

    def recon_args(**kw):
        r = _native.LecRecon()
        r.geom, r.K, r.rows, r.n, r.D, r.ld = 1, 0.1, fake, 10, 4, 4
        r.tin, r.tout, r.u_begin, r.u_end = fake, fake, 0, 10
        r.workspace, r.workspace_bytes = fake, nb
        for k, v in kw.items():
            setattr(r, k, v)
        return r

    def pass_(r, h, x=None):
        return lib.lec_recon_pass_heldout(ctypes.byref(r), None if x is None else ctypes.byref(x),
                                          None if h is None else ctypes.byref(h), null)

    assert lib.lec_recon_pass_heldout(None, None, ctypes.byref(held()), null) == -1
    assert pass_(recon_args(workspace=0), held()) == -1
    assert pass_(recon_args(D=65, ld=68), held()) == -2
    assert pass_(recon_args(geom=9), held()) == -3
    assert pass_(recon_args(workspace_bytes=nb - 1), held()) == -4
    assert pass_(recon_args(workspace=0x1008), held()) == -5
    assert pass_(recon_args(), held(closure_ptr=0)) == -1
    assert pass_(recon_args(), held(slot_map=0)) == -1
    assert pass_(recon_args(), held(n_closure=-5)) == -4
    x = _native.LecReconExtra(fake, fake, fake, 3)
    assert pass_(recon_args(), held(xcum=0), x) == -1
    x = _native.LecReconExtra(fake, fake, fake, 101)
    assert pass_(recon_args(), held(), x) == -4
    x = _native.LecReconExtra(0, fake, fake, 3)
    assert pass_(recon_args(), held(), x) == -1
    # an empty apex range launches nothing: valid arguments return 0, with or without a held-out set
    assert pass_(recon_args(u_begin=4, u_end=4), held()) == 0
    assert pass_(recon_args(u_begin=4, u_end=4), None) == 0
    assert pass_(recon_args(u_begin=4, u_end=4), held(xcum=0)) == 0              # a forest needs no xcum

    def fin(r, o=out, s=out):
        return lib.lec_recon_finish_at(ctypes.byref(r), 0.5, o, s, null)

    assert lib.lec_recon_finish_at(None, 0.5, out, out, null) == -1
    assert fin(recon_args(), o=null) == -1
    assert fin(recon_args(), s=null) == -1
    assert fin(recon_args(D=0)) == -2
    assert fin(recon_args(geom=-1)) == -3
    assert fin(recon_args(u_begin=3, u_end=2)) == -4
    assert fin(recon_args(rows=0x1004)) == -5
