"""Reconstruction F1 (lec_recon_*): the C ABI's argument checks, Hierarchy.from_closure_edges and the oracle's pair
split, without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from learning_embeddings_b200 import _native, hierarchy
from oracle import cones

FAKE = 0x1000   # 16-byte aligned, never dereferenced: validation fails first


def reconstruction_pairs(h):
    """Every ordered pair u != v of the hierarchy's nodes (int64 tensors, row-major) and whether v is a strict
    descendant of u: the closure edges of check_graph_embedding (order_embeddings.py:519-531)."""
    u, v = np.nonzero(~np.eye(h.n, dtype=bool))
    pos = torch.from_numpy(h.is_descendant(u, v))
    return torch.from_numpy(u), torch.from_numpy(v), pos


def reconstruction_f1(emb, h, geom, K):
    """Oracle restatement of check_graph_embedding (order_embeddings.py:512-559): dense pair lists, the oracle's
    energy in emb's dtype, then its best_f1_sweep.  O(n^2) memory."""
    u, v, pos = reconstruction_pairs(h)
    step = 1 << 20
    E = torch.cat([cones.energy(geom, emb[u[s:s + step]], emb[v[s:s + step]], K) for s in range(0, len(u), step)])
    return cones.best_f1_sweep(E[pos], E[~pos])


def recon(**kw):
    r = _native.LecRecon()
    r.geom, r.K, r.rows, r.n, r.D, r.ld = 1, 0.1, FAKE, 100, 10, 12
    r.tin, r.tout, r.u_begin, r.u_end = FAKE, FAKE, 0, 100
    r.workspace, r.workspace_bytes = FAKE, _native.lib().lec_recon_workspace_bytes(1)
    for k, v in kw.items():
        setattr(r, k, v)
    return r


def test_exports_and_workspace_sizes():
    lib = _native.lib()
    for name in ("lec_recon_workspace_bytes", "lec_recon_counter_bytes", "lec_recon_pass", "lec_recon_finish"):
        assert name in _native.EXPORTS and hasattr(lib, name)
    one, two = lib.lec_recon_workspace_bytes(1), lib.lec_recon_workspace_bytes(2)
    assert 0 < one < two and two - one >= 2 * 65536 * 8     # a fine round counts 65 536 keys x 2 signs per open bin
    assert lib.lec_recon_workspace_bytes(0) == -4
    assert lib.lec_recon_counter_bytes(one - 1) == -4
    assert 0 < lib.lec_recon_counter_bytes(one) < lib.lec_recon_counter_bytes(two) < two
    assert lib.lec_recon_counter_bytes(two) % 8 == 0
    assert lib.lec_recon_workspace_bytes(128) < 256 << 20   # the default of metrics.reconstruction_f1


@pytest.mark.parametrize("fields, code", [
    (dict(rows=0), -1), (dict(tin=0), -1), (dict(tout=0), -1), (dict(workspace=0), -1),
    (dict(D=0), -2), (dict(D=65, ld=68), -2), (dict(ld=8), -2), (dict(ld=14), -2),
    (dict(geom=3), -3), (dict(geom=-1), -3),
    (dict(n=-1, u_end=0), -4), (dict(u_begin=-1), -4), (dict(u_end=101), -4), (dict(u_begin=60, u_end=50), -4),
    (dict(workspace_bytes=1024), -4),
    (dict(rows=0x1004), -5), (dict(workspace=0x1008), -5),
])
def test_argument_validation_codes(fields, code):
    lib = _native.lib()
    null = ctypes.c_void_p(0)
    r = recon(**fields)
    assert lib.lec_recon_pass(ctypes.byref(r), null) == code
    assert lib.lec_recon_finish(ctypes.byref(r), ctypes.c_void_p(FAKE), ctypes.c_void_p(FAKE), null) == code


def test_argument_validation_edges():
    lib = _native.lib()
    null = ctypes.c_void_p(0)
    assert lib.lec_recon_pass(None, null) == -1
    assert lib.lec_recon_finish(ctypes.byref(recon()), null, ctypes.c_void_p(FAKE), null) == -1
    assert lib.lec_recon_finish(ctypes.byref(recon()), ctypes.c_void_p(FAKE), null, null) == -1
    # an empty apex range is a no-op success; ld == D is accepted for any D (a plain [n, D] table)
    assert lib.lec_recon_pass(ctypes.byref(recon(u_begin=40, u_end=40)), null) == 0
    assert lib.lec_recon_pass(ctypes.byref(recon(D=10, ld=10, u_begin=0, u_end=0)), null) == 0


@pytest.mark.parametrize("make", [hierarchy.ethec, lambda: hierarchy.random_tree(2000, 1.0831)], ids=["ethec", "random_tree"])
def test_from_closure_edges_round_trip(make):
    h = make()
    e = h.closure_edges()
    rng = np.random.default_rng(0)
    g = hierarchy.Hierarchy.from_closure_edges(h.n, e[rng.permutation(len(e))])   # any edge order
    assert np.array_equal(g.parents, h.parents)
    assert np.array_equal(g.tin, h.tin) and np.array_equal(g.tout, h.tout)


def test_from_closure_edges_rejects_non_forests():
    # diamond 0 -> {1, 2} -> 3
    with pytest.raises(ValueError):
        hierarchy.Hierarchy.from_closure_edges(4, [(0, 1), (0, 2), (1, 3), (2, 3), (0, 3)])
    with pytest.raises(ValueError):   # a transitive edge missing
        hierarchy.Hierarchy.from_closure_edges(3, [(0, 1), (1, 2)])
    with pytest.raises(ValueError):   # a cycle
        hierarchy.Hierarchy.from_closure_edges(2, [(0, 1), (1, 0)])
    with pytest.raises(ValueError):
        hierarchy.Hierarchy.from_closure_edges(2, [(0, 2)])
    g = hierarchy.Hierarchy.from_closure_edges(5, np.zeros((0, 2), dtype=np.int64))
    assert np.array_equal(g.parents, np.full(5, -1))


def test_oracle_pair_split_ethec():
    h = hierarchy.ethec()
    u, v, pos = reconstruction_pairs(h)
    assert int(pos.sum()) == 1974 and int((~pos).sum()) == 520032
    assert not bool((u == v).any())
    e = h.closure_edges()
    assert set(zip(u[pos].tolist(), v[pos].tolist())) == set(map(tuple, e.tolist()))


def test_oracle_reconstruction_row_ethec():
    # fp64 rows on the shell: a finite best row whose counts are consistent with the pair split
    h = hierarchy.ethec()
    g = torch.Generator().manual_seed(0)
    w = torch.randn(h.n, 10, generator=g, dtype=torch.float64)
    emb = (cones.inner_radius(0.1) + 0.05 * torch.rand(h.n, 1, generator=g, dtype=torch.float64)) * w / w.norm(dim=1, keepdim=True)
    f1, t, acc, prec, rec, cp, cn = reconstruction_f1(emb, h, "hyp", 0.1)
    assert 0.0 < f1 <= 1.0 and 0 < cp <= 1974 and 0 <= cn <= 520032
    assert rec == cp / 1974 and acc == (cp + cn) / (1974 + 520032)
