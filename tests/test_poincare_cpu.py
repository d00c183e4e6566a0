"""Poincare embeddings (Nickel & Kiela 2017) without a GPU: an fp64 torch reference of the distance, the softmax loss
and the update rule (the GPU tests compare the kernels against it), its closed-form gradient against autograd, and the
argument codes of the new and extended entry points."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from learning_embeddings_b200 import _native

MAX_NORM = 1.0 - 1e-5


# ---- fp64 reference -------------------------------------------------------------------------------------------------
def poincare_distance(x, y):
    """arcosh(1 + delta), delta = 2|x-y|^2 / ((1-|x|^2)(1-|y|^2)), as log1p(delta + sqrt(delta (delta + 2)))."""
    A, B = (x * x).sum(-1), (y * y).sum(-1)
    s = ((x - y) ** 2).sum(-1)
    delta = 2.0 * s / ((1.0 - A) * (1.0 - B))
    return torch.log1p(delta + torch.sqrt(delta * (delta + 2.0)))


def distance_grad(x, y):
    """Closed-form dd/dx, dd/dy (zero where delta = 0)."""
    A, B = (x * x).sum(-1, keepdim=True), (y * y).sum(-1, keepdim=True)
    p = (x * y).sum(-1, keepdim=True)
    s = ((x - y) ** 2).sum(-1, keepdim=True)
    delta = 2.0 * s / ((1.0 - A) * (1.0 - B))
    r = torch.sqrt(delta * (delta + 2.0))
    safe = torch.where(delta > 0, r, torch.ones_like(r))
    gx = 4.0 / ((1.0 - B) * safe) * ((B - 2.0 * p + 1.0) / (1.0 - A) ** 2 * x - y / (1.0 - A))
    gy = 4.0 / ((1.0 - A) * safe) * ((A - 2.0 * p + 1.0) / (1.0 - B) ** 2 * y - x / (1.0 - B))
    zero = delta <= 0
    return torch.where(zero, torch.zeros_like(gx), gx), torch.where(zero, torch.zeros_like(gy), gy)


def poincare_loss_ref(W, u, v, neg):
    """W [n, D] fp64; u, v [B]; neg [B, N].  Returns (loss, E_pos [B], E_neg [B, N], dloss/dW [n, D]), all fp64, the
    gradient from the closed form."""
    W = W.double()
    u, v, neg = (torch.as_tensor(t, dtype=torch.int64) for t in (u, v, neg))
    Bn, Nn = neg.shape
    others = torch.cat([v[:, None], neg], 1)                       # [B, 1 + N]
    X = W[u][:, None, :].expand(Bn, Nn + 1, W.shape[1])
    Y = W[others]
    d = poincare_distance(X, Y)
    lse = torch.logsumexp(-d, 1)
    loss = (d[:, 0] + lse).sum()
    p = torch.softmax(-d, 1)
    c = -p
    c[:, 0] += 1.0
    gx, gy = distance_grad(X, Y)
    G = torch.zeros_like(W)
    G.index_add_(0, u, (c[..., None] * gx).sum(1))
    G.index_add_(0, others.reshape(-1), (c[..., None] * gy).reshape(-1, W.shape[1]))
    return loss, d[:, 0], d[:, 1:], G


def retract_update(W, G, lr):
    """Nickel & Kiela eq. 5-7: w <- proj(w - lr (1 - |w|^2)^2 / 4 g); proj rescales |w| >= 1 - 1e-5 to 1 - 1e-5.
    Returns (new W, rescaled gradient)."""
    W, G = W.double(), G.double()
    rg = (1.0 - (W * W).sum(1, keepdim=True)) ** 2 / 4.0 * G
    out = W - lr * rg
    nrm = out.norm(dim=1, keepdim=True)
    out = torch.where(nrm >= MAX_NORM, out / nrm * MAX_NORM, out)
    return out, rg


def random_ball(n, D, gen, rmax=0.9):
    x = torch.randn(n, D, generator=gen, dtype=torch.float64)
    return x / x.norm(dim=1, keepdim=True) * rmax * torch.rand(n, 1, generator=gen, dtype=torch.float64)


# ---- the reference itself -------------------------------------------------------------------------------------------
def test_distance_properties():
    g = torch.Generator().manual_seed(0)
    x, y = random_ball(50, 7, g), random_ball(50, 7, g)
    d = poincare_distance(x, y)
    assert torch.allclose(d, poincare_distance(y, x), rtol=0, atol=1e-14)
    assert torch.equal(poincare_distance(x, x), torch.zeros(50, dtype=torch.float64))
    # arcosh form
    A, B = (x * x).sum(1), (y * y).sum(1)
    ref = torch.acosh(1 + 2 * ((x - y) ** 2).sum(1) / ((1 - A) * (1 - B)))
    assert torch.allclose(d, ref, rtol=1e-12, atol=1e-12)
    # from the origin: d(0, y) = 2 artanh |y|
    z = torch.zeros_like(y)
    assert torch.allclose(poincare_distance(z, y), 2 * torch.atanh(y.norm(dim=1)), rtol=1e-12)


@pytest.mark.parametrize("case", ["random", "near_coincident", "near_boundary"])
def test_closed_form_gradient_matches_autograd(case):
    g = torch.Generator().manual_seed(1)
    D = 5
    x, y = random_ball(6, D, g), random_ball(6, D, g)
    if case == "near_coincident":
        y = x + 1e-7 * torch.randn(6, D, generator=g, dtype=torch.float64)
    elif case == "near_boundary":
        x = x / x.norm(dim=1, keepdim=True) * (1 - 1e-5)
        y = y / y.norm(dim=1, keepdim=True) * (1 - 3e-5)
    gx, gy = distance_grad(x, y)
    xa, ya = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    poincare_distance(xa, ya).sum().backward()
    torch.testing.assert_close(gx, xa.grad, rtol=1e-6, atol=1e-9)
    torch.testing.assert_close(gy, ya.grad, rtol=1e-6, atol=1e-9)
    if case == "random":
        assert torch.autograd.gradcheck(lambda a, b: poincare_distance(a, b), (xa.detach().requires_grad_(True),
                                                                                 ya.detach().requires_grad_(True)))


def test_gradient_is_zero_at_delta_zero():
    x = torch.tensor([[0.1, -0.2, 0.3]], dtype=torch.float64)
    gx, gy = distance_grad(x, x.clone())
    assert torch.equal(gx, torch.zeros_like(x)) and torch.equal(gy, torch.zeros_like(x))
    W = torch.cat([x, x])
    loss, E_pos, E_neg, G = poincare_loss_ref(W, [0], [1], [[0]])
    assert float(E_pos[0]) == 0.0 and float(E_neg[0, 0]) == 0.0
    assert torch.equal(G, torch.zeros_like(W))
    assert abs(float(loss) - np.log(2.0)) < 1e-15


def test_loss_and_gradient_against_autograd():
    g = torch.Generator().manual_seed(2)
    n, D, Bn, Nn = 30, 4, 12, 6
    W = random_ball(n, D, g)
    u = torch.randint(0, n, (Bn,), generator=g)
    v = torch.randint(0, n, (Bn,), generator=g)
    neg = torch.randint(0, n, (Bn, Nn), generator=g)
    neg[0, :] = neg[0, 0]                                      # a repeated negative counts once per draw
    v = torch.where(v == u, (v + 1) % n, v)                    # autograd's sqrt has no derivative at delta = 0
    neg = torch.where(neg == u[:, None], (neg + 1) % n, neg)
    loss, E_pos, E_neg, G = poincare_loss_ref(W, u, v, neg)

    def f(Wa):
        d_pos = poincare_distance(Wa[u], Wa[v])
        d_all = poincare_distance(Wa[u][:, None, :], Wa[torch.cat([v[:, None], neg], 1)])
        return (d_pos + torch.logsumexp(-d_all, 1)).sum()

    Wa = W.clone().requires_grad_(True)
    la = f(Wa)
    la.backward()
    assert abs(float(loss) - float(la.detach())) <= 1e-12 * abs(float(la.detach()))
    torch.testing.assert_close(G, Wa.grad, rtol=1e-9, atol=1e-12)
    assert torch.autograd.gradcheck(f, (W.clone().requires_grad_(True),))


def test_update_rule_reference():
    g = torch.Generator().manual_seed(3)
    W = random_ball(8, 3, g)
    W[0] = W[0] / W[0].norm() * (1 - 1e-6)            # outside the projection radius already
    G = torch.randn(8, 3, generator=g, dtype=torch.float64)
    out, rg = retract_update(W, G, 0.5)
    torch.testing.assert_close(rg, ((1 - (W * W).sum(1, keepdim=True)) ** 2 / 4) * G)
    assert float(out.norm(dim=1).max()) <= MAX_NORM + 1e-15
    big = W - 0.5 * rg
    keep = big.norm(dim=1) < MAX_NORM
    torch.testing.assert_close(out[keep], big[keep])
    torch.testing.assert_close(out[0].norm(), torch.tensor(MAX_NORM, dtype=torch.float64))


# ---- argument codes -------------------------------------------------------------------------------------------------
def test_poincare_constants():
    assert _native.GEOM["poincare"] == 4 and _native.UPD_RSGD_RETRACT == 4 and _native.ABI_VERSION == 14


def test_argument_validation_codes():
    lib = _native.lib()
    fake = ctypes.c_void_p(0x1000)       # 16-byte aligned, never dereferenced: validation fails first
    odd = ctypes.c_void_p(0x1004)
    null = ctypes.c_void_p(0)
    F64, F32 = _native.PREC_F64CORE, _native.PREC_F32

    def pairs(prec=F64, rows=fake, n=10, D=4, ld=4, pf=fake, pt=fake, nt=fake, ib=4, B=5, Nn=3, ep=fake, en=fake,
              grad=null, R=1):
        return lib.lec_pairs_poincare(prec, rows, n, D, ld, pf, pt, nt, ib, B, Nn, ep, en, null, grad, R, null)

    assert pairs(prec=F32) == -3                          # only the fp64 core
    assert pairs(ib=3) == -3
    assert pairs(B=-1) == -4 and pairs(Nn=-1) == -4 and pairs(n=-1) == -4
    assert pairs(rows=null) == -1
    assert pairs(D=0) == -2 and pairs(ld=6) == -2 and pairs(D=8, ld=4) == -2
    assert pairs(rows=odd) == -5 and pairs(grad=odd) == -5
    assert pairs(grad=fake, R=0) == -7
    assert pairs(pf=null) == -1 and pairs(ep=null) == -1
    assert pairs(nt=null) == -1 and pairs(en=null) == -1
    assert pairs(B=0, pf=null, pt=null, nt=null, ep=null, en=null) == 0      # empty batch
    # the cone entry points keep rejecting the Poincare distance
    assert lib.lec_pairs_flat(4, 1, fake, fake, 10, 4, 4, fake, fake, 8, null, null, 5, 0.1, 1.0, fake, null, null, 1,
                              null) == -3
    assert lib.lec_pairs_grouped(4, 1, fake, fake, 10, 4, 4, fake, fake, fake, fake, 4, 5, 3, null, null, 0.1, 1.0, fake,
                                 fake, null, null, 1, null) == -3
    assert lib.lec_energy_dense(4, 1, fake, fake, 5, 4, 0.1, fake, null) == -3
    assert lib.lec_energy_dense_bwd(4, 1, fake, fake, fake, 5, 4, 0.1, fake, fake, null) == -3
    assert lib.lec_pairs_grouped(3, 1, fake, fake, 10, 4, 4, fake, fake, fake, fake, 4, 5, 3, null, null, 0.1, 1.0, fake,
                                 fake, null, null, 1, null) == -3

    # scoring: fp32 SIMT only, D <= 64
    def score(geom=4, prec=F32, D=10, N=0, L=5):
        return lib.lec_score_topk_ex(geom, prec, fake, L, fake, N, D, 0.0, null, null, 0, 1, fake, 1, null, null, null)

    assert score(prec=F64) == -3
    assert score(D=65) == -2 and score(D=0) == -2
    assert score() == 0                                                       # no image: nothing launched
    assert score(geom=3) == -3
    assert lib.lec_score_topk(4, F64, fake, 5, fake, 0, 10, 0.0, null, null, 0, 1, fake, null, null, null) == -3
    assert lib.lec_score_topk(4, F32, fake, 5, fake, 0, 10, 0.0, null, null, 0, 1, fake, null, null, null) == 0
    assert lib.lec_score_tc_supported(4, F32, 10, 100, 1) == 0
    assert lib.lec_score_topk_tc(4, F32, fake, 5, fake, 5, 10, 0.0, null, null, 0, 1, fake, null, null, fake, 1 << 20,
                                 null) == -3

    # the update rule: table modes only, row_mode NONE, no aux terms for geometry 4
    def upd(**kw):
        u = _native.LecUpdate()
        u.rule, u.row_mode, u.geom = _native.UPD_RSGD_RETRACT, _native.ROWS_NONE, 4
        u.table, u.grad_rows, u.grad_replicas, u.n, u.D, u.ld = 0x1000, 0x1000, 1, 0, 4, 4
        for k, v in kw.items():
            setattr(u, k, v)
        return lib.lec_update_rows(ctypes.byref(u), None, null)

    assert upd() == 0                                                         # an empty table launches nothing
    assert upd(row_mode=_native.ROWS_HYP_SHELL) == -3
    assert upd(row_mode=_native.ROWS_EUC_SOFTCLIP) == -3
    assert upd(rule=5) == -3
    assert upd(aux_out=0x1000) == -3                                          # geometry 4 has no aux terms
    assert upd(rule=_native.UPD_RSGD, row_mode=_native.ROWS_HYP_SHELL, geom=1) == 0   # other rules unchanged

    # lec_cone_step with geometry 4
    def step(**kw):
        s = _native.LecStep()
        s.geom, s.precision, s.fused = 4, F64, 1
        s.pos_from = s.pos_to = s.neg_to = s.E_pos = s.E_neg = 0x1000
        s.idx_bytes, s.B, s.N = 4, 5, 3
        u = s.upd
        u.rule, u.row_mode, u.geom = _native.UPD_RSGD_RETRACT, _native.ROWS_NONE, 4
        u.table, u.grad_rows, u.grad_replicas, u.n, u.D, u.ld = 0x1000, 0x1000, 1, 10, 4, 4
        u.rows_out, u.loss_acc = 0x1000, 0x1000
        for k, v in kw.items():
            if k.startswith("upd_"):
                setattr(u, k[4:], v)
            else:
                setattr(s, k, v)
        return lib.lec_cone_step(ctypes.byref(s), null)

    assert step(precision=F32) == -3
    assert step(w_pos=0x1000) == -3 and step(w_neg=0x1000) == -3
    assert step(upd_rule=_native.UPD_NONE, upd_row_mode=_native.ROWS_HYP_SHELL) == -3
    assert step(upd_aux_out=0x1000) == -3
    assert step(upd_rows_out=0) == -1

    # evaluation passes: geometry 4 passes the geometry check (the size error behind it is what is reported)
    nb = int(lib.lec_recon_workspace_bytes(1))
    r = _native.LecRecon()
    r.geom, r.rows, r.n, r.D, r.ld = 4, 0x1000, 10, 4, 4
    r.tin, r.tout, r.u_begin, r.u_end, r.workspace, r.workspace_bytes = 0x1000, 0x1000, 3, 2, 0x1000, nb
    out = ctypes.c_void_p(0x1000)
    assert lib.lec_recon_pass(ctypes.byref(r), null) == -4
    assert lib.lec_recon_pass_dag(ctypes.byref(r), None, null) == -4
    assert lib.lec_recon_pass_heldout(ctypes.byref(r), None, None, null) == -4
    assert lib.lec_recon_finish(ctypes.byref(r), out, out, null) == -4
    assert lib.lec_recon_finish_at(ctypes.byref(r), 0.5, out, out, null) == -4
    r.u_begin, r.u_end = 4, 4
    assert lib.lec_recon_pass(ctypes.byref(r), null) == 0
    r.D, r.ld = 65, 68
    assert lib.lec_recon_pass(ctypes.byref(r), null) == -2                    # D <= 64, as for the cones
    r.D, r.ld, r.geom = 4, 4, 3
    assert lib.lec_recon_pass(ctypes.byref(r), null) == -3
    k = _native.LecRank()
    k.geom, k.rows, k.n, k.D, k.ld = 4, 0x1000, 10, 4, 4
    k.tin, k.tout, k.pos_ptr, k.n_pos, k.u_begin, k.u_end = 0x1000, 0x1000, 0x1000, 9, 0, 11
    k.workspace, k.workspace_bytes = 0x1000, 1 << 20
    assert lib.lec_rank_run(ctypes.byref(k), out, out, null, null) == -4
    assert lib.lec_rank_run_heldout(ctypes.byref(k), None, out, out, null, null) == -4
    k.geom = 3
    assert lib.lec_rank_run(ctypes.byref(k), out, out, null, null) == -3


def test_doc_binding_of_the_pair_kernel():
    from test_integration_doc import doc_namespace
    ns = doc_namespace()
    assert list(ns["lib"].lec_pairs_poincare.argtypes) == list(_native.lib().lec_pairs_poincare.argtypes)
    hdr = open(os.path.join(ROOT, "include", "lec_b200.h")).read()
    decl = re.search(r"int lec_pairs_poincare\((.*?)\);", hdr, re.S).group(1)
    assert len(decl.split(",")) == len(_native.lib().lec_pairs_poincare.argtypes)
