"""Lorentz-model embeddings (Nickel & Kiela 2018) without a GPU: an fp64 torch reference of the distance, the softmax loss
and the update rule in the spatial chart (the GPU tests compare the kernels against it), checked against autograd, the
ambient hyperboloid form of the update, the Poincare distance through the ball map and exact distances on a ray; and the
argument codes of the new and extended entry points."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from learning_embeddings_b200 import _native, ops
from test_poincare_cpu import poincare_distance

EPS64 = 2.0 ** -53


# ---- fp64 reference -------------------------------------------------------------------------------------------------
def lorentz_w(x, y):
    """w = -<X,Y>_L - 1 in the difference form (s - (x0 - y0)^2) / 2, x0 - y0 = (A - B) / (x0 + y0) with
    A - B = <x - y, x + y>, clamped at 0."""
    A, B = (x * x).sum(-1), (y * y).sum(-1)
    s = ((x - y) ** 2).sum(-1)
    t = ((x - y) * (x + y)).sum(-1) / (torch.sqrt(1.0 + A) + torch.sqrt(1.0 + B))
    return torch.clamp(0.5 * (s - t * t), min=0.0)


def lorentz_distance(x, y):
    """arcosh(1 + w) as log1p(w + sqrt(w (w + 2)))."""
    w = lorentz_w(x, y)
    return torch.log1p(w + torch.sqrt(w * (w + 2.0)))


def distance_grad(x, y):
    """Closed-form dd/dx = (y0/x0 x - y) / r, dd/dy = (x0/y0 y - x) / r, r = sqrt(w (w + 2)); zero where w = 0."""
    x0 = torch.sqrt(1.0 + (x * x).sum(-1, keepdim=True))
    y0 = torch.sqrt(1.0 + (y * y).sum(-1, keepdim=True))
    w = lorentz_w(x, y)[..., None]
    r = torch.sqrt(w * (w + 2.0))
    safe = torch.where(w > 0, r, torch.ones_like(r))
    gx = (y0 / x0 * x - y) / safe
    gy = (x0 / y0 * y - x) / safe
    zero = w <= 0
    return torch.where(zero, torch.zeros_like(gx), gx), torch.where(zero, torch.zeros_like(gy), gy)


def lorentz_loss_ref(W, u, v, neg):
    """W [n, D] fp64 spatial parts; u, v [B]; neg [B, N].  Returns (loss, E_pos [B], E_neg [B, N], dloss/dW [n, D]),
    all fp64, the gradient from the closed form."""
    W = W.double()
    u, v, neg = (torch.as_tensor(t, dtype=torch.int64) for t in (u, v, neg))
    Bn, Nn = neg.shape
    others = torch.cat([v[:, None], neg], 1)
    X = W[u][:, None, :].expand(Bn, Nn + 1, W.shape[1])
    Y = W[others]
    d = lorentz_distance(X, Y)
    lse = torch.logsumexp(-d, 1)
    loss = (d[:, 0] + lse).sum()
    c = -torch.softmax(-d, 1)
    c[:, 0] += 1.0
    gx, gy = distance_grad(X, Y)
    G = torch.zeros_like(W)
    G.index_add_(0, u, (c[..., None] * gx).sum(1))
    G.index_add_(0, others.reshape(-1), (c[..., None] * gy).reshape(-1, W.shape[1]))
    return loss, d[:, 0], d[:, 1:], G


def lorentz_update(W, G, lr):
    """LEC_UPD_RSGD_LORENTZ in the spatial chart: r = g + <x,g> x, nu = sqrt(|g|^2 + <x,g>^2), t = lr nu,
    x <- cosh(t) x - lr sinh(t)/t r (unchanged where nu = 0).  Returns (new W, r)."""
    W, G = W.double(), G.double()
    c = (W * G).sum(1, keepdim=True)
    r = G + c * W
    nu = torch.sqrt((G * G).sum(1, keepdim=True) + c * c)
    t = lr * nu
    shc = torch.where(t > 0, torch.sinh(t) / torch.where(t > 0, t, torch.ones_like(t)), torch.ones_like(t))
    out = torch.cosh(t) * W - lr * shc * r
    return torch.where(nu > 0, out, W), r


def ambient_update(W, G_amb, lr):
    """Nickel & Kiela 2018 on the hyperboloid X = (x0, x): h = (-G0, Gs), h <- h + <X,h>_L X, X <- exp_X(-lr h).
    G_amb [n, D + 1] is the Euclidean gradient with respect to (X0, Xs).  Returns the new points [n, D + 1]."""
    x0 = torch.sqrt(1.0 + (W * W).sum(1, keepdim=True))
    X = torch.cat([x0, W], 1)

    def ldot(a, b):
        return -a[:, :1] * b[:, :1] + (a[:, 1:] * b[:, 1:]).sum(1, keepdim=True)

    h = torch.cat([-G_amb[:, :1], G_amb[:, 1:]], 1)
    h = h + ldot(X, h) * X
    v = -lr * h
    nv = torch.sqrt(torch.clamp(ldot(v, v), min=0.0))
    safe = torch.where(nv > 0, nv, torch.ones_like(nv))
    return torch.where(nv > 0, torch.cosh(nv) * X + torch.sinh(nv) * v / safe, X)


def random_points(n, D, gen, rmax=3.0):
    """spatial parts of points at hyperbolic radius up to rmax: |x| = sinh(radius)"""
    x = torch.randn(n, D, generator=gen, dtype=torch.float64)
    rad = rmax * torch.rand(n, 1, generator=gen, dtype=torch.float64)
    return x / x.norm(dim=1, keepdim=True) * torch.sinh(rad)


# ---- the reference itself -------------------------------------------------------------------------------------------
def test_distance_properties():
    g = torch.Generator().manual_seed(0)
    x, y = random_points(50, 7, g), random_points(50, 7, g)
    d = lorentz_distance(x, y)
    assert torch.allclose(d, lorentz_distance(y, x), rtol=0, atol=1e-13)
    assert torch.equal(lorentz_distance(x, x), torch.zeros(50, dtype=torch.float64))
    # arcosh(-<X,Y>_L) directly (accurate here: moderate radii, points apart)
    x0, y0 = torch.sqrt(1 + (x * x).sum(1)), torch.sqrt(1 + (y * y).sum(1))
    torch.testing.assert_close(d, torch.acosh(x0 * y0 - (x * y).sum(1)), rtol=1e-10, atol=1e-10)
    # from the origin: d(0, y) = asinh |y|
    torch.testing.assert_close(lorentz_distance(torch.zeros_like(y), y), torch.asinh(y.norm(dim=1)), rtol=1e-13, atol=0)


def test_distance_equals_poincare_through_the_ball_map():
    g = torch.Generator().manual_seed(1)
    x, y = random_points(200, 5, g, rmax=6.0), random_points(200, 5, g, rmax=6.0)
    px = x / (1 + torch.sqrt(1 + (x * x).sum(1, keepdim=True)))
    py = y / (1 + torch.sqrt(1 + (y * y).sum(1, keepdim=True)))
    torch.testing.assert_close(lorentz_distance(x, y), poincare_distance(px, py), rtol=1e-9, atol=1e-9)


def test_ball_maps_round_trip():
    g = torch.Generator().manual_seed(2)
    W = random_points(300, 10, g, rmax=8.0).float()
    P = ops.lorentz_to_ball(W)
    assert P.dtype == torch.float32 and float(P.double().norm(dim=1).max()) < 1.0
    P64 = W.double() / (1 + torch.sqrt(1 + (W.double() ** 2).sum(1, keepdim=True)))
    torch.testing.assert_close(P, P64.float(), rtol=0, atol=0)
    # the inverse in fp64 of the fp32 ball points: 1 - |p|^2 keeps few digits at radius 8 (|p| = tanh(4)), so the round
    # trip is exact only up to the conditioning of 2p / (1 - |p|^2), ~ (1 + x0) ulp of p relative
    back = ops.ball_to_lorentz(P)
    x0 = torch.sqrt(1 + (W.double() ** 2).sum(1))
    err = (back.double() - W.double()).norm(dim=1) / W.double().norm(dim=1).clamp(min=1e-30)
    assert bool((err <= 4 * (1 + x0) * 2.0 ** -24 + 2.0 ** -23).all()), float(err.max())
    # exact in fp64 arithmetic for moderate points
    Wm = random_points(50, 4, g, rmax=2.0)
    Pm = Wm / (1 + torch.sqrt(1 + (Wm * Wm).sum(1, keepdim=True)))
    torch.testing.assert_close(2 * Pm / (1 - (Pm * Pm).sum(1, keepdim=True)), Wm, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("radius", [0.5, 3.0, 8.0, 12.0, 15.0])
def test_points_on_a_ray_against_the_exact_distance(radius):
    """x = a e, y = b e: d = |asinh a - asinh b| exactly.  Every input of the difference form's last subtraction
    s - t^2 is accurate to a few ulp of s (A - B is summed from the differences), so |dw| <= (3D + 12) eps s and, through
    arcosh, |dd| <= (3D + 12) eps s / r + 4 eps d with r = sqrt(w (w + 2)) = sinh d.  Along a ray s - t^2 is itself
    ill-conditioned far out (w / s ~ 1 / sinh^2 radius), so at radius 15 that is ~1e-3 for d ~ 1; the naive
    x0 y0 - 1 - <x,y> instead loses everything for nearby points."""
    g = torch.Generator().manual_seed(3)
    D = 6
    e = torch.randn(1, D, generator=g, dtype=torch.float64)
    e = e / e.norm()
    xi = radius - 2.0 * torch.rand(64, 1, generator=g, dtype=torch.float64)
    eta = xi - torch.logspace(-6, 0.5, 64, dtype=torch.float64)[:, None]
    a, b = torch.sinh(xi), torch.sinh(eta)
    x, y = a * e, b * e
    d = lorentz_distance(x, y)
    an, bn = (x * e).sum(1), (y * e).sum(1)         # the rounded points' own signed coordinates along the ray
    exact = (torch.asinh(an) - torch.asinh(bn)).abs()
    s = ((x - y) ** 2).sum(1)
    r = torch.sinh(exact)
    # plus the rounding of the reference itself (two asinh values of their own size)
    bound = (3 * D + 12) * EPS64 * s / r + 4 * EPS64 * (exact + torch.asinh(an).abs() + torch.asinh(bn).abs())
    assert bool(((d - exact).abs() <= bound).all()), float(((d - exact).abs() / bound).max())
    # the naive form x0 y0 - 1 - <x,y> breaks down for nearby points far out
    if radius >= 12.0:
        x0, y0 = torch.sqrt(1 + an ** 2), torch.sqrt(1 + bn ** 2)
        naive = torch.acosh(torch.clamp(x0 * y0 - (x * y).sum(1), min=1.0))
        assert float((naive - exact).abs()[:8].max()) > 1e3 * float(bound[:8].max())


def test_w_zero():
    x = torch.tensor([[1.5, -20.0, 3.0]], dtype=torch.float64)
    assert float(lorentz_w(x, x.clone())) == 0.0
    gx, gy = distance_grad(x, x.clone())
    assert torch.equal(gx, torch.zeros_like(x)) and torch.equal(gy, torch.zeros_like(x))
    W = torch.cat([x, x])
    loss, E_pos, E_neg, G = lorentz_loss_ref(W, [0], [1], [[0]])
    assert float(E_pos[0]) == 0.0 and float(E_neg[0, 0]) == 0.0
    assert torch.equal(G, torch.zeros_like(W))
    assert abs(float(loss) - np.log(2.0)) < 1e-15


@pytest.mark.parametrize("case", ["random", "near_coincident", "far_out"])
def test_closed_form_gradient_matches_autograd(case):
    g = torch.Generator().manual_seed(4)
    D = 5
    x, y = random_points(6, D, g), random_points(6, D, g)
    if case == "near_coincident":
        y = x + 1e-6 * torch.randn(6, D, generator=g, dtype=torch.float64)
    elif case == "far_out":
        x, y = random_points(6, D, g, rmax=10.0), random_points(6, D, g, rmax=10.0)
    gx, gy = distance_grad(x, y)
    xa, ya = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    lorentz_distance(xa, ya).sum().backward()
    torch.testing.assert_close(gx, xa.grad, rtol=1e-6, atol=1e-9)
    torch.testing.assert_close(gy, ya.grad, rtol=1e-6, atol=1e-9)
    if case == "random":
        assert torch.autograd.gradcheck(lambda a, b: lorentz_distance(a, b), (xa.detach().requires_grad_(True),
                                                                                ya.detach().requires_grad_(True)))


def test_loss_and_gradient_against_autograd():
    g = torch.Generator().manual_seed(5)
    n, D, Bn, Nn = 30, 4, 12, 6
    W = random_points(n, D, g)
    u = torch.randint(0, n, (Bn,), generator=g)
    v = torch.randint(0, n, (Bn,), generator=g)
    neg = torch.randint(0, n, (Bn, Nn), generator=g)
    neg[0, :] = neg[0, 0]
    v = torch.where(v == u, (v + 1) % n, v)
    neg = torch.where(neg == u[:, None], (neg + 1) % n, neg)
    loss, E_pos, E_neg, G = lorentz_loss_ref(W, u, v, neg)

    def f(Wa):
        d_pos = lorentz_distance(Wa[u], Wa[v])
        d_all = lorentz_distance(Wa[u][:, None, :], Wa[torch.cat([v[:, None], neg], 1)])
        return (d_pos + torch.logsumexp(-d_all, 1)).sum()

    Wa = W.clone().requires_grad_(True)
    la = f(Wa)
    la.backward()
    assert abs(float(loss) - float(la.detach())) <= 1e-12 * abs(float(la.detach()))
    torch.testing.assert_close(G, Wa.grad, rtol=1e-9, atol=1e-12)
    assert torch.autograd.gradcheck(f, (W.clone().requires_grad_(True),))


@pytest.mark.parametrize("lr", [1e-3, 0.3, 2.0])
def test_chart_update_equals_the_ambient_update(lr):
    """The same loss written on the ambient coordinates (X0 free) has a different Euclidean gradient, but the same
    Riemannian one: the spatial part of N&K's ambient step equals the chart step."""
    g = torch.Generator().manual_seed(6)
    n, D = 20, 4
    W = random_points(n, D, g, rmax=4.0)
    Y = random_points(n, D, g, rmax=4.0)
    Y0 = torch.sqrt(1 + (Y * Y).sum(1, keepdim=True))

    def loss_chart(Wc):
        return torch.acosh(torch.sqrt(1 + (Wc * Wc).sum(1)) * Y0[:, 0] - (Wc * Y).sum(1)).sum()

    def loss_ambient(X):
        return torch.acosh(X[:, 0] * Y0[:, 0] - (X[:, 1:] * Y).sum(1)).sum()

    Wc = W.clone().requires_grad_(True)
    loss_chart(Wc).backward()
    X = torch.cat([torch.sqrt(1 + (W * W).sum(1, keepdim=True)), W], 1).requires_grad_(True)
    loss_ambient(X).backward()
    new_chart, r = lorentz_update(W, Wc.grad, lr)
    new_amb = ambient_update(W, X.grad, lr)
    torch.testing.assert_close(new_chart, new_amb[:, 1:], rtol=1e-10, atol=1e-10)
    # the result is on the hyperboloid: its time coordinate is the implied one
    torch.testing.assert_close(new_amb[:, 0], torch.sqrt(1 + (new_amb[:, 1:] ** 2).sum(1)), rtol=1e-10, atol=0)
    # r is the spatial part of the tangent vector h
    c = (W * Wc.grad).sum(1, keepdim=True)
    torch.testing.assert_close(r, Wc.grad + c * W)
    # a zero gradient leaves the row alone
    same, _ = lorentz_update(W, torch.zeros_like(W), lr)
    assert torch.equal(same, W)


def test_update_step_length():
    """the step moves the point by exactly t = lr nu along the geodesic"""
    g = torch.Generator().manual_seed(7)
    W = random_points(16, 3, g)
    G = torch.randn(16, 3, generator=g, dtype=torch.float64)
    lr = 0.1
    out, _ = lorentz_update(W, G, lr)
    c = (W * G).sum(1)
    nu = torch.sqrt((G * G).sum(1) + c * c)
    torch.testing.assert_close(lorentz_distance(W, out), lr * nu, rtol=1e-9, atol=1e-12)


# ---- argument codes -------------------------------------------------------------------------------------------------
def test_lorentz_constants():
    assert _native.GEOM["lorentz"] == 5 and _native.UPD_RSGD_LORENTZ == 5 and _native.ABI_VERSION == 14
    lib = _native.lib()
    assert lib.lec_abi_version() == 14


def test_argument_validation_codes():
    lib = _native.lib()
    fake = ctypes.c_void_p(0x1000)
    odd = ctypes.c_void_p(0x1004)
    null = ctypes.c_void_p(0)
    F64, F32 = _native.PREC_F64CORE, _native.PREC_F32
    LOR = _native.GEOM["lorentz"]

    def pairs(prec=F64, rows=fake, n=10, D=4, ld=4, pf=fake, pt=fake, nt=fake, ib=4, B=5, Nn=3, ep=fake, en=fake,
              grad=null, R=1):
        return lib.lec_pairs_lorentz(prec, rows, n, D, ld, pf, pt, nt, ib, B, Nn, ep, en, null, grad, R, null)

    assert pairs(prec=F32) == -3
    assert pairs(ib=3) == -3
    assert pairs(B=-1) == -4 and pairs(Nn=-1) == -4 and pairs(n=-1) == -4
    assert pairs(rows=null) == -1
    assert pairs(D=0) == -2 and pairs(ld=6) == -2 and pairs(D=8, ld=4) == -2
    assert pairs(rows=odd) == -5 and pairs(grad=odd) == -5
    assert pairs(grad=fake, R=0) == -7
    assert pairs(pf=null) == -1 and pairs(ep=null) == -1
    assert pairs(nt=null) == -1 and pairs(en=null) == -1
    assert pairs(B=0, pf=null, pt=null, nt=null, ep=null, en=null) == 0
    # the cone entry points reject the Lorentz distance
    assert lib.lec_pairs_flat(LOR, 1, fake, fake, 10, 4, 4, fake, fake, 8, null, null, 5, 0.1, 1.0, fake, null, null, 1,
                              null) == -3
    assert lib.lec_pairs_grouped(LOR, 1, fake, fake, 10, 4, 4, fake, fake, fake, fake, 4, 5, 3, null, null, 0.1, 1.0,
                                 fake, fake, null, null, 1, null) == -3
    assert lib.lec_energy_dense(LOR, 1, fake, fake, 5, 4, 0.1, fake, null) == -3
    assert lib.lec_energy_dense_bwd(LOR, 1, fake, fake, fake, 5, 4, 0.1, fake, fake, null) == -3
    assert lib.lec_pairs_grouped(6, 1, fake, fake, 10, 4, 4, fake, fake, fake, fake, 4, 5, 3, null, null, 0.1, 1.0, fake,
                                 fake, null, null, 1, null) == -3

    # scoring: fp32 SIMT only, D <= 64
    def score(geom=LOR, prec=F32, D=10, N=0, L=5):
        return lib.lec_score_topk_ex(geom, prec, fake, L, fake, N, D, 0.0, null, null, 0, 1, fake, 1, null, null, null)

    assert score(prec=F64) == -3
    assert score(D=65) == -2 and score(D=0) == -2
    assert score() == 0
    assert score(geom=6) == -3
    assert lib.lec_score_topk(LOR, F64, fake, 5, fake, 0, 10, 0.0, null, null, 0, 1, fake, null, null, null) == -3
    assert lib.lec_score_topk(LOR, F32, fake, 5, fake, 0, 10, 0.0, null, null, 0, 1, fake, null, null, null) == 0
    assert lib.lec_score_tc_supported(LOR, F32, 10, 100, 1) == 0
    assert lib.lec_score_topk_tc(LOR, F32, fake, 5, fake, 5, 10, 0.0, null, null, 0, 1, fake, null, null, fake, 1 << 20,
                                 null) == -3

    # the update rule: geometry 5, row_mode NONE, no aux terms
    def upd(**kw):
        u = _native.LecUpdate()
        u.rule, u.row_mode, u.geom = _native.UPD_RSGD_LORENTZ, _native.ROWS_NONE, LOR
        u.table, u.grad_rows, u.grad_replicas, u.n, u.D, u.ld = 0x1000, 0x1000, 1, 0, 4, 4
        for k, v in kw.items():
            setattr(u, k, v)
        return lib.lec_update_rows(ctypes.byref(u), None, null)

    assert upd() == 0
    assert upd(row_mode=_native.ROWS_HYP_SHELL) == -3
    assert upd(row_mode=_native.ROWS_EUC_SOFTCLIP) == -3
    assert upd(aux_out=0x1000) == -3
    assert upd(geom=4) == -3 and upd(geom=1) == -3                            # the hyperboloid's rule only
    assert upd(rule=6) == -3
    assert upd(rule=_native.UPD_RSGD_RETRACT, geom=4) == 0                    # the other rules unchanged
    assert upd(rule=_native.UPD_NONE) == 0

    def step(**kw):
        s = _native.LecStep()
        s.geom, s.precision, s.fused = LOR, F64, 1
        s.pos_from = s.pos_to = s.neg_to = s.E_pos = s.E_neg = 0x1000
        s.idx_bytes, s.B, s.N = 4, 5, 3
        u = s.upd
        u.rule, u.row_mode, u.geom = _native.UPD_RSGD_LORENTZ, _native.ROWS_NONE, LOR
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
    assert step(B=-1) == -4

    # evaluation passes accept geometry 5 (the size error behind the geometry check is what is reported)
    nb = int(lib.lec_recon_workspace_bytes(1))
    r = _native.LecRecon()
    r.geom, r.rows, r.n, r.D, r.ld = LOR, 0x1000, 10, 4, 4
    r.tin, r.tout, r.u_begin, r.u_end, r.workspace, r.workspace_bytes = 0x1000, 0x1000, 3, 2, 0x1000, nb
    out = ctypes.c_void_p(0x1000)
    assert lib.lec_recon_pass(ctypes.byref(r), null) == -4
    assert lib.lec_recon_pass_dag(ctypes.byref(r), None, null) == -4
    assert lib.lec_recon_pass_heldout(ctypes.byref(r), None, None, null) == -4
    assert lib.lec_recon_finish(ctypes.byref(r), out, out, null) == -4
    r.u_begin, r.u_end = 4, 4
    assert lib.lec_recon_pass(ctypes.byref(r), null) == 0
    r.D, r.ld = 65, 68
    assert lib.lec_recon_pass(ctypes.byref(r), null) == -2
    r.D, r.ld, r.geom = 4, 4, 6
    assert lib.lec_recon_pass(ctypes.byref(r), null) == -3
    k = _native.LecRank()
    k.geom, k.rows, k.n, k.D, k.ld = LOR, 0x1000, 10, 4, 4
    k.tin, k.tout, k.pos_ptr, k.n_pos, k.u_begin, k.u_end = 0x1000, 0x1000, 0x1000, 9, 0, 11
    k.workspace, k.workspace_bytes = 0x1000, 1 << 20
    assert lib.lec_rank_run(ctypes.byref(k), out, out, null, null) == -4
    assert lib.lec_rank_run_heldout(ctypes.byref(k), None, out, out, null, null) == -4
    k.geom = 6
    assert lib.lec_rank_run(ctypes.byref(k), out, out, null, null) == -3


def test_engine_rule_name():
    from learning_embeddings_b200.engine import RULES
    assert RULES["rsgd_lorentz"] == _native.UPD_RSGD_LORENTZ


def test_doc_binding_of_the_pair_kernel():
    from test_integration_doc import doc_namespace
    ns = doc_namespace()
    assert list(ns["lib"].lec_pairs_lorentz.argtypes) == list(_native.lib().lec_pairs_lorentz.argtypes)
    hdr = open(os.path.join(ROOT, "include", "lec_b200.h")).read()
    decl = re.search(r"int lec_pairs_lorentz\((.*?)\);", hdr, re.S).group(1)
    assert len(decl.split(",")) == len(_native.lib().lec_pairs_lorentz.argtypes)
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert "lorentz_to_ball" in doc and 'ConeStep(W, "lorentz"' in doc
