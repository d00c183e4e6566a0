"""Lorentz-model embeddings on the GPU: the pair kernel against the fp64 reference of test_lorentz_cpu, the engine steps,
the in-process peer exchange, scoring and every evaluation pass on Lorentz rows, and a short ETHEC training run whose
ball image then seeds the hyperbolic cones."""
import functools
import math

import numpy as np
import pytest
import torch

from learning_embeddings_b200 import _native, hierarchy, metrics, ops, sharding
from learning_embeddings_b200.engine import ConeStep, pack_index_block
from learning_embeddings_b200.sampler import SamplerGraph
from oracle import cones
from test_link_prediction_cpu import link_prediction_oracle
from test_lorentz_cpu import distance_grad, lorentz_distance, lorentz_loss_ref, lorentz_update, lorentz_w
from test_reconstruction_dag_gpu import dag
from test_reconstruction_ranks_cpu import reconstruction_ranks_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
EPS32 = 2.0 ** -24   # unit roundoff of fp32
EPS64 = 2.0 ** -53


@functools.lru_cache(maxsize=None)
def graph(name):
    if name == "ethec":
        return hierarchy.ethec()
    if name == "tree4000":
        return hierarchy.random_tree(4000, 1.0831, seed=1)
    return dag(name)


def lorentz_table(n, D, seed=0, rmax=3.0, far=0, far_r=(10.0, 12.0)):
    """fp32 spatial parts of points at hyperbolic radius up to rmax (|x| = sinh(radius)); the first `far` rows at radius
    in far_r"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, D, generator=g, dtype=torch.float64)
    x = x / x.norm(dim=1, keepdim=True)
    rad = rmax * torch.rand(n, 1, generator=g, dtype=torch.float64)
    if far:
        rad[:far] = far_r[0] + (far_r[1] - far_r[0]) * torch.rand(far, 1, generator=g, dtype=torch.float64)
    return (x * torch.sinh(rad)).float()


def energy_bound(X, Y, D):
    """|kernel d - fp64 reference d|: the kernel's fp64 d rounded once to fp32, and the difference form's own fp64
    rounding (|dw| <= (3D + 12) eps64 s, through arcosh) in both the kernel and the reference"""
    d = lorentz_distance(X, Y)
    s = ((X - Y) ** 2).sum(-1)
    w = lorentz_w(X, Y)
    r = torch.sqrt(w * (w + 2)).clamp(min=1e-300)
    return d, EPS32 * d + 2 * (3 * D + 12) * EPS64 * s / r + 1e-300


def draw_batch(n, B, Nn, seed):
    g = torch.Generator().manual_seed(seed)
    u = torch.randint(0, n, (B,), generator=g)
    v = torch.randint(0, n, (B,), generator=g)
    v = torch.where(v == u, (v + 1) % n, v)
    neg = torch.randint(0, n, (B, Nn), generator=g)
    neg[:3] = u[:3, None]               # delta = 0 pairs (d = 0, no gradient)
    neg[3, 1:] = neg[3, 0]              # a repeated negative
    return u, v, neg


def abs_grad_ref(W, u, v, neg):
    """sum of |contribution| per gradient element, term by term (c (cxx x + cxy y) has two terms of size sinh(radius)
    that cancel far out): the scale of the fp32 rounding in the kernel's gradient"""
    W = W.double()
    others = torch.cat([v[:, None], neg], 1)
    X = W[u][:, None, :].expand(-1, others.shape[1], -1)
    Y = W[others]
    d = lorentz_distance(X, Y)
    c = -torch.softmax(-d, 1)
    c[:, 0] += 1.0
    x0 = torch.sqrt(1 + (X * X).sum(-1, keepdim=True))
    y0 = torch.sqrt(1 + (Y * Y).sum(-1, keepdim=True))
    w = lorentz_w(X, Y)[..., None]
    ir = torch.where(w > 0, 1 / torch.sqrt(w * (w + 2)).clamp(min=1e-300), torch.zeros_like(w))
    ax = ir * (y0 / x0 * X.abs() + Y.abs())
    ay = ir * (x0 / y0 * Y.abs() + X.abs())
    A = torch.zeros_like(W)
    A.index_add_(0, u, (c.abs()[..., None] * ax).sum(1))
    A.index_add_(0, others.reshape(-1), (c.abs()[..., None] * ay).reshape(-1, W.shape[1]))
    return A


# ---- pair kernel ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("replicas", [1, 8])
@pytest.mark.parametrize("idx_dtype", [torch.int16, torch.int32, torch.int64])
@pytest.mark.parametrize("D", [2, 5, 10, 50, 128])
def test_pair_kernel_against_fp64_reference(D, idx_dtype, replicas):
    n, B, Nn = 500, 300, 7
    W = lorentz_table(n, D, seed=D, far=20, far_r=(11.0, 12.0))    # out to hyperbolic radius 12
    u, v, neg = draw_batch(n, B, Nn, seed=D + 1)
    ld = ops.padded_dim(D)
    rows = torch.zeros((n, ld), device=DEV)
    rows[:, :D] = W.to(DEV)
    cast = (lambda t: t.to(torch.int16).view(torch.uint16)) if idx_dtype == torch.int16 else (lambda t: t.to(idx_dtype))
    pf, pt, nt = (cast(t).contiguous().to(DEV) for t in (u, v, neg))
    E_pos = torch.empty(B, device=DEV)
    E_neg = torch.empty((B, Nn), device=DEV)
    loss = torch.zeros(1, device=DEV, dtype=torch.float64)
    grad = torch.zeros((replicas, n, ld), device=DEV)
    _native.check(_native.lib().lec_pairs_lorentz(
        _native.PREC_F64CORE, _native._p(rows), n, D, ld, _native._p(pf), _native._p(pt), _native._p(nt),
        pf.element_size(), B, Nn, _native._p(E_pos), _native._p(E_neg), _native._p(loss), _native._p(grad), replicas,
        _native.stream_ptr()), "lec_pairs_lorentz")
    torch.cuda.synchronize()
    L_ref, Ep_ref, En_ref, G_ref = lorentz_loss_ref(W.double(), u, v, neg)
    Wd = W.double()
    _, bp = energy_bound(Wd[u], Wd[v], D)
    _, bn = energy_bound(Wd[u][:, None, :], Wd[neg], D)
    assert torch.all((E_pos.cpu().double() - Ep_ref).abs() <= bp)
    assert torch.all((E_neg.cpu().double() - En_ref).abs() <= bn)
    assert float(E_neg[0, 0]) == 0.0
    # loss: fp64 throughout, only the summation order and the energies' own fp64 rounding differ
    assert abs(float(loss) - float(L_ref)) <= 1e-11 * abs(float(L_ref)) + 2 * float(bp.sum() + bn.sum())
    # gradient: fp32 coefficients (one rounding) times fp32 rows, accumulated in fp32 over at most 2 + 2N terms per
    # group and added with fp32 reductions: bound each element by (terms + 2) * u * (sum of |contributions|)
    G = grad.sum(0)[:, :D].cpu().double()
    assert torch.all(grad.sum(0)[:, D:] == 0)
    bound = (2 * Nn + 6) * EPS32 * abs_grad_ref(W.double(), u, v, neg) * max(1, B * (Nn + 1) // n) + 1e-30
    err = (G - G_ref).abs()
    assert torch.all(err <= bound), float((err / bound).max())


def test_pair_kernel_out_of_range_ids():
    n, D, B, Nn = 40, 6, 8, 3
    W = lorentz_table(n, D, seed=5)
    u, v, neg = draw_batch(n, B, Nn, seed=6)
    u[1] = n + 3                     # a bad apex: the whole group is NaN, no loss, no gradient
    neg[2, 1] = -1                   # a bad negative: left out of its group's sum
    _native.index_errors(reset=True)
    rows = W.to(DEV)
    loss, E_pos, E_neg = ops.lorentz_loss(rows.clone().requires_grad_(True), D, u.to(DEV), v.to(DEV), neg.to(DEV))
    assert _native.index_errors(reset=True) == 2
    assert torch.isnan(E_pos[1]) and torch.all(torch.isnan(E_neg[1])) and torch.isnan(E_neg[2, 1])
    keep = torch.tensor([i for i in range(B) if i != 1])
    negs2 = torch.cat([neg[2, :1], neg[2, 2:]])
    L_ref = lorentz_loss_ref(W.double(), u[keep[keep != 2]], v[keep[keep != 2]], neg[keep[keep != 2]])[0]
    L_ref = L_ref + lorentz_loss_ref(W.double(), u[2:3], v[2:3], negs2[None])[0]
    assert abs(float(loss) - float(L_ref)) <= 1e-11 * abs(float(L_ref))


def test_autograd_function_matches_reference():
    n, D, B, Nn = 100, 10, 64, 5
    W = lorentz_table(n, D, seed=7)
    u, v, neg = draw_batch(n, B, Nn, seed=8)
    Wd = W.to(DEV).requires_grad_(True)
    loss, _, _ = ops.lorentz_loss(Wd, D, u.to(DEV), v.to(DEV), neg.to(DEV))
    (2.0 * loss).backward()
    L_ref, _, _, G_ref = lorentz_loss_ref(W.double(), u, v, neg)
    assert abs(float(loss) - float(L_ref)) <= 1e-11 * abs(float(L_ref))
    np.testing.assert_allclose(Wd.grad.cpu().double().numpy(), 2.0 * G_ref.numpy(), rtol=1e-5, atol=1e-6)


# ---- engine steps -----------------------------------------------------------------------------------------------------
def ethec_batches(steps, B, Nn, seed):
    h = graph("ethec")
    rng = np.random.default_rng(seed)
    e = h.closure_edges()
    out = []
    for _ in range(steps):
        sel = rng.integers(0, len(e), size=B)
        u, v = e[sel, 0], e[sel, 1]
        nt, nf = h.sample_negatives(u, v, Nn, rng)
        out.append((u, v, nt, nf))
    return h, out


@pytest.mark.parametrize("D", [2, 10, 50])
def test_engine_steps_against_fp64_host_loop(D):
    Nn, B, lr = 10, 512, 0.3
    h, batches = ethec_batches(5, B, Nn, seed=D)
    W0 = lorentz_table(h.n, D, seed=D, rmax=1.5, far=3, far_r=(8.0, 10.0))
    eng = ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=lr)
    eng.write_grad_table = True
    assert eng.E_neg.shape == (B, Nn) and eng.update == "rsgd_lorentz" and eng.aux is None
    ref = ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=lr)
    for i, (u, v, nt, nf) in enumerate(batches):
        W_prev = eng.table.cpu().double()
        blk = pack_index_block(u, v, nt, nf, n_rows=h.n).to(DEV)
        eng.step_device(*eng._split(blk, B))
        # the same step through the three-launch path (rows re-derived from the table) on a copy of the table
        ref.table.copy_(W_prev.float().to(DEV))
        ref.invalidate_rows()
        ref.step_device(*ref._split(blk, B))
        torch.cuda.synchronize()
        assert ref._struct.fused == 0 and eng._struct.fused == (1 if i else 0)
        ut, vt, ntt = (torch.as_tensor(t) for t in (u, v, nt))
        L, Ep, En, G = lorentz_loss_ref(W_prev, ut, vt, ntt)
        W_ref, r = lorentz_update(W_prev, G, lr)
        _, bn = energy_bound(W_prev[ut][:, None, :], W_prev[ntt], D)
        assert abs(float(eng.loss) - float(L)) <= 1e-10 * abs(float(L))
        assert torch.all((eng.E_neg[:B].cpu().double() - En).abs() <= bn)
        # the gradient is summed in fp32 (hot ETHEC rows take thousands of terms): a bound relative to its largest
        # element, times the row's size for r = g + <x,g> x
        scale = 1 + W_prev.norm(dim=1, keepdim=True) ** 2
        g_tol = 1e-5 * float(G.abs().max()) * scale
        assert torch.all((eng.grad_table.cpu().double() - r).abs() <= 2e-4 * r.abs() + g_tol)
        assert torch.all((eng.table.cpu().double() - W_ref).abs() <= 1e-6 * W_ref.abs() + 4 * lr * g_tol + 1e-7)
        assert torch.isfinite(eng.table).all()
        # fused == three-launch step (gradient reductions are added in no fixed order: fp32 last bits)
        np.testing.assert_allclose(eng.table.cpu().numpy(), ref.table.cpu().numpy(), rtol=1e-5, atol=1e-6)
        assert abs(float(eng.loss) - float(ref.loss)) <= 1e-12 * abs(float(L))
        assert torch.equal(eng.rows[:, :D], eng.table) and torch.all(eng.rows[:, D:] == 0)


def test_engine_sampled_and_pipelined_paths():
    """step_sampled, submit_host and submit_host_sampled run the same kernels (neg_from is drawn and ignored)"""
    h = graph("ethec")
    Nn, B, D = 10, 256, 10
    graph_s = SamplerGraph.from_hierarchy(h)
    e = h.closure_edges()
    rng = np.random.default_rng(0)
    W0 = lorentz_table(h.n, D, seed=1, rmax=1e-3)
    a = ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=0.1)
    b = ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=0.1)
    losses = []
    for step in range(4):
        sel = rng.integers(0, len(e), size=B)
        u = torch.as_tensor(e[sel, 0].astype(np.int32), device=DEV)
        v = torch.as_tensor(e[sel, 1].astype(np.int32), device=DEV)
        losses.append(float(a.step_sampled(graph_s, u, v, seed=7, step=step)))
        nt, nf = graph_s.draw_philox(u, v, Nn, 7, step)
        blk = pack_index_block(u.cpu().numpy(), v.cpu().numpy(), nt.cpu().numpy(), np.zeros_like(nf.cpu().numpy()))
        b.submit_host(blk, B)
    got = b.drain()
    torch.cuda.synchronize()
    np.testing.assert_allclose(got, losses, rtol=1e-5)
    np.testing.assert_allclose(a.table.cpu().numpy(), b.table.cpu().numpy(), rtol=1e-5, atol=1e-7)
    pos = pack_index_block(e[:B, 0], e[:B, 1], np.zeros((0,), np.int64), np.zeros((0,), np.int64))
    b.submit_host_sampled(graph_s, pos, B, seed=3)
    assert np.isfinite(b.drain()).all()


@pytest.mark.parametrize("D,world,mode", [(10, 2, 0), (50, 3, 0), (10, 2, 1), (50, 4, 1)])
def test_multi_rank_exchange_in_process(D, world, mode):
    """as test_update_gpu's exchange test: the ranks' tables are bit-identical, and equal the one-rank table up to the
    fp32 summation order of the gradient"""
    Nn, B = 10, 2048
    h, batches = ethec_batches(4, B, Nn, seed=3)
    W0 = lorentz_table(h.n, D, seed=2, rmax=1.0)
    single = ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=0.1)
    xs = sharding.LocalExchange.make(world, h.n, ops.padded_dim(D), torch.device(DEV), mode=mode)
    streams = [torch.cuda.Stream() for _ in range(world)]
    engs = []
    for r in range(world):
        with torch.cuda.stream(streams[r]):
            engs.append(ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=0.1, exchange=xs[r]))
    torch.cuda.synchronize()
    for (u, v, nt, nf) in batches:
        single.step_device(*single._split(pack_index_block(u, v, nt, nf).to(DEV), B))
        parts = []
        for r in range(world):
            lo, hi = sharding.shard_bounds(B, r, world)
            parts.append((pack_index_block(u[lo:hi], v[lo:hi], nt[lo:hi], nf[lo:hi]).to(DEV), hi - lo))
        if mode == 0:
            for r in range(world):
                with torch.cuda.stream(streams[r]):
                    parts[r][0].record_stream(streams[r])
                    engs[r].step_device(*engs[r]._split(*parts[r]))
        else:
            torch.cuda.synchronize()
            for r in range(world):
                engs[r].forward_backward(*engs[r]._split(*parts[r]))
            for phase in (1, 2, 4):
                for r in range(world):
                    engs[r].reduce_and_update(phases=phase)
        torch.cuda.synchronize()
        for r in range(world):
            engs[r].check_exchange()
        total = sum(float(e.loss.item()) for e in engs)
        assert abs(total - float(single.loss.item())) <= 1e-6 * abs(total)
        for e in engs:
            assert abs(float(e.loss_global.item()) - total) <= 1e-12 * abs(total)
    for r in range(1, world):
        assert torch.equal(engs[r].table, engs[0].table) and torch.equal(engs[r].rows, engs[0].rows)
    np.testing.assert_allclose(engs[0].table.cpu().numpy(), single.table.cpu().numpy(), rtol=1e-5, atol=1e-6)


# ---- scoring and evaluation ---------------------------------------------------------------------------------------------
def score_matrix(x, y, geom="lorentz"):
    S = torch.empty((x.shape[0], y.shape[0]), device=DEV)
    ops.score_topk_into(x, y, geom, None, [], [], 1, None, None, S, 1, engine="simt")
    return S


@pytest.mark.parametrize("D", [2, 5, 10, 50, 64])
def test_scoring_against_fp64_distance(D):
    L, n_img = 300, 2000
    lab = lorentz_table(L, D, seed=D, far=60, far_r=(10.0, 15.0))
    img = lorentz_table(n_img, D, seed=D + 100, far=400, far_r=(10.0, 15.0))
    ls, le = [0, 40, 120], [40, 120, 300]
    idx, val, sc = ops.score_topk(lab.to(DEV), img.to(DEV), "lorentz", None, ls, le, k=5, want_scores=True)
    x, y = lab.double()[None, :, :], img.double()[:, None, :]
    ref = lorentz_distance(x, y)                                                      # [N, L]
    # bound (DESIGN.md): w = e_x y0 + (e_y - p) in fp32 from per-row constants rounded once is off by at most
    # Delta = (D + 8) u (x0 y0 - 1 + |x||y|) (the dot product's gamma_D and five roundings); d = arcosh(1 + w) then lies
    # between arcosh(1 + max(w - Delta, 0)) and arcosh(1 + w + Delta), plus a few ulp of the final log1p / sqrt
    x0 = torch.sqrt(1 + (x * x).sum(-1))
    y0 = torch.sqrt(1 + (y * y).sum(-1))
    w = lorentz_w(x, y)
    delta = (D + 8) * EPS32 * (x0 * y0 - 1 + x.norm(dim=-1) * y.norm(dim=-1))
    d_hi = torch.acosh(1 + w + delta)
    d_lo = torch.acosh(1 + torch.clamp(w - delta, min=0))
    slack = 8 * EPS32 * (1 + ref) + 1e-7
    S = sc.cpu().double()
    assert torch.all(S <= d_hi + slack), float((S - d_hi - slack).max())
    assert torch.all(S >= d_lo - slack), float((d_lo - slack - S).max())
    # far out (radius 10 - 15) and apart, the fp32 Lorentz energies keep their digits; the same points on the ball in
    # fp32 (|p| = tanh(radius / 2)) keep few correct digits of 1 - |p|^2, and the Poincare energies lose them
    # ("apart": w > 1000 Delta, where the bound above keeps d to 1e-3 or better)
    far = torch.zeros_like(ref, dtype=torch.bool)
    far[:400, :60] = True
    far &= w > 1e3 * delta
    assert int(far.sum()) > 1000
    err_l = (S - ref).abs()[far]
    P = score_matrix(ops.lorentz_to_ball(lab).to(DEV), ops.lorentz_to_ball(img).to(DEV), "poincare").t().cpu().double()
    err_p = torch.nan_to_num((P - ref).abs()[far], nan=math.inf)
    assert float(err_p.max()) > 10 * float(err_l.max()), (float(err_p.max()), float(err_l.max()))
    # top-k consistent with the matrix (the same instructions)
    Sf = sc.cpu()
    for lvl, (a, b) in enumerate(zip(ls, le)):
        want_v, want_i = torch.sort(Sf[:, a:b], dim=1, stable=True)
        assert torch.equal(val.cpu()[:, lvl], want_v[:, :5])
        assert torch.equal(idx.cpu()[:, lvl].long(), want_i[:, :5] + a)


@functools.lru_cache(maxsize=None)
def lorentz_rows(name, D):
    """rows after 100 engine steps on the closure of `name` (padded [n, ld])"""
    h = graph(name)
    Nn, B = 10, 1024
    eng = ConeStep(lorentz_table(h.n, D, seed=3, rmax=1e-3).to(DEV), "lorentz", Nn, B, lr=0.5)
    e = h.closure_edges()
    rng = np.random.default_rng(0)
    for _ in range(100):
        sel = rng.integers(0, len(e), size=B)
        u, v = e[sel, 0], e[sel, 1]
        nt, nf = h.sample_negatives(u, v, Nn, rng)
        eng.step_device(*eng._split(pack_index_block(u, v, nt, nf).to(DEV), B))
    torch.cuda.synchronize()
    return eng.rows.clone()


def dense_masks(h, edges=None):
    n = h.n
    below = h.is_descendant(np.arange(n)[:, None], np.arange(n)[None, :])
    held = below if edges is None else np.zeros_like(below)
    if edges is not None:
        held[edges[:, 0], edges[:, 1]] = True
    return below, held


@pytest.mark.parametrize("name", ["ethec", "tree4000", "dag4000"])
@pytest.mark.parametrize("D", [2, 10, 50])
def test_evaluation_passes_equal_the_materialised_matrix(name, D):
    h = graph(name)
    rows = lorentz_rows(name, D)
    x = rows[:, :D].contiguous()
    S = score_matrix(x, x)
    below, _ = dense_masks(h)
    off = ~np.eye(h.n, dtype=bool)
    below_t = torch.as_tensor(below, device=DEV)
    off_t = torch.as_tensor(off, device=DEV)
    # reconstruction F1 (padded rows, D given)
    got = metrics.reconstruction_f1(rows, h, "lorentz", None, D=D)
    want = metrics.best_f1_sweep(S[below_t], S[off_t & ~below_t])
    assert np.array_equal(got, want, equal_nan=True), (got, want)
    # reconstruction ranks
    r = metrics.reconstruction_ranks(rows, h, "lorentz", None, D=D, return_ranks=True)
    ranks, ap = reconstruction_ranks_oracle(S.cpu().numpy(), below)
    assert np.array_equal(r["ranks"].cpu().numpy(), ranks)
    has = h.n_desc > 0
    np.testing.assert_allclose(r["ap"][has], ap[has], rtol=1e-12, atol=0)
    assert r["mean_rank"] == ranks[:, 1].sum() / len(ranks)
    assert abs(r["map"] - math.fsum(ap[has].tolist()) / int(has.sum())) <= 1e-12 * r["map"]
    # link prediction on a held-out split
    split = hierarchy.split_edges(h, 0.1, 0.1, 0.5, seed=1)
    edges = split["test"]
    lp = metrics.link_prediction_ranks(rows, h, edges, "lorentz", None, D=D, return_ranks=True)
    _, held = dense_masks(h, edges)
    lranks, lap = link_prediction_oracle(S.cpu().numpy(), below, held)
    order = np.lexsort((edges[:, 1], edges[:, 0]))
    assert np.array_equal(lp["ranks"].cpu().numpy()[order], lranks)
    hh = held.any(1)
    np.testing.assert_allclose(lp["ap"][hh], lap[hh], rtol=1e-12, atol=0)
    f1 = metrics.link_prediction_f1(rows, h, edges, "lorentz", None, D=D)
    neg = ~below & off
    ep, en = S[torch.as_tensor(held, device=DEV)], S[torch.as_tensor(neg, device=DEV)]
    assert np.array_equal(np.asarray(f1, dtype=np.float64), np.asarray(metrics.best_f1_sweep(ep, en), dtype=np.float64),
                          equal_nan=True)
    t = float(np.median(ep.cpu().numpy()))
    row = metrics.link_prediction_f1(rows, h, edges, "lorentz", None, D=D, threshold=t)
    want = metrics.EmbeddingMetrics(ep, en, t, "test").calculate_metrics()
    assert np.array_equal(np.asarray(row, dtype=np.float64), np.asarray(want, dtype=np.float64), equal_nan=True)


# ---- training and hand-off ------------------------------------------------------------------------------------------
def test_ethec_training_raises_map_and_hands_off_to_the_cones():
    h = graph("ethec")
    D, Nn, B, steps = 10, 50, 2520, 400
    graph_s = SamplerGraph.from_hierarchy(h)
    e = h.closure_edges()
    g = torch.Generator().manual_seed(0)
    W0 = (torch.rand(h.n, D, generator=g) * 2 - 1) * 1e-3         # near the origin, as N&K's initial table
    before = metrics.reconstruction_ranks(W0.to(DEV), h, "lorentz", None)
    eng = ConeStep(W0.to(DEV).clone(), "lorentz", Nn, B, lr=0.1)
    rng = np.random.default_rng(0)
    for step in range(steps):
        eng.set_lr(0.01 if step < 20 else 0.3)                     # burn-in at a lower rate
        sel = rng.integers(0, len(e), size=B)
        u = torch.as_tensor(e[sel, 0].astype(np.int32), device=DEV)
        v = torch.as_tensor(e[sel, 1].astype(np.int32), device=DEV)
        eng.step_sampled(graph_s, u, v, seed=11, step=step)
    torch.cuda.synchronize()
    assert torch.isfinite(eng.table).all()
    after = metrics.reconstruction_ranks(eng.table, h, "lorentz", None)
    assert after["map"] > before["map"] + 0.2, (before["map"], after["map"])
    assert after["mean_rank"] < before["mean_rank"]
    # the ball image scored with the Poincare distance: the map keeps d, and the only change is the fp32 rounding of the
    # ball points, which moves d by ~(1 + x0) ulp -- far below the gaps between the energies that decide the ranks, but
    # able to swap a few near-ties.  A tolerance of 0.01 on MAP allows dozens of swapped pairs out of ~2 000 positives.
    P = ops.lorentz_to_ball(eng.table)
    assert float(P.double().norm(dim=1).max()) < 1.0
    ball = metrics.reconstruction_ranks(P, h, "poincare", None)
    assert abs(ball["map"] - after["map"]) <= 0.01, (ball["map"], after["map"])
    # hand-off: the ball image initialises the hyperbolic cones (their shell transform projects it)
    cone = ConeStep(P.clone(), "hyp", 5, 1024, K=0.1, alpha=0.05, lr=0.01)
    for _ in range(5):
        sel = rng.integers(0, len(e), size=1024)
        uu, vv = e[sel, 0], e[sel, 1]
        nt, nf = h.sample_negatives(uu, vv, 5, rng)
        cone.step_device(*cone._split(pack_index_block(uu, vv, nt, nf).to(DEV), 1024))
        torch.cuda.synchronize()
        assert math.isfinite(float(cone.loss))
    assert torch.isfinite(cone.table).all()


def test_rsgd_lorentz_is_the_hyperboloid_rule_only():
    W = lorentz_table(16, 4).to(DEV)
    with pytest.raises(_native.LecError):
        ConeStep(W.clone(), "poincare", 5, 16, update="rsgd_lorentz")
    with pytest.raises(_native.LecError):
        ConeStep(W.clone(), "lorentz", 5, 16, update="rsgd_retract")
    with pytest.raises(_native.LecError):
        ConeStep(W.clone(), "lorentz", 5, 16, update="sgd")
    assert ConeStep(W.clone(), "lorentz", 5, 16, update="none").update == "none"
