"""Poincare embeddings on the GPU: the pair kernel against the fp64 reference of test_poincare_cpu, the engine steps,
the in-process peer exchange, scoring and every evaluation pass on Poincare rows, and a short ETHEC training run whose
table then seeds the hyperbolic cones."""
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
from test_poincare_cpu import MAX_NORM, distance_grad, poincare_distance, poincare_loss_ref, retract_update
from test_reconstruction_dag_gpu import dag
from test_reconstruction_ranks_cpu import reconstruction_ranks_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
EPS32 = 2.0 ** -24   # unit roundoff of fp32


@functools.lru_cache(maxsize=None)
def graph(name):
    if name == "ethec":
        return hierarchy.ethec()
    if name == "tree4000":
        return hierarchy.random_tree(4000, 1.0831, seed=1)
    return dag(name)


def ball_table(n, D, seed=0, rmax=0.9, boundary=0):
    """fp32 points in the unit ball; the first `boundary` rows at |x| = 1 - 1e-5 (the projection radius)"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, D, generator=g, dtype=torch.float64)
    x = x / x.norm(dim=1, keepdim=True)
    x = x * (rmax * torch.rand(n, 1, generator=g, dtype=torch.float64))
    if boundary:
        x[:boundary] = x[:boundary] / x[:boundary].norm(dim=1, keepdim=True) * MAX_NORM
    return x.float()


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
    """sum of |contribution| per gradient element: the scale of the fp32 rounding in the kernel's gradient"""
    W = W.double()
    others = torch.cat([v[:, None], neg], 1)
    X = W[u][:, None, :].expand(-1, others.shape[1], -1)
    Y = W[others]
    d = poincare_distance(X, Y)
    c = -torch.softmax(-d, 1)
    c[:, 0] += 1.0
    gx, gy = distance_grad(X, Y)
    A = torch.zeros_like(W)
    A.index_add_(0, u, (c.abs()[..., None] * gx.abs()).sum(1))
    A.index_add_(0, others.reshape(-1), (c.abs()[..., None] * gy.abs()).reshape(-1, W.shape[1]))
    return A


# ---- pair kernel ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("replicas", [1, 8])
@pytest.mark.parametrize("idx_dtype", [torch.int16, torch.int32, torch.int64])
@pytest.mark.parametrize("D", [2, 5, 10, 50, 128])
def test_pair_kernel_against_fp64_reference(D, idx_dtype, replicas):
    n, B, Nn = 500, 300, 7
    W = ball_table(n, D, seed=D, boundary=20)
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
    _native.check(_native.lib().lec_pairs_poincare(
        _native.PREC_F64CORE, _native._p(rows), n, D, ld, _native._p(pf), _native._p(pt), _native._p(nt),
        pf.element_size(), B, Nn, _native._p(E_pos), _native._p(E_neg), _native._p(loss), _native._p(grad), replicas,
        _native.stream_ptr()), "lec_pairs_poincare")
    torch.cuda.synchronize()
    L_ref, Ep_ref, En_ref, G_ref = poincare_loss_ref(W.double(), u, v, neg)
    # energies: the kernel's fp64 d rounded once to fp32
    np.testing.assert_allclose(E_pos.cpu().double().numpy(), Ep_ref.numpy(), rtol=EPS32, atol=1e-30)
    np.testing.assert_allclose(E_neg.cpu().double().numpy(), En_ref.numpy(), rtol=EPS32, atol=1e-30)
    assert float(E_neg[0, 0]) == 0.0
    # loss: fp64 throughout, only the summation order differs
    assert abs(float(loss) - float(L_ref)) <= 1e-11 * abs(float(L_ref))
    # gradient: fp32 coefficients (one rounding) times fp32 rows, accumulated in fp32 over at most 2 + 2N terms per
    # group and added with fp32 reductions: bound each element by (terms + 2) * u * (sum of |contributions|)
    G = grad.sum(0)[:, :D].cpu().double()
    assert torch.all(grad.sum(0)[:, D:] == 0)
    bound = (2 * Nn + 6) * EPS32 * abs_grad_ref(W.double(), u, v, neg) * max(1, B * (Nn + 1) // n) + 1e-30
    err = (G - G_ref).abs()
    assert torch.all(err <= bound), float((err / bound).max())


def test_pair_kernel_out_of_range_ids():
    n, D, B, Nn = 40, 6, 8, 3
    W = ball_table(n, D, seed=5)
    u, v, neg = draw_batch(n, B, Nn, seed=6)
    u[1] = n + 3                     # a bad apex: the whole group is NaN, no loss, no gradient
    neg[2, 1] = -1                   # a bad negative: left out of its group's sum
    _native.index_errors(reset=True)
    rows = W.to(DEV)
    loss, E_pos, E_neg = ops.poincare_loss(rows.clone().requires_grad_(True), D, u.to(DEV), v.to(DEV), neg.to(DEV))
    assert _native.index_errors(reset=True) == 2
    assert torch.isnan(E_pos[1]) and torch.all(torch.isnan(E_neg[1])) and torch.isnan(E_neg[2, 1])
    keep = torch.tensor([i for i in range(B) if i != 1])
    negs2 = torch.cat([neg[2, :1], neg[2, 2:]])
    L_ref = poincare_loss_ref(W.double(), u[keep[keep != 2]], v[keep[keep != 2]], neg[keep[keep != 2]])[0]
    L_ref = L_ref + poincare_loss_ref(W.double(), u[2:3], v[2:3], negs2[None])[0]
    assert abs(float(loss) - float(L_ref)) <= 1e-11 * abs(float(L_ref))


def test_autograd_function_matches_reference():
    n, D, B, Nn = 100, 10, 64, 5
    W = ball_table(n, D, seed=7)
    u, v, neg = draw_batch(n, B, Nn, seed=8)
    Wd = W.to(DEV).requires_grad_(True)
    loss, _, _ = ops.poincare_loss(Wd, D, u.to(DEV), v.to(DEV), neg.to(DEV))
    (2.0 * loss).backward()
    L_ref, _, _, G_ref = poincare_loss_ref(W.double(), u, v, neg)
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
    W0 = ball_table(h.n, D, seed=D, rmax=0.5, boundary=3)
    eng = ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=lr)
    eng.write_grad_table = True
    assert eng.E_neg.shape == (B, Nn) and eng.update == "rsgd_retract"
    ref = ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=lr)
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
        L, Ep, En, G = poincare_loss_ref(W_prev, torch.as_tensor(u), torch.as_tensor(v), torch.as_tensor(nt))
        W_ref, rg = retract_update(W_prev, G, lr)
        assert abs(float(eng.loss) - float(L)) <= 1e-10 * abs(float(L))
        np.testing.assert_allclose(eng.E_neg[:B].cpu().double().numpy(), En.numpy(), rtol=EPS32, atol=1e-30)
        # the gradient is summed in fp32 (hot ETHEC rows take thousands of terms): a bound relative to its largest element
        g_tol = 1e-5 * float(rg.abs().max())
        np.testing.assert_allclose(eng.grad_table.cpu().double().numpy(), rg.numpy(), rtol=2e-4, atol=g_tol)
        np.testing.assert_allclose(eng.table.cpu().double().numpy(), W_ref.numpy(), rtol=1e-6, atol=lr * g_tol + 1e-7)
        assert float(eng.table.double().norm(dim=1).max()) <= MAX_NORM * (1 + 1e-7)
        # fused == three-launch step (gradient reductions are added in no fixed order: fp32 last bits)
        np.testing.assert_allclose(eng.table.cpu().numpy(), ref.table.cpu().numpy(), rtol=1e-6, atol=1e-7)
        assert abs(float(eng.loss) - float(ref.loss)) <= 1e-12 * abs(float(L))
        assert torch.equal(eng.rows[:, :D], eng.table) and torch.all(eng.rows[:, D:] == 0)


def test_engine_sampled_and_pipelined_paths():
    """step_sampled, submit_host and submit_host_sampled run the same kernels (neg_from is drawn and ignored)"""
    h = graph("ethec")
    Nn, B, D = 10, 256, 10
    graph_s = SamplerGraph.from_hierarchy(h)
    e = h.closure_edges()
    rng = np.random.default_rng(0)
    W0 = ball_table(h.n, D, seed=1, rmax=1e-3)
    a = ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=0.1)
    b = ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=0.1)
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
    W0 = ball_table(h.n, D, seed=2, rmax=0.5)
    single = ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=0.1)
    xs = sharding.LocalExchange.make(world, h.n, ops.padded_dim(D), torch.device(DEV), mode=mode)
    streams = [torch.cuda.Stream() for _ in range(world)]
    engs = []
    for r in range(world):
        with torch.cuda.stream(streams[r]):
            engs.append(ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=0.1, exchange=xs[r]))
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
def score_matrix(x, y):
    S = torch.empty((x.shape[0], y.shape[0]), device=DEV)
    ops.score_topk_into(x, y, "poincare", None, [], [], 1, None, None, S, 1, engine="simt")
    return S


@pytest.mark.parametrize("D", [2, 5, 10, 50, 64])
def test_scoring_against_fp64_distance(D):
    L, n_img = 300, 2000
    lab, img = ball_table(L, D, seed=D, boundary=5), ball_table(n_img, D, seed=D + 100)
    ls, le = [0, 40, 120], [40, 120, 300]
    idx, val, sc = ops.score_topk(lab.to(DEV), img.to(DEV), "poincare", None, ls, le, k=5, want_scores=True)
    ref = poincare_distance(lab.double()[None, :, :], img.double()[:, None, :])      # [N, L]
    # bound: |x-y|^2 = A + B - 2p in fp32 loses ~4 u (A + B) absolutely; through delta = 2s/((1-A)(1-B)) and
    # d = arcosh(1 + delta) (dd/ddelta = 1/sqrt(delta (delta + 2))) that is the first term; the rest is a few ulps of d
    A = (lab.double() ** 2).sum(1)[None, :]
    B = (img.double() ** 2).sum(1)[:, None]
    delta = 2 * ((lab.double()[None] - img.double()[:, None]) ** 2).sum(2) / ((1 - A) * (1 - B))
    s_err = 8 * EPS32 * (A + B) * 2 / ((1 - A) * (1 - B))
    bound = s_err / torch.sqrt(torch.clamp(delta * (delta + 2), min=s_err * s_err)) + 8 * EPS32 * ref + 1e-7
    err = (sc.cpu().double() - ref).abs()
    assert torch.all(err <= bound), float((err / bound).max())
    # top-k consistent with the matrix (the same instructions)
    S = sc.cpu()
    for lvl, (a, b) in enumerate(zip(ls, le)):
        want_v, want_i = torch.sort(S[:, a:b], dim=1, stable=True)
        assert torch.equal(val.cpu()[:, lvl], want_v[:, :5])
        assert torch.equal(idx.cpu()[:, lvl].long(), want_i[:, :5] + a)


@functools.lru_cache(maxsize=None)
def poincare_rows(name, D):
    """rows after 100 engine steps on the closure of `name` (padded [n, ld])"""
    h = graph(name)
    Nn, B = 10, 1024
    eng = ConeStep(ball_table(h.n, D, seed=3, rmax=1e-3).to(DEV), "poincare", Nn, B, lr=0.5)
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
    rows = poincare_rows(name, D)
    x = rows[:, :D].contiguous()
    S = score_matrix(x, x)
    below, _ = dense_masks(h)
    off = ~np.eye(h.n, dtype=bool)
    below_t = torch.as_tensor(below, device=DEV)
    off_t = torch.as_tensor(off, device=DEV)
    # reconstruction F1 (padded rows, D given)
    got = metrics.reconstruction_f1(rows, h, "poincare", None, D=D)
    want = metrics.best_f1_sweep(S[below_t], S[off_t & ~below_t])
    assert np.array_equal(got, want, equal_nan=True), (got, want)
    # reconstruction ranks
    r = metrics.reconstruction_ranks(rows, h, "poincare", None, D=D, return_ranks=True)
    ranks, ap = reconstruction_ranks_oracle(S.cpu().numpy(), below)
    assert np.array_equal(r["ranks"].cpu().numpy(), ranks)
    has = h.n_desc > 0
    np.testing.assert_allclose(r["ap"][has], ap[has], rtol=1e-12, atol=0)
    assert r["mean_rank"] == ranks[:, 1].sum() / len(ranks)
    assert abs(r["map"] - math.fsum(ap[has].tolist()) / int(has.sum())) <= 1e-12 * r["map"]
    # link prediction on a held-out split
    split = hierarchy.split_edges(h, 0.1, 0.1, 0.5, seed=1)
    edges = split["test"]
    lp = metrics.link_prediction_ranks(rows, h, edges, "poincare", None, D=D, return_ranks=True)
    _, held = dense_masks(h, edges)
    lranks, lap = link_prediction_oracle(S.cpu().numpy(), below, held)
    order = np.lexsort((edges[:, 1], edges[:, 0]))
    assert np.array_equal(lp["ranks"].cpu().numpy()[order], lranks)
    hh = held.any(1)
    np.testing.assert_allclose(lp["ap"][hh], lap[hh], rtol=1e-12, atol=0)
    f1 = metrics.link_prediction_f1(rows, h, edges, "poincare", None, D=D)
    neg = ~below & off
    ep, en = S[torch.as_tensor(held, device=DEV)], S[torch.as_tensor(neg, device=DEV)]
    assert np.array_equal(np.asarray(f1, dtype=np.float64), np.asarray(metrics.best_f1_sweep(ep, en), dtype=np.float64),
                          equal_nan=True)
    t = float(np.median(ep.cpu().numpy()))
    row = metrics.link_prediction_f1(rows, h, edges, "poincare", None, D=D, threshold=t)
    want = metrics.EmbeddingMetrics(ep, en, t, "test").calculate_metrics()
    assert np.array_equal(np.asarray(row, dtype=np.float64), np.asarray(want, dtype=np.float64), equal_nan=True)


# ---- training and hand-off ------------------------------------------------------------------------------------------
def test_ethec_training_raises_map_and_hands_off_to_the_cones():
    h = graph("ethec")
    D, Nn, B, steps = 10, 50, 2520, 400
    graph_s = SamplerGraph.from_hierarchy(h)
    e = h.closure_edges()
    g = torch.Generator().manual_seed(0)
    W0 = (torch.rand(h.n, D, generator=g) * 2 - 1) * 1e-3         # N&K's uniform(-1e-3, 1e-3) initial table
    before = metrics.reconstruction_ranks(W0.to(DEV), h, "poincare", None)
    eng = ConeStep(W0.to(DEV).clone(), "poincare", Nn, B, lr=0.1)
    rng = np.random.default_rng(0)
    for step in range(steps):
        eng.set_lr(0.01 if step < 20 else 0.3)                     # burn-in at a lower rate
        sel = rng.integers(0, len(e), size=B)
        u = torch.as_tensor(e[sel, 0].astype(np.int32), device=DEV)
        v = torch.as_tensor(e[sel, 1].astype(np.int32), device=DEV)
        eng.step_sampled(graph_s, u, v, seed=11, step=step)
    torch.cuda.synchronize()
    assert torch.isfinite(eng.table).all()
    assert float(eng.table.double().norm(dim=1).max()) <= MAX_NORM * (1 + 1e-7)
    after = metrics.reconstruction_ranks(eng.table, h, "poincare", None)
    assert after["map"] > before["map"] + 0.2, (before["map"], after["map"])
    assert after["mean_rank"] < before["mean_rank"]
    # hand-off: the trained table initialises the hyperbolic cones (their shell transform projects it)
    cone = ConeStep(eng.table.clone(), "hyp", 5, 1024, K=0.1, alpha=0.05, lr=0.01)
    for _ in range(5):
        sel = rng.integers(0, len(e), size=1024)
        uu, vv = e[sel, 0], e[sel, 1]
        nt, nf = h.sample_negatives(uu, vv, 5, rng)
        cone.step_device(*cone._split(pack_index_block(uu, vv, nt, nf).to(DEV), 1024))
        torch.cuda.synchronize()
        assert math.isfinite(float(cone.loss))
    assert torch.isfinite(cone.table).all()
