"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the reference's golden
vectors.  Tolerance contract (SURVEY.md 8c), written out here:

    |new - ref64| <= max(1e-5 * |ref64|, 2 * |ref32 - ref64|, 2e-6)

where ref64 / ref32 are the reference's own FP64 / FP32 results on the same FP32 inputs; for
gradients the same inequality on per-row L2 norms.  Indices and predicted label sets: bit-exact
(away from energy ties > 1e-5).
"""
import random

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import cones, sampler

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from learning_embeddings_b200 import _native as N
    from learning_embeddings_b200 import ops

DEV = "cuda"
DIMS = (2, 10, 50)
PRECS = (0, 1)


def t(a, dtype=None):
    x = torch.from_numpy(np.ascontiguousarray(a))
    return x.to(dtype) if dtype is not None else x


def contract(new, ref64, ref32, what, rel=1e-5, floor=2e-6, fp32_core=False):
    """fp32_core=True (LEC_PREC_F32 on the hyperbolic energy): the kernel then does the same class of
    arithmetic as the reference's own FP32 run, whose error against FP64 is O(1e-5) near the acos clamp
    (SURVEY F13); pointwise it may land on the other side of the truth, so the bound also admits 4x the
    reference's own worst FP32 error on the batch."""
    new, ref64, ref32 = (np.asarray(a, dtype=np.float64) for a in (new, ref64, ref32))
    finite = np.isfinite(ref64)
    assert (np.isnan(new) == np.isnan(ref64)).all(), what + ": NaN pattern differs"
    err = np.abs(new - ref64)[finite]
    if fp32_core:
        floor = max(floor, 4 * float(np.abs(ref32 - ref64)[finite].max()))
    bound = np.maximum.reduce([rel * np.abs(ref64), 2 * np.abs(ref32 - ref64), np.full_like(ref64, floor)])[finite]
    bad = err > bound
    assert not bad.any(), "%s: %d/%d outside the contract, worst err %.3e (bound %.3e)" % (
        what, bad.sum(), bad.size, err[bad].max(), bound[bad][err[bad].argmax()])


def contract_rows(new, ref64, ref32, what, rel=1e-5, floor=2e-6, fp32_core=False):
    new, ref64, ref32 = (np.asarray(a, dtype=np.float64) for a in (new, ref64, ref32))
    err = np.linalg.norm(new - ref64, axis=1)
    if fp32_core:
        floor = max(floor, 4 * float(np.linalg.norm(ref32 - ref64, axis=1).max()))
    bound = np.maximum.reduce([rel * np.linalg.norm(ref64, axis=1), 2 * np.linalg.norm(ref32 - ref64, axis=1),
                               np.full(len(err), floor)])
    bad = err > bound
    assert not bad.any(), "%s: %d/%d rows outside the contract, worst err %.3e (bound %.3e)" % (
        what, bad.sum(), bad.size, err[bad].max(), bound[bad][err[bad].argmax()])


def padded(x):
    P, D = x.shape
    ld = ops.padded_dim(D)
    out = torch.zeros(P, ld)
    out[:, :D] = x
    return out


def pair_files():
    out = []
    for D in DIMS:
        for a in ("1p0", "0p05"):
            out.append(("euc", "pairs_euc_D%d_a%s" % (D, a)))
            out.append(("hyp", "pairs_hyp_D%d_a%s" % (D, a)))
        out.append(("oe", "pairs_oe_D%d" % D))
    return out


# ------------------------------------------------------------------------------------------------
# pair kernels vs the reference's golden vectors
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("idx_dtype", (torch.int32, torch.int64))
@pytest.mark.parametrize("geom,name", pair_files())
def test_flat_kernel_matches_reference(geom, name, idx_dtype, prec):
    g = load_golden(name)
    x, y = t(g["x"]), t(g["y"])
    P, D = x.shape
    K, alpha = float(g.get("K", 0.0)), float(g["alpha"])
    rows, aux = ops.rows_forward(torch.cat([x, y]).to(DEV), N.ROWS_NONE, K, geom)
    assert torch.equal(rows.cpu(), torch.cat([padded(x), padded(y)]))
    fi = torch.arange(P, dtype=idx_dtype, device=DEV)
    ti = fi + P
    grad = torch.zeros_like(rows)
    loss, E = ops.pairs_flat_raw(geom, rows, aux, D, fi, ti, K, alpha, w=t(g["w"]).to(DEV),
                                 is_pos=t(g["is_pos"]).to(torch.uint8).to(DEV), grad_rows=grad, precision=prec)
    torch.cuda.synchronize()
    f32c = (geom == "hyp" and prec == 0)
    contract(E.cpu().numpy(), g["E64"], g["E32"], name + " E", fp32_core=f32c)
    assert abs(float(loss) - float(g["L64"])) <= max(1e-5 * abs(float(g["L64"])), 4 * abs(float(g["L32"]) - float(g["L64"])))
    gx, gy = grad[:P, :D].cpu().numpy(), grad[P:, :D].cpu().numpy()
    contract_rows(gx, g["gx64"], g["gx32"], name + " gx", fp32_core=f32c)
    contract_rows(gy, g["gy64"], g["gy32"], name + " gy", fp32_core=f32c)
    if rows.shape[1] > D:
        assert float(grad[:, D:].abs().max()) == 0.0
    # scattering into several gradient replicas gives the same sum
    grad_r = torch.zeros((5,) + tuple(rows.shape), device=DEV)
    ops.pairs_flat_raw(geom, rows, aux, D, fi, ti, K, alpha, w=t(g["w"]).to(DEV),
                       is_pos=t(g["is_pos"]).to(torch.uint8).to(DEV), grad_rows=grad_r, precision=prec)
    scale = float(grad.abs().max())
    np.testing.assert_allclose(ops.reduce_replicas(grad_r).cpu().numpy(), grad.cpu().numpy(), rtol=1e-5, atol=1e-6 * scale)
    # hinge-active sets identical away from ties
    z64 = g["E64"]
    act_new = (np.linalg.norm(gx, axis=1) > 0)
    act_ref = (np.linalg.norm(g["gx64"], axis=1) > 0)
    far = (np.abs(z64) > 1e-5) & (np.abs(alpha - z64) > 1e-5)
    assert (act_new[far] == act_ref[far]).all()


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("geom,name", pair_files())
def test_dense_energy_and_backward_match_reference(geom, name, prec):
    g = load_golden(name)
    K, alpha = float(g.get("K", 0.0)), float(g["alpha"])
    x = t(g["x"]).to(DEV).requires_grad_(True)
    y = t(g["y"]).to(DEV).requires_grad_(True)
    E = ops.energy(x, y, geom, K, prec)
    pos = t(g["is_pos"]).to(DEV).bool()
    w = t(g["w"]).to(DEV)
    loss = (w * E)[pos].sum() + (w * (alpha - E).clamp(min=0))[~pos].sum()
    loss.backward()
    f32c = (geom == "hyp" and prec == 0)
    contract(E.detach().cpu().numpy(), g["E64"], g["E32"], name + " E", fp32_core=f32c)
    contract_rows(x.grad.cpu().numpy(), g["gx64"], g["gx32"], name + " gx", fp32_core=f32c)
    contract_rows(y.grad.cpu().numpy(), g["gy64"], g["gy32"], name + " gy", fp32_core=f32c)


# ------------------------------------------------------------------------------------------------
# row transforms and RSGD vs golden
# ------------------------------------------------------------------------------------------------
ROW_CASES = [("rows_euc", 1, "W"), ("rows_hyp_shell", 2, "W"), ("rows_hyp_tanh", 3, "W"),
             ("feat_euc", 1, "Z"), ("feat_hyp", 4, "Z")]


@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("prefix,mode,key", ROW_CASES)
def test_row_transforms_match_reference(prefix, mode, key, D):
    g = load_golden("%s_D%d" % (prefix, D))
    K = float(g["K"])
    W = t(g[key]).to(DEV).requires_grad_(True)
    rows, _ = ops.transform_rows(W, mode, K)
    assert rows.shape[1] == ops.padded_dim(D)
    if key == "W":
        idx = t(g["idx"]).to(DEV)
        out = rows.index_select(0, idx)[:, :D]
    else:
        out = rows[:, :D]
    out.backward(t(g["G_up"]).to(DEV))
    got = out.detach().cpu().numpy()
    # Rows whose tanh saturates sit exactly on the reference's `norm >= 1.0` projection test
    # (oe_h.py:103): the fp32 rounding of the row norm decides whether the (1 - 1e-5) factor is applied,
    # a tie inside the reference itself.  They may differ by that factor; everything else is tight.
    sat = np.linalg.norm(g["out"], axis=1) >= 1.0 - 2.5e-5
    np.testing.assert_allclose(got[~sat], g["out"][~sat], rtol=3e-6, atol=2e-7)
    np.testing.assert_allclose(got[sat], g["out"][sat], rtol=1.2e-5, atol=2e-7)
    gref = g["gW"] if key == "W" else g["gZ"]
    scale = np.abs(gref).max()
    np.testing.assert_allclose(W.grad.cpu().numpy(), gref, rtol=2e-4, atol=5e-6 * scale)
    if rows.shape[1] > D:
        assert float(rows[:, D:].abs().max()) == 0.0


@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("lr", ("0p001", "0p1"))
def test_rsgd_update_matches_reference(D, lr):
    g = load_golden("rsgd_D%d_lr%s" % (D, lr))
    W = t(g["W"]).to(DEV).clone()
    grad = t(g["grad"]).to(DEV).clone()
    ops.rsgd_update_(W, grad, float(g["lr"]), float(g["r_in"]))
    # the update is fp32 arithmetic of the same class as the reference's: batch-level clause (see contract)
    contract(W.cpu().numpy(), g["W_new64"], g["W_new"], "rsgd W", rel=1e-5, floor=1e-6, fp32_core=True)
    np.testing.assert_allclose(grad.cpu().numpy(), g["rescaled_grad"], rtol=1e-5, atol=0)
    # padded gradient input gives the same update
    W2 = t(g["W"]).to(DEV).clone()
    gp = padded(t(g["grad"])).to(DEV)
    ops.rsgd_update_(W2, gp, float(g["lr"]), float(g["r_in"]))
    assert torch.equal(W, W2)
    # ... and so do gradient replicas that sum to the same gradient
    W3 = t(g["W"]).to(DEV).clone()
    g3 = torch.stack([0.25 * gp, 0.5 * gp, 0.25 * gp])
    ops.rsgd_update_(W3, g3, float(g["lr"]), float(g["r_in"]))
    np.testing.assert_allclose(W3.cpu().numpy(), W.cpu().numpy(), rtol=2e-6, atol=1e-7)


# ------------------------------------------------------------------------------------------------
# full training / eval steps on the ETHEC hierarchy: grouped kernel + row transform + sampler
# ------------------------------------------------------------------------------------------------
STEP_CASES = [
    ("step_euc_D2", "euc", 1), ("step_euc_D2_a0p05", "euc", 1), ("step_euc_D10_ppl", "euc", 1),
    ("step_hyp_D10", "hyp", 2), ("step_hyp_D10_a0p05", "hyp", 2), ("step_hyp_D50_ppl", "hyp", 2),
    ("step_oe_D10", "oe", 0),
]


def _neg_adj(h):
    n = len(h["parents"])
    A = np.ones((n, n), dtype=bool)
    A[h["tc_edges"][:, 0], h["tc_edges"][:, 1]] = False
    np.fill_diagonal(A, False)
    return A


class _LabelMap:
    def __init__(self, h):
        self.levels = h["levels"].tolist()
        self.level_start = h["level_start"].tolist()
        self.level_stop = h["level_stop"].tolist()
        self.level_names = ["family", "subfamily", "genus", "genus_specific_epithet"]
        self.n_classes = int(sum(self.levels))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name,geom,mode", STEP_CASES)
def test_grouped_step_matches_reference(name, geom, mode, prec, ethec):
    g = load_golden(name)
    Nn, K, alpha = int(g["N"]), float(g["K"]), float(g["alpha"])
    B = len(g["u"])
    D = g["W0"].shape[1]
    drawn = g["drawn"].reshape(B, Nn, 2)
    neg_to, neg_from = drawn[:, :, 0].copy(), drawn[:, :, 1].copy()
    W = t(g["W0"]).to(DEV).requires_grad_(True)
    rows, aux = ops.transform_rows(W, mode, K, geom)
    loss, E_pos, E_neg = ops.grouped_pair_loss(rows, aux, D, t(g["u"]).to(DEV), t(g["v"]).to(DEV), t(neg_to).to(DEV),
                                               t(neg_from).to(DEV), Nn, geom, K, alpha, precision=prec)
    loss.backward()
    # ground truth: oracle in fp64 on the same fp32 table; like-for-like: the reference's fp32 golden
    nf = np.concatenate([np.repeat(g["u"][:, None], Nn, 1), neg_from], 1).reshape(-1)
    nt = np.concatenate([neg_to, np.repeat(g["v"][:, None], Nn, 1)], 1).reshape(-1)
    r64 = cones.label_step(geom, t(g["W0"], torch.float64), mode, K, alpha, t(g["u"]), t(g["v"]), t(nf), t(nt))
    f32c = (geom == "hyp" and prec == 0)
    contract(E_pos.cpu().numpy(), r64["E_pos"].numpy(), g["E_pos"], name + " E_pos", fp32_core=f32c)
    contract(E_neg.reshape(-1).cpu().numpy(), r64["E_neg"].numpy(), g["E_neg"], name + " E_neg", fp32_core=f32c)
    assert abs(float(loss) - float(r64["loss"])) <= max(1e-5 * abs(float(r64["loss"])),
                                                       4 * abs(float(g["loss"]) - float(r64["loss"])))
    contract_rows(W.grad.cpu().numpy(), r64["gW"].numpy(), g["gW"], name + " gW", floor=2e-5, fp32_core=f32c)
    np.testing.assert_allclose(rows.index_select(0, t(g["u"]).to(DEV))[:, :D].detach().cpu().numpy(), g["from_emb"],
                               rtol=3e-6, atol=2e-7)
    # the flat kernel on the expanded pair list gives the same numbers
    W2 = t(g["W0"]).to(DEV).requires_grad_(True)
    rows2, aux2 = ops.transform_rows(W2, mode, K, geom)
    fi = torch.cat([t(g["u"]), t(nf)]).to(DEV)
    ti = torch.cat([t(g["v"]), t(nt)]).to(DEV)
    is_pos = torch.cat([torch.ones(B), torch.zeros(len(nf))]).to(torch.uint8).to(DEV)
    loss2, E2 = ops.flat_pair_loss(rows2, aux2, D, fi, ti, geom, K, alpha, is_pos=is_pos, precision=prec)
    loss2.backward()
    np.testing.assert_allclose(E2[:B].cpu().numpy(), E_pos.cpu().numpy(), rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(E2[B:].cpu().numpy(), E_neg.reshape(-1).cpu().numpy(), rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(float(loss2), float(loss), rtol=1e-6)
    scale = float(W.grad.abs().max())
    np.testing.assert_allclose(W2.grad.cpu().numpy(), W.grad.cpu().numpy(), rtol=1e-4, atol=1e-5 * scale)


@pytest.mark.parametrize("name,geom", [("step_euc_D2_a0p05", "euc"), ("step_euc_D10_ppl", "euc"),
                                       ("step_hyp_D10_a0p05", "hyp"), ("step_hyp_D50_ppl", "hyp"),
                                       ("step_oe_D10", "oe"), ("step_oe_D10_weighted", "oe")])
def test_dropin_criterion_reproduces_reference_step(name, geom, ethec):
    """The reference-facing classes: same ctor, same forward signature, bit-exact negatives."""
    from learning_embeddings_b200 import order_embeddings as oe_mod
    from learning_embeddings_b200 import order_embeddings_h as oeh_mod
    import networkx as nx

    g = load_golden(name)
    lm = _LabelMap(ethec)
    Nn, alpha = int(g["N"]), float(g["alpha"])
    D = g["W0"].shape[1]
    ppl = bool(g["pick_per_level"])
    if geom == "euc":
        crit = oe_mod.EucConesLoss(lm, Nn, alpha=alpha, pick_per_level=ppl)
        model = oe_mod.Embedder(D, lm, K=crit.K)
    elif geom == "hyp":
        crit = oeh_mod.EucConesLoss(lm, Nn, alpha=alpha, pick_per_level=ppl)
        model = oeh_mod.Embedder(D, lm, K=crit.K)
    else:
        kw = dict(weigh_neg_term=True, level_weights=t(g["level_weights"])) if bool(g["weigh_neg_term"]) else {}
        crit = oe_mod.OrderEmbeddingLoss(lm, Nn, alpha=alpha, pick_per_level=ppl, **kw)
        model = oe_mod.Embedder(D, lm)
    with torch.no_grad():
        model.embeddings.weight.copy_(t(g["W0"]))
    model = model.to(DEV)
    ident = {i: i for i in range(lm.n_classes)}
    crit.set_negative_graph(_neg_adj(ethec), ident, ident)
    G_tc = nx.DiGraph()
    G_tc.add_nodes_from(range(lm.n_classes))
    G_tc.add_edges_from(ethec["tc_edges"].tolist())
    crit.set_graph_tc(G_tc)
    random.seed(0)
    u, v = g["u"].tolist(), g["v"].tolist()
    status = torch.ones(len(u), dtype=torch.int64)
    from_emb, to_emb, loss, E_pos, E_neg = crit(model, u, v, status, "train", Nn)
    loss.backward()
    nf, nt = crit.last_negatives
    B = len(u)
    drawn = np.stack([nt.reshape(B, 2 * Nn)[:, :Nn], nf.reshape(B, 2 * Nn)[:, Nn:]], axis=2).reshape(-1)
    assert drawn.tolist() == g["drawn"].tolist()  # bit-exact negative indices
    np.testing.assert_allclose(float(loss), float(g["loss"]), rtol=2e-5)
    np.testing.assert_allclose(from_emb.detach().cpu().numpy(), g["from_emb"], rtol=3e-6, atol=2e-7)
    np.testing.assert_allclose(to_emb.detach().cpu().numpy(), g["to_emb"], rtol=3e-6, atol=2e-7)
    gW = model.embeddings.weight.grad.cpu().numpy()
    if not bool(g["weigh_neg_term"]):   # the weighted order-embedding golden keeps the coarse bound below
        # The SURVEY 8(c) contract, pointwise: the golden is the reference's own FP32 run, whose error against the truth
        # is O(1e-5) near the acos clamp, so the drop-in is held to the FP64 oracle on the same pairs -- within 1e-5
        # relative, or within twice the reference's own FP32 error where that is larger.
        mode = {"euc": cones.ROW_EUC_SOFTCLIP, "hyp": cones.ROW_HYP_SHELL, "oe": cones.ROW_NONE}[geom]
        r64 = cones.label_step(geom, t(g["W0"], torch.float64), mode, float(crit.K) if geom != "oe" else 0.0, alpha,
                               t(g["u"]), t(g["v"]), t(nf.reshape(-1)), t(nt.reshape(-1)))
        contract(E_pos.cpu().numpy(), r64["E_pos"].numpy(), g["E_pos"], name + " E_pos")
        contract(E_neg.cpu().numpy().reshape(-1), r64["E_neg"].numpy(), g["E_neg"].reshape(-1), name + " E_neg")
        contract_rows(gW, r64["gW"].numpy(), g["gW"], name + " gW", floor=2e-5)
    else:
        np.testing.assert_allclose(E_pos.cpu().numpy(), g["E_pos"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(E_neg.cpu().numpy(), g["E_neg"], rtol=1e-4, atol=1e-4)
        scale = np.abs(g["gW"]).max()
        np.testing.assert_allclose(gW, g["gW"], rtol=5e-3, atol=1e-4 * scale)
    # eval phase on a mixed-status batch
    with torch.no_grad():
        _, _, ev_loss, ev_Ep, ev_En = crit(model, g["ev_from"].tolist(), g["ev_to"].tolist(), t(g["ev_status"]),
                                           "val", Nn)
    # pairs with identical endpoints are 0/0 in the hyperbolic energy: the reference returns NaN or a
    # clamped angle depending on how its norms round; the kernels return NaN.  Compare everything else.
    same = (g["ev_from"] == g["ev_to"])[g["ev_status"] == 0]
    if geom != "hyp":
        same[:] = False
    got_En = ev_En.cpu().numpy()
    np.testing.assert_allclose(ev_Ep.cpu().numpy(), g["ev_E_pos"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(got_En[~same], g["ev_E_neg"][~same], rtol=1e-4, atol=1e-4)
    assert np.isnan(got_En[same]).all()
    if not same.any():
        np.testing.assert_allclose(float(ev_loss), float(g["ev_loss"]), rtol=2e-5)
    # E_operator on CPU tensors (the reference's reconstruction check does this)
    e_cpu = crit.E_operator(from_emb.detach().cpu(), to_emb.detach().cpu())
    assert not e_cpu.is_cuda
    np.testing.assert_allclose(e_cpu.numpy(), g["E_pos"], rtol=1e-4, atol=1e-4)


def test_hyperbolic_training_step_with_rsgd_matches_reference_update(ethec):
    """criterion -> backward -> rsgd_step, against oracle.rsgd_step on the reference's own gradient."""
    from learning_embeddings_b200 import order_embeddings_h as oeh_mod
    g = load_golden("step_hyp_D10_a0p05")
    lm = _LabelMap(ethec)
    crit = oeh_mod.EucConesLoss(lm, 5, alpha=0.05)
    model = oeh_mod.Embedder(10, lm, K=crit.K)
    with torch.no_grad():
        model.embeddings.weight.copy_(t(g["W0"]))
    model = model.to(DEV)
    ident = {i: i for i in range(lm.n_classes)}
    crit.set_negative_graph(_neg_adj(ethec), ident, ident)
    random.seed(0)
    _, _, loss, _, _ = crit(model, g["u"].tolist(), g["v"].tolist(), torch.ones(len(g["u"]), dtype=torch.int64), "train", 5)
    loss.backward()
    oeh_mod.rsgd_step(model, 0.001, crit.inner_radius)
    _, W_ref = cones.rsgd_step(t(g["W0"]), t(g["gW"]), 0.001, crit.inner_radius)
    np.testing.assert_allclose(model.embeddings.weight.detach().cpu().numpy(), W_ref.numpy(), rtol=1e-4, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# scoring
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("engine", ("simt", "tc"))
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name,geom", [("scoring_hyp_D10", "hyp"), ("scoring_hyp_D50", "hyp"),
                                       ("scoring_euc_D10", "euc"), ("scoring_oe_D10", "oe")])
def test_scoring_matches_reference_loop(name, geom, prec, engine):
    """engine "simt": packed-FMA tile kernel (lec_score_topk_ex); "tc": tcgen05 3xTF32 contraction with the fused
    epilogue (lec_score_topk_tc, hyperbolic + fp32 core only).  Same contract for both."""
    if engine == "tc" and not (geom == "hyp" and prec == 0):
        pytest.skip("the tensor-core path is built for the hyperbolic energy with the fp32 core")
    g = load_golden(name)
    K = float(g["K"])
    idx, val, scores = ops.score_topk(t(g["labels"]).to(DEV), t(g["images"]).to(DEV), geom, K, g["level_start"],
                                      g["level_stop"], k=5, want_scores=True, precision=prec, engine=engine)
    contract(scores.cpu().numpy(), g["E64"], g["E"], name + " scores", fp32_core=(geom == "hyp" and prec == 0))
    tv = g["top_val"]
    contract(val.cpu().numpy(), tv, tv, name + " topk values", floor=5e-6)
    distinct = np.ones_like(tv, dtype=bool)
    gap = (tv[..., 1:] - tv[..., :-1]) > 1e-5
    distinct[..., 1:] &= gap
    distinct[..., :-1] &= gap
    assert (idx.cpu().numpy()[distinct] == g["top_idx"][distinct]).all()  # predicted label sets
    # cones: the zero label row (the reference's off-by-one, SURVEY F9) scores NaN and is never predicted
    if geom != "oe":
        assert not (idx.cpu().numpy() == g["labels"].shape[0] - 1).any()
    # top-k agrees with torch.topk over the kernel's own full score matrix
    ridx, rval = cones.topk_per_level(scores.cpu(), g["level_start"], g["level_stop"], 5)
    np.testing.assert_array_equal(val.cpu().numpy(), rval.numpy())
    # top-k only (no matrix) returns the same values bit for bit (tc: deferred-angle path), and so does matrix only
    idx2, val2, _ = ops.score_topk(t(g["labels"]).to(DEV), t(g["images"]).to(DEV), geom, K, g["level_start"],
                                   g["level_stop"], k=5, want_scores=False, precision=prec, engine=engine)
    if engine == "tc" and g["labels"].shape[1] > 30:
        # wide rows: the matrix + top-k launch contracts all three bilinear forms on the tensor cores, the top-k-only
        # launch one (lec_score_mma.cu, mma_forms) -- two evaluation orders of the same energies
        np.testing.assert_allclose(val2.cpu().numpy(), val.cpu().numpy(), rtol=1e-5, atol=5e-6)
    else:
        assert torch.equal(val2, val)
    assert (idx2.cpu().numpy()[distinct] == g["top_idx"][distinct]).all()


# ------------------------------------------------------------------------------------------------
# size-independent properties at larger sizes + edge cases
# ------------------------------------------------------------------------------------------------
def _ball(gen, n, D, lo, hi):
    d = torch.randn(n, D, generator=gen)
    return d / d.norm(dim=1, keepdim=True) * (lo + (hi - lo) * torch.rand(n, 1, generator=gen))


@pytest.mark.parametrize("geom,D", [("hyp", 10), ("hyp", 50), ("euc", 10), ("oe", 10), ("hyp", 3), ("euc", 129),
                                    ("hyp", 300), ("oe", 1)])
def test_grouped_equals_flat_and_oracle_on_random_tree_batches(geom, D):
    gen = torch.Generator().manual_seed(D)
    n, B, Nn = 2000, 3001, 7
    K = {"euc": 3.0, "hyp": 0.1, "oe": 0.0}[geom]
    mode = {"euc": 1, "hyp": 2, "oe": 0}[geom]
    W = _ball(gen, n, D, 0.1, 0.95) if geom == "hyp" else torch.randn(n, D, generator=gen)
    u = torch.randint(0, n, (B,), generator=gen)
    v = (u + 1 + torch.randint(0, n - 1, (B,), generator=gen)) % n
    neg_to = torch.randint(0, n, (B, Nn), generator=gen)
    neg_from = torch.randint(0, n, (B, Nn), generator=gen)
    neg_to = torch.where(neg_to == u[:, None], (neg_to + 1) % n, neg_to)
    neg_from = torch.where(neg_from == v[:, None], (neg_from + 1) % n, neg_from)
    w_pos = 0.5 + torch.rand(B, generator=gen)
    w_neg = 0.5 + torch.rand(B, 2 * Nn, generator=gen)
    nf = torch.cat([u[:, None].expand(B, Nn), neg_from], 1).reshape(-1)
    nt = torch.cat([neg_to, v[:, None].expand(B, Nn)], 1).reshape(-1)
    ref = cones.label_step(geom, W.double(), mode, K, 0.7, u, v, nf, nt, w_pos=w_pos.double(),
                           w_neg=w_neg.reshape(-1).double())
    ref32 = cones.label_step(geom, W, mode, K, 0.7, u, v, nf, nt, w_pos=w_pos, w_neg=w_neg.reshape(-1))
    for prec in PRECS:
        Wd = W.to(DEV).requires_grad_(True)
        rows, aux = ops.transform_rows(Wd, mode, K, geom)
        loss, E_pos, E_neg = ops.grouped_pair_loss(rows, aux, D, u.to(DEV).int(), v.to(DEV).int(), neg_to.to(DEV).int(),
                                                   neg_from.to(DEV).int(), Nn, geom, K, 0.7, w_pos=w_pos, w_neg=w_neg,
                                                   precision=prec)
        loss.backward()
        f32c = (geom == "hyp" and prec == 0)
        contract(E_pos.cpu().numpy(), ref["E_pos"].numpy(), ref32["E_pos"].numpy(), "E_pos", fp32_core=f32c)
        contract(E_neg.reshape(-1).cpu().numpy(), ref["E_neg"].numpy(), ref32["E_neg"].numpy(), "E_neg", fp32_core=f32c)
        contract_rows(Wd.grad.cpu().numpy(), ref["gW"].numpy(), ref32["gW"].numpy(), "gW", floor=2e-5, fp32_core=f32c)
        assert abs(float(loss) - float(ref["loss"])) <= 1e-5 * abs(float(ref["loss"])) + 2 * abs(
            float(ref32["loss"]) - float(ref["loss"]))


def test_empty_and_degenerate_batches():
    rows, aux = ops.rows_forward(torch.rand(8, 10, device=DEV) * 0.2 + 0.05, N.ROWS_NONE, 0.1, "hyp")
    e = torch.empty(0, dtype=torch.int64, device=DEV)
    loss, E = ops.pairs_flat_raw("hyp", rows, aux, 10, e, e, 0.1, 1.0)
    assert E.numel() == 0 and float(loss) == 0.0
    loss, Ep, En = ops.pairs_grouped_raw("hyp", rows, aux, 10, e, e, e.view(0, 5), e.view(0, 5), 5, 0.1, 1.0)
    assert Ep.numel() == 0 and float(loss) == 0.0
    # N = 0: positives only
    u = torch.tensor([0, 1, 2], device=DEV)
    v = torch.tensor([3, 4, 5], device=DEV)
    grad = torch.zeros_like(rows)
    loss, Ep, En = ops.pairs_grouped_raw("hyp", rows, aux, 10, u, v, e.view(3, 0), e.view(3, 0), 0, 0.1, 1.0, grad_rows=grad)
    ref = cones.energy_hyp(rows[u, :10].cpu().double(), rows[v, :10].cpu().double(), 0.1)
    np.testing.assert_allclose(Ep.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=2e-6)
    assert En.numel() == 0
    # x == y: the reference yields NaN (0/0); so do we
    E = ops.energy(rows[:2, :10].contiguous(), rows[:2, :10].contiguous(), "hyp", 0.1)
    assert torch.isnan(E).all()
    # Euclidean apex inside the K-ball: NaN like the reference (SURVEY F8)
    x = torch.full((1, 4), 0.1, device=DEV)
    y = torch.ones(1, 4, device=DEV)
    assert torch.isnan(ops.energy(x, y, "euc", 3.0)).all()
    assert torch.isnan(cones.energy_euc(x.cpu(), y.cpu(), 3.0)).all()


@pytest.mark.parametrize("engine,D", [("simt", 10), ("tc", 10), ("tc", 50)])
def test_scoring_full_size_properties(engine, D):
    """1 M-image scale is covered by bench.py; here 40 K images x 723 labels: top-k of the kernel equals
    torch.topk of its own score matrix, shards concatenate, and image order does not matter."""
    import functools
    gen = torch.Generator().manual_seed(3)
    h = load_golden("ethec_hierarchy")
    L, n_img = 723, 40000 + 37   # not a multiple of any tile size
    score_topk = functools.partial(ops.score_topk, engine=engine)
    labels = torch.zeros(L, D)
    for l in range(4):
        s, e = int(h["level_start"][l]), int(h["level_stop"][l])
        labels[s:e] = _ball(gen, e - s, D, 0.10 + 0.2 * l, 0.30 + 0.2 * l)
    images = _ball(gen, n_img, D, 0.30, 0.95)
    lab_d, img_d = labels.to(DEV), images.to(DEV)
    idx, val, scores = score_topk(lab_d, img_d, "hyp", 0.1, h["level_start"], h["level_stop"], k=5, want_scores=True)
    ridx, rval = cones.topk_per_level(scores.cpu(), h["level_start"], h["level_stop"], 5)
    np.testing.assert_array_equal(val.cpu().numpy(), rval.numpy())
    # exact ties (also one between the k-th and the (k+1)-th energy) leave the label choice open
    _, rval6 = cones.topk_per_level(scores.cpu(), h["level_start"], h["level_stop"], 6)
    ties = (rval6[..., 1:] == rval6[..., :-1]).any(dim=-1)
    assert (idx.cpu()[~ties] == ridx[~ties].int()).all()
    ref = cones.score_matrix("hyp", labels.double(), images[:512].double(), 0.1)
    ref32 = cones.score_matrix("hyp", labels, images[:512], 0.1)
    contract(scores[:512].cpu().numpy(), ref.numpy(), ref32.numpy(), "scores", fp32_core=True)
    # the top-k-only launch (wide rows on the tensor cores: another evaluation order, see mma_forms) agrees with it
    idx_t, val_t, _ = score_topk(lab_d, img_d, "hyp", 0.1, h["level_start"], h["level_stop"], k=5)
    if engine == "tc" and D > 30:
        np.testing.assert_allclose(val_t.cpu().numpy(), val.cpu().numpy(), rtol=1e-5, atol=5e-6)
    else:
        assert torch.equal(idx_t, idx) and torch.equal(val_t, val)
    # sharding: two halves give the same answer as one call
    i1, v1, _ = score_topk(lab_d, img_d[: n_img // 2], "hyp", 0.1, h["level_start"], h["level_stop"], k=5)
    i2, v2, _ = score_topk(lab_d, img_d[n_img // 2:], "hyp", 0.1, h["level_start"], h["level_stop"], k=5)
    assert torch.equal(torch.cat([i1, i2]), idx_t) and torch.equal(torch.cat([v1, v2]), val_t)
    perm = torch.randperm(n_img, generator=gen).to(DEV)
    ip, vp, _ = score_topk(lab_d, img_d[perm], "hyp", 0.1, h["level_start"], h["level_stop"], k=5)
    assert torch.equal(ip, idx_t[perm]) and torch.equal(vp, val_t[perm])


@pytest.mark.parametrize("engine", ("simt", "tc"))
def test_score_pipeline_host_to_host_equals_device_call(engine):
    """ops.ScorePipeline (sliced, copies overlapped with the kernel) returns exactly what one device call returns."""
    gen = torch.Generator().manual_seed(11)
    h = load_golden("ethec_hierarchy")
    D, n_img = 10, 5000 + 3
    labels = _ball(gen, 723, D, 0.1, 0.9).to(DEV)
    images = _ball(gen, n_img, D, 0.30, 0.95)
    idx, val, _ = ops.score_topk(labels, images.to(DEV), "hyp", 0.1, h["level_start"], h["level_stop"], k=5, engine=engine)
    pipe = ops.ScorePipeline(labels, "hyp", 0.1, h["level_start"], h["level_stop"], k=5, slice_images=1024, engine=engine)
    out_idx = torch.empty((n_img, 4, 5), dtype=torch.int32).pin_memory()
    out_val = torch.empty((n_img, 4, 5), dtype=torch.float32).pin_memory()
    for _ in range(2):   # the second run reuses the slots
        out_idx.fill_(-7)
        pipe.run(images.pin_memory(), out_idx, out_val)
        assert torch.equal(out_idx, idx.cpu()) and torch.equal(out_val, val.cpu())
    out16 = torch.empty((n_img, 4, 5), dtype=torch.int16).pin_memory()   # narrow label ids: half the download
    pipe.run(images.pin_memory(), out16)
    assert torch.equal(out16.int(), idx.cpu())
    with pytest.raises(N.LecError):
        pipe.run(images.to(DEV), out_idx)


# ------------------------------------------------------------------------------------------------
# joint image+label criteria (oe.py / oe_h.py drop-ins)
# ------------------------------------------------------------------------------------------------
class _SmallLabelMap:
    def __init__(self, g):
        self.level_start = g["level_start"].tolist()
        self.level_stop = g["level_stop"].tolist()
        self.levels = [e - s for s, e in zip(self.level_start, self.level_stop)]
        self.level_names = ["family", "subfamily", "genus", "genus_specific_epithet"]
        self.n_classes = int(g["n_lab"])


@pytest.mark.parametrize("name,geom", [("joint_euc", "euc"), ("joint_euc_ppl", "euc"), ("joint_oe", "oe"),
                                       ("joint_hyp", "hyp")])
def test_joint_dropin_reproduces_reference_step(name, geom):
    from learning_embeddings_b200 import oe as oe_mod
    from learning_embeddings_b200 import oe_h as oeh_mod
    g = load_golden(name)
    lm = _SmallLabelMap(g)
    Nn, K, alpha, n_lab, nn_ = int(g["N"]), float(g["K"]), float(g["alpha"]), int(g["n_lab"]), int(g["n_nodes"])
    D, F = g["W0"].shape[1], g["feat"].shape[1]
    A = np.unpackbits(g["neg_adj"], axis=1)[:, :nn_].astype(bool)
    ix2node = {i: (i if i < n_lab else "img_%d" % i) for i in range(nn_)}
    node2ix = {v: k for k, v in ix2node.items()}
    feats = {ix2node[n_lab + i]: g["feat"][i].tolist() for i in range(nn_ - n_lab)}
    ppl = bool(g["pick_per_level"])
    if geom == "euc":
        crit = oe_mod.EuclideanConesWithImagesHypernymLoss(lm, Nn, feats, alpha, pick_per_level=ppl, K=K)
        model, fnet = oe_mod.Embedder(D, lm, None, K=K), oe_mod.FeatNet(None, input_dim=F, output_dim=D, K=K)
    elif geom == "oe":
        crit = oe_mod.OrderEmbeddingWithImagesHypernymLoss(lm, Nn, feats, alpha, pick_per_level=ppl)
        model, fnet = oe_mod.Embedder(D, lm, None, K=None), oe_mod.FeatNet(None, input_dim=F, output_dim=D, K=None)
    else:
        crit = oeh_mod.EuclideanConesWithImagesHypernymLoss(lm, Nn, feats, alpha, pick_per_level=ppl, K=K)
        model, fnet = oeh_mod.Embedder(D, lm, None, K=K), oeh_mod.FeatNet(None, input_dim=F, output_dim=D, K=K)
    with torch.no_grad():
        model.embeddings.weight.copy_(t(g["W0"]))
        fnet.fc1.weight.copy_(t(g["fc_w"]))
        fnet.fc1.bias.copy_(t(g["fc_b"]))
    model, fnet = model.to(DEV), fnet.to(DEV)
    crit.set_negative_graph(A, node2ix, ix2node)
    b_from = [ix2node[int(i)] for i in g["b_from"]]
    b_to = [ix2node[int(i)] for i in g["b_to"]]
    random.seed(0)
    loss, E_pos, E_neg = crit(model, fnet, b_from, b_to, b_from, b_to, torch.ones(len(b_from), dtype=torch.int64), "train")
    loss.backward()
    nf, nt = crit.last_negatives
    B = len(b_from)
    drawn = []
    for i in range(B):
        for p in range(Nn):
            drawn += [node2ix[nt[2 * Nn * i + p]], node2ix[nf[2 * Nn * i + Nn + p]]]
    assert drawn == g["drawn"].tolist()  # bit-exact negative indices, labels and images
    assert tuple(E_neg.shape) == (B, 2 * Nn, 1) and tuple(E_pos.shape) == (B,)
    np.testing.assert_allclose(E_pos.cpu().numpy(), g["E_pos"].reshape(-1), rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(E_neg.reshape(-1).cpu().numpy(), g["E_neg"].reshape(-1), rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(float(loss), float(g["loss"]), rtol=2e-5)
    for got, key in ((model.embeddings.weight.grad, "gW"), (fnet.fc1.weight.grad, "g_fc_w"), (fnet.fc1.bias.grad, "g_fc_b")):
        scale = np.abs(g[key]).max()
        np.testing.assert_allclose(got.cpu().numpy(), g[key], rtol=2e-3, atol=5e-5 * scale)


# ------------------------------------------------------------------------------------------------
# step engine (lec_cone_step: the whole step in one library call)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,geom,mode", [("step_hyp_D10_a0p05", "hyp", 2), ("step_hyp_D50_ppl", "hyp", 2),
                                            ("step_euc_D10_ppl", "euc", 1)])
def test_engine_step_matches_oracle(name, geom, mode):
    from learning_embeddings_b200.engine import ConeStep, pack_index_block
    g = load_golden(name)
    Nn, K, alpha = int(g["N"]), float(g["K"]), float(g["alpha"])
    B = len(g["u"])
    drawn = g["drawn"].reshape(B, Nn, 2)
    neg_to, neg_from = drawn[:, :, 0].copy(), drawn[:, :, 1].copy()
    nf = np.concatenate([np.repeat(g["u"][:, None], Nn, 1), neg_from], 1).reshape(-1)
    nt = np.concatenate([neg_to, np.repeat(g["v"][:, None], Nn, 1)], 1).reshape(-1)
    r64 = cones.label_step(geom, t(g["W0"], torch.float64), mode, K, alpha, t(g["u"]), t(g["v"]), t(nf), t(nt))
    lr = 0.01
    table = t(g["W0"]).to(DEV).clone()
    update = "rsgd" if geom == "hyp" else "none"
    eng = ConeStep(table, geom, Nn, B, K=K, alpha=alpha, lr=lr, update=update)
    eng.write_grad_table = True    # keep the gradient the update rule saw (what the reference leaves in weight.grad)
    blk = pack_index_block(g["u"], g["v"], neg_to, neg_from, n_rows=table.shape[0])
    loss = eng.step_host(blk, B)   # H2D of the index block, fused step, loss read-back
    assert abs(loss - float(r64["loss"])) <= 1e-5 * abs(float(r64["loss"]))
    contract(eng.E_pos.cpu().numpy(), r64["E_pos"].numpy(), g["E_pos"], name + " E_pos")
    contract(eng.E_neg.reshape(-1).cpu().numpy(), r64["E_neg"].numpy(), g["E_neg"], name + " E_neg")
    if geom == "hyp":
        _, W_ref = cones.rsgd_step(t(g["W0"], torch.float64), r64["gW"], lr, cones.inner_radius(K))
        np.testing.assert_allclose(table.cpu().numpy(), W_ref.numpy(), rtol=2e-5, atol=2e-7)
        # the Riemannian gradient is left in grad_table like the reference leaves it in weight.grad
        rg, _ = cones.rsgd_step(t(g["W0"], torch.float64), r64["gW"], lr, cones.inner_radius(K))
        scale = float(rg.abs().max())
        np.testing.assert_allclose(eng.grad_table.cpu().numpy(), rg.numpy(), rtol=1e-3, atol=1e-5 * scale)
    else:
        contract_rows(eng.grad_table.cpu().numpy(), r64["gW"].numpy(), g["gW"], name + " gW", floor=2e-5)
        assert torch.equal(table.cpu(), t(g["W0"]))
    # a second step through the per-kernel path gives the same numbers as the fused call
    t2 = t(g["W0"]).to(DEV).clone()
    e2 = ConeStep(t2, geom, Nn, B, K=K, alpha=alpha, lr=lr, update=update)
    d = blk.to(DEV)
    e2.forward_backward(*e2._split(d, B))
    e2.reduce_and_update()
    np.testing.assert_allclose(e2.E_neg.cpu().numpy(), eng.E_neg.cpu().numpy(), rtol=0, atol=0)
    np.testing.assert_allclose(t2.cpu().numpy(), table.cpu().numpy(), rtol=1e-5, atol=1e-7)


def test_engine_step_at_wordnet_scale_matches_fp64_oracle():
    """BASELINE config 5 shape: 82 115 rows x 50 (17 MB table, int32 indices, ONE gradient replica, groups split over
    several teams because 2 569 positives cannot fill the GPU), 50 negatives per edge.  One fused step against the fp64
    oracle: pointwise energy contract, loss, and every row of the updated table (touched or not: the reference's RSGD
    moves all rows, SURVEY F5)."""
    from learning_embeddings_b200.engine import ConeStep, pack_index_block
    gen = torch.Generator().manual_seed(82115)
    n, D, B, Nn, K, alpha, lr = 82115, 50, 2569, 25, 0.1, 0.05, 0.01
    r_in = cones.inner_radius(K)
    d = torch.randn(n, D, generator=gen)
    W0 = d / d.norm(dim=1, keepdim=True) * (r_in + 0.02 + 0.7 * torch.rand(n, 1, generator=gen))
    u = torch.randint(0, n, (B,), generator=gen)
    v = (u + 1 + torch.randint(0, n - 1, (B,), generator=gen)) % n
    neg_to = torch.randint(0, n, (B, Nn), generator=gen)
    neg_from = torch.randint(0, n, (B, Nn), generator=gen)
    neg_to = torch.where(neg_to == u[:, None], (neg_to + 1) % n, neg_to)
    neg_from = torch.where(neg_from == v[:, None], (neg_from + 1) % n, neg_from)
    # a few hub rows shared by many groups: same-address reductions into the single replica
    u[:200] = u[0]
    neg_to = torch.where(neg_to == u[:, None], (neg_to + 1) % n, neg_to)
    nf = torch.cat([u[:, None].expand(B, Nn), neg_from], 1).reshape(-1)
    nt = torch.cat([neg_to, v[:, None].expand(B, Nn)], 1).reshape(-1)
    r64 = cones.label_step("hyp", W0.double(), cones.ROW_HYP_SHELL, K, alpha, u, v, nf, nt)
    r32 = cones.label_step("hyp", W0, cones.ROW_HYP_SHELL, K, alpha, u, v, nf, nt)
    table = W0.to(DEV).clone()
    eng = ConeStep(table, "hyp", Nn, B, K=K, alpha=alpha, lr=lr)
    assert eng.replicas == 1
    blk = pack_index_block(u.numpy(), v.numpy(), neg_to.numpy(), neg_from.numpy(), n_rows=n)
    assert blk.dtype == torch.int32
    loss = eng.step_host(blk, B)
    assert abs(loss - float(r64["loss"])) <= 1e-5 * abs(float(r64["loss"]))
    contract(eng.E_pos.cpu().numpy(), r64["E_pos"].numpy(), r32["E_pos"].numpy(), "E_pos at 82K x 50")
    contract(eng.E_neg.reshape(-1).cpu().numpy(), r64["E_neg"].numpy(), r32["E_neg"].numpy(), "E_neg at 82K x 50")
    _, W_ref = cones.rsgd_step(W0.double(), r64["gW"], lr, r_in)
    np.testing.assert_allclose(table.cpu().numpy(), W_ref.numpy(), rtol=2e-5, atol=2e-7)
    assert N.index_errors(torch.device(DEV)) == 0


@pytest.mark.parametrize("D", (2, 10, 50))
def test_fused_step_equals_three_launch_step_after_invalidate_rows(D):
    """lec_cone_step with fused = 1 (pairs -> lec_update_rows: update + the next step's Embedder.forward in one launch)
    must leave the same tables and losses as the three-launch step (lec_rows_fwd first, which invalidate_rows() asks
    for), and the same rows / aperture terms as a separate lec_rows_fwd of the updated table."""
    from learning_embeddings_b200.engine import ConeStep, pack_index_block
    from learning_embeddings_b200 import hierarchy
    ethec = hierarchy.ethec()
    rng = np.random.default_rng(17)
    Nn, B = 5, 3000
    edges = ethec.closure_edges()
    gen = torch.Generator().manual_seed(4)
    w = torch.randn(ethec.n, D, generator=gen)
    w = w / w.norm(dim=1, keepdim=True) * (0.05 + 0.9 * torch.rand(ethec.n, 1, generator=gen))   # some rows inside r_in
    tabs = [w.to(DEV).clone() for _ in range(2)]
    engs = [ConeStep(tab, "hyp", Nn, B, K=0.1, alpha=0.05, lr=0.01) for tab in tabs]

    def step_both(blk):
        engs[1].invalidate_rows()   # every step of the second engine is the three-launch step
        return [e.step_host(blk, B) for e in engs]

    for step in range(4):
        sel = rng.integers(0, len(edges), size=B)
        u, v = edges[sel, 0], edges[sel, 1]
        neg_to, neg_from = ethec.sample_negatives(u, v, Nn, rng)
        blk = pack_index_block(u, v, neg_to, neg_from)
        losses = step_both(blk)
        # the gradient scatter uses fp32 L2 reductions, whose order differs from launch to launch: two runs of the SAME
        # step agree to ~1e-5 on the table, not bit for bit -- that is the resolution of this comparison
        assert np.isfinite(losses[0]) and abs(losses[0] - losses[1]) <= 1e-6 * abs(losses[1])
        assert float((tabs[0] - tabs[1]).abs().max()) < 5e-5
        np.testing.assert_allclose(engs[0].E_neg.cpu().numpy(), engs[1].E_neg.cpu().numpy(), rtol=0, atol=2e-3)
    assert engs[0]._struct.fused == 1 and engs[1]._struct.fused == 0
    # the fused engine already holds the rows of the NEXT step: what a separate lec_rows_fwd of its table gives
    rows, aux = ops.rows_forward(tabs[0], N.ROWS_HYP_SHELL, 0.1, geom="hyp")
    # (the two kernels reduce a row's norm over different team widths, so a row sitting exactly on the inner shell can
    # differ by one fp32 rounding)
    np.testing.assert_allclose(engs[0].rows.cpu().numpy(), rows.cpu().numpy(), rtol=1e-6, atol=0)
    np.testing.assert_allclose(engs[0].aux.cpu().numpy(), aux.cpu().numpy(), rtol=2e-6, atol=0)
    assert float(engs[0].grad_rows.abs().max()) == 0.0
    # an outside change of the table must be announced
    with torch.no_grad():
        tabs[0].mul_(0.5)
        tabs[1].copy_(tabs[0])
    engs[0].invalidate_rows()
    losses = step_both(blk)
    assert abs(losses[0] - losses[1]) <= 1e-6 * abs(losses[1]) and float((tabs[0] - tabs[1]).abs().max()) < 5e-5


@pytest.mark.parametrize("idx_np", (np.uint16, np.int32))
def test_pipelined_host_steps_equal_synchronous_steps(idx_np):
    """ConeStep.submit_host/drain (copy of step i+1 overlapping step i, uint16 or int32 index blocks) must leave the
    same table and return the same losses as step_host called step by step."""
    from learning_embeddings_b200.engine import ConeStep, pack_index_block
    from learning_embeddings_b200 import hierarchy
    ethec = hierarchy.ethec()
    rng = np.random.default_rng(5)
    Nn, B, D = 5, 4096, 10
    edges = ethec.closure_edges()
    blocks = []
    for _ in range(5):
        sel = rng.integers(0, len(edges), size=B)
        u, v = edges[sel, 0], edges[sel, 1]
        neg_to, neg_from = ethec.sample_negatives(u, v, Nn, rng)
        blocks.append(pack_index_block(u, v, neg_to, neg_from, dtype=idx_np))
    g = torch.Generator().manual_seed(3)
    w = torch.randn(ethec.n, D, generator=g)
    W0 = (cones.inner_radius(0.1) + 0.05 * torch.rand(ethec.n, 1, generator=g)) * w / w.norm(dim=1, keepdim=True)
    ta, tb = W0.to(DEV).clone(), W0.to(DEV).clone()
    ea = ConeStep(ta, "hyp", Nn, B, K=0.1, alpha=0.05, lr=0.01)
    eb = ConeStep(tb, "hyp", Nn, B, K=0.1, alpha=0.05, lr=0.01)
    sync_losses = [ea.step_host(b, B) for b in blocks]
    for b in blocks:
        eb.submit_host(b, B)
    pipe_losses = eb.drain()
    assert len(pipe_losses) == len(blocks) and eb.drain() == []
    # fp32 vector reductions into the gradient replicas are not order-deterministic: tolerance, not equality
    np.testing.assert_allclose(pipe_losses, sync_losses, rtol=1e-6)
    np.testing.assert_allclose(tb.cpu().numpy(), ta.cpu().numpy(), rtol=1e-4, atol=2e-5)
    # the int64 reference layout gives the same first-step energies as the narrow block
    tc = W0.to(DEV).clone()
    ec = ConeStep(tc, "hyp", Nn, B, K=0.1, alpha=0.05, lr=0.01)
    ec.step_device(*ec._split(torch.from_numpy(blocks[0].numpy().astype(np.int64)).to(DEV), B))
    ed = ConeStep(W0.to(DEV).clone(), "hyp", Nn, B, K=0.1, alpha=0.05, lr=0.01)
    ed.step_host(blocks[0], B)
    assert torch.equal(ec.E_neg, ed.E_neg) and torch.equal(ec.E_pos, ed.E_pos)


@pytest.mark.parametrize("name,geom", [("joint_euc", "euc"), ("joint_oe", "oe"), ("joint_hyp", "hyp")])
def test_joint_engine_step_matches_reference_gradients(name, geom):
    """engine.JointConeStep (gather -> fc1 -> row transforms -> fused pair kernel -> VJPs -> fc1 gradients) against the
    reference's loss, energies and the three parameter gradients of the same step (golden, from oe.py / oe_h.py)."""
    from learning_embeddings_b200.engine import JointConeStep, pack_index_block
    g = load_golden(name)
    Nn, K, alpha, n_lab = int(g["N"]), float(g["K"]), float(g["alpha"]), int(g["n_lab"])
    B = len(g["b_from"])
    drawn = g["drawn"].reshape(B, Nn, 2)
    neg_to, neg_from = drawn[:, :, 0].copy(), drawn[:, :, 1].copy()
    m = g["feat"].shape[0]
    table, fw, fb = (t(g[k]).to(DEV).clone() for k in ("W0", "fc_w", "fc_b"))
    feats = t(g["feat"]).to(DEV)
    eng = JointConeStep(table, fw, fb, feats, geom, Nn, B, m, K=K if geom != "oe" else None, alpha=alpha, lr=1e-3,
                        update="none")
    blk = pack_index_block(g["b_from"], g["b_to"], neg_to, neg_from, dtype=np.uint16, n_rows=n_lab + m)
    loss = eng.step_host(torch.arange(m, dtype=torch.int64), blk, B)
    np.testing.assert_allclose(loss, float(g["loss"]), rtol=2e-5)
    np.testing.assert_allclose(eng.E_pos.cpu().numpy(), g["E_pos"].reshape(-1), rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(eng.E_neg.reshape(-1).cpu().numpy(), g["E_neg"].reshape(-1), rtol=2e-5, atol=2e-5)
    for got, key in ((eng.g_table, "gW"), (eng.g_w, "g_fc_w"), (eng.g_b, "g_fc_b")):
        scale = np.abs(g[key]).max()
        np.testing.assert_allclose(got.cpu().numpy(), g[key], rtol=2e-3, atol=5e-5 * scale)
    # update="none": parameters untouched, gradients only
    assert torch.equal(table.cpu(), t(g["W0"])) and torch.equal(eng.fc_w.cpu(), t(g["fc_w"]))
    assert n_lab == table.shape[0]
    # the fused FeatNet projection equals the stock linear layer
    Y_ref = torch.nn.functional.linear(feats, fw, fb)
    np.testing.assert_allclose(eng.Y[:m].cpu().numpy(), Y_ref.cpu().numpy(), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("name,geom,update", [("joint_upd_euc", "euc", "adam"), ("joint_upd_hyp", "hyp", "adam"),
                                              ("joint_upd_hyp_rsgd", "hyp", "rsgd")])
def test_joint_engine_updates_match_reference_training_iterations(name, geom, update):
    """Three consecutive training iterations of the reference's joint trainers INCLUDING the parameter update
    (oe.py:1505-1524; oe_h.py:1755-1771 default branch and use_rsgd branch; goldens from the unmodified reference):
    losses and all three parameter tensors after every iteration."""
    from learning_embeddings_b200.engine import JointConeStep, pack_index_block
    g = load_golden(name)
    Nn, K, alpha, n_lab, steps = int(g["N"]), float(g["K"]), float(g["alpha"]), int(g["n_lab"]), int(g["steps"])
    m = g["feat"].shape[0]
    B = len(g["b_from0"])
    table, fw, fb = (t(g[k]).to(DEV).clone() for k in ("W0", "fc_w0", "fc_b0"))
    eng = JointConeStep(table, fw, fb, t(g["feat"]).to(DEV), geom, Nn, B, m, K=K, alpha=alpha, lr=float(g["lr_labels"]),
                        lr_fc=float(g["lr_fc"]), update=update)
    lr_max = max(float(g["lr_labels"]), float(g["lr_fc"]))
    for k in range(steps):
        drawn = g["drawn%d" % k].reshape(B, Nn, 2)
        blk = pack_index_block(g["b_from%d" % k], g["b_to%d" % k], drawn[:, :, 0].copy(), drawn[:, :, 1].copy(),
                               dtype=np.uint16, n_rows=n_lab + m)
        loss = eng.step_host(torch.arange(m, dtype=torch.int64), blk, B)
        np.testing.assert_allclose(loss, float(g["loss%d" % k]), rtol=5e-5, err_msg="loss of iteration %d" % k)
        for got, key in ((table, "W"), (eng.fc_w, "fc_w"), (eng.fc_b, "fc_b")):
            a, b = got.cpu().numpy(), g["%s%d" % (key, k + 1)]
            # Adam moves an element by ~lr * sign(g) whatever |g| is: an element whose gradient cancels to rounding noise
            # may land elsewhere when the fp32 summation order differs -- tight bound on the bulk, count on the rest
            far = np.abs(a - b) > 2e-6 + 5e-5 * np.abs(b)
            assert far.mean() <= 0.002 and np.abs(a - b).max() <= 2.5 * lr_max * (k + 1), (key, k, far.sum(), np.abs(a - b).max())
