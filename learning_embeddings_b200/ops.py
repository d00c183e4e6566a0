"""torch-facing operators over the C ABI (include/lec_b200.h).

Everything here is thin plumbing: allocate outputs with torch, pass raw device pointers and the
current CUDA stream to liblec_b200.so.  The autograd Functions follow the scheme of SURVEY.md 8b:
the fused kernels produce d loss / d rows in the forward launch; backward only scales it by the
incoming gradient of the scalar loss.
"""
import ctypes

import torch

from . import _native as N
from ._native import GEOM, PREC_F32, PREC_F64CORE  # noqa: F401  (re-exported)


def default_replicas(n_rows, ld):
    """How many private copies of the gradient table the pair kernels scatter into.

    Same-address L2 reductions serialise, so a small hot table (ETHEC: 723 rows) is replicated; a big
    table (82 K rows) has little per-address contention and stays single.  Budget: 2 M floats, at most 8 copies
    (r1g sweep: 4..32 replicas differ by < 2 us in the pair kernel; 8 keeps the update short)."""
    return int(max(1, min(8, (2 << 20) // max(1, int(n_rows) * int(ld)))))


def reduce_replicas(grad_rows):
    """[R, n, ld] -> [n, ld] (lec_reduce_replicas)."""
    R = grad_rows.shape[0]
    if R == 1:
        return grad_rows[0]
    out = torch.empty_like(grad_rows[0])
    N.check(N.lib().lec_reduce_replicas(N._p(grad_rows), R, out.numel(), N._p(out), N.stream_ptr(out.device)),
            "lec_reduce_replicas")
    return out


def padded_dim(D):
    """Row stride of the transformed table: D rounded up to a multiple of 4 floats (16-byte chunks)."""
    return (int(D) + 3) // 4 * 4


def _idx(t, device):
    if not torch.is_tensor(t):
        t = torch.as_tensor(t)
    if t.dtype not in (torch.int32, torch.int64):
        t = t.to(torch.int64)
    if t.device != device:
        t = t.to(device, non_blocking=True)
    return t.contiguous()


def _f32(t, device):
    if t is None:
        return None
    if not torch.is_tensor(t):
        t = torch.as_tensor(t, dtype=torch.float32)
    return t.to(device=device, dtype=torch.float32, non_blocking=True).contiguous()


# --------------------------------------------------------------------------------------------------
# Row transforms
# --------------------------------------------------------------------------------------------------
def rows_forward(W, mode, K, geom=None, zero_out=None):
    """Transformed table [n, ld] of the raw parameter rows W [n, D], plus (when `geom` is given) the
    per-row aperture terms aux [n, 4] float64 the pair kernels consume (lec_rows_fwd)."""
    N.require_cuda(W)
    W = W.detach().contiguous().float()
    n, D = W.shape
    ld = padded_dim(D)
    rows = torch.empty((n, ld), device=W.device, dtype=torch.float32)
    aux = torch.empty((n, 4), device=W.device, dtype=torch.float64) if geom is not None else None
    zr = 0 if zero_out is None else (zero_out.shape[0] if zero_out.dim() == 3 else 1)
    N.check(N.lib().lec_rows_fwd(N._p(W), n, D, int(mode), GEOM[geom] if geom is not None else 0, float(K or 0.0),
                                 N._p(rows), ld, N._p(aux), N._p(zero_out), zr, 0, N._p(None), N.stream_ptr(W.device)),
            "lec_rows_fwd")
    return rows, aux


def rows_backward(W, grad_rows, mode, K, out=None, accumulate=False):
    """grad wrt the raw rows W [n, D] from grad wrt the transformed rows [n, ld] or [R, n, ld] (lec_rows_bwd)."""
    N.require_cuda(W, grad_rows)
    W = W.detach().contiguous().float()
    grad_rows = grad_rows.contiguous()
    R = grad_rows.shape[0] if grad_rows.dim() == 3 else 1
    n, D = W.shape
    if out is None:
        out = torch.empty((n, D), device=W.device, dtype=torch.float32)
        accumulate = False
    N.check(N.lib().lec_rows_bwd(N._p(W), N._p(grad_rows), R, 0, n, D, grad_rows.shape[-1], int(mode), float(K or 0.0),
                                 N._p(out), int(bool(accumulate)), N.stream_ptr(W.device)), "lec_rows_bwd")
    return out


class RowTransform(torch.autograd.Function):
    """rows, aux = transform(W); rows is differentiable (straight-through where the reference is), aux
    (the per-row aperture terms of energy `geom`) is a by-product of the same launch."""

    @staticmethod
    def forward(ctx, W, mode, K, geom):
        ctx.mode, ctx.K = int(mode), float(K or 0.0)
        ctx.save_for_backward(W)
        rows, aux = rows_forward(W, mode, K, geom)
        if aux is None:
            aux = torch.empty((0, 4), device=W.device, dtype=torch.float64)
        ctx.mark_non_differentiable(aux)
        return rows, aux

    @staticmethod
    def backward(ctx, grad_rows, _grad_aux):
        (W,) = ctx.saved_tensors
        return rows_backward(W, grad_rows, ctx.mode, ctx.K), None, None, None


def transform_rows(W, mode, K, geom=None):
    """-> (rows [n, ld], aux [n, 4] float64 or an empty tensor when geom is None)."""
    return RowTransform.apply(W, mode, K, geom)


# --------------------------------------------------------------------------------------------------
# Pair losses on gathered rows
# --------------------------------------------------------------------------------------------------
def _aux_ptr(geom, aux):
    if aux is None or aux.numel() == 0:
        if geom != "oe":
            raise N.LecError("the %s energy needs the per-row aux terms (transform_rows(..., geom=%r))" % (geom, geom))
        return N._p(None)
    return N._p(aux)


def pairs_grouped_raw(geom, rows, aux, D, pos_from, pos_to, neg_to, neg_from, n_neg, K, alpha, w_pos=None, w_neg=None,
                      grad_rows=None, loss_out=None, precision=PREC_F64CORE, E_pos=None, E_neg=None):
    """Direct call of lec_pairs_grouped on preallocated buffers (used by the step engine and bench)."""
    dev = rows.device
    B = int(pos_from.numel())
    if E_pos is None:
        E_pos = torch.empty(B, device=dev, dtype=torch.float32)
    if E_neg is None:
        E_neg = torch.empty((B, 2 * n_neg), device=dev, dtype=torch.float32)
    if loss_out is None:
        loss_out = torch.zeros(1, device=dev, dtype=torch.float64)
    R = 1 if grad_rows is None or grad_rows.dim() == 2 else grad_rows.shape[0]
    N.check(N.lib().lec_pairs_grouped(
        GEOM[geom], int(precision), N._p(rows), _aux_ptr(geom, aux), rows.shape[0], int(D), rows.shape[1],
        N._p(pos_from), N._p(pos_to),
        N._p(neg_to), N._p(neg_from), pos_from.element_size(), B, int(n_neg), N._p(w_pos), N._p(w_neg),
        float(K or 0.0), float(alpha), N._p(E_pos), N._p(E_neg), N._p(loss_out), N._p(grad_rows), R,
        N.stream_ptr(dev)), "lec_pairs_grouped")
    return loss_out, E_pos, E_neg


class GroupedPairLoss(torch.autograd.Function):
    """loss, E_pos[B], E_neg[B, 2N] for the training layout (include/lec_b200.h: lec_pairs_grouped)."""

    @staticmethod
    def forward(ctx, rows, aux, D, pos_from, pos_to, neg_to, neg_from, n_neg, w_pos, w_neg, geom, K, alpha, precision):
        N.require_cuda(rows)
        dev = rows.device
        rows_c = rows.detach().contiguous()
        pos_from, pos_to = _idx(pos_from, dev), _idx(pos_to, dev)
        neg_to, neg_from = _idx(neg_to, dev), _idx(neg_from, dev)
        if not (pos_from.dtype == pos_to.dtype == neg_to.dtype == neg_from.dtype):
            pos_from, pos_to, neg_to, neg_from = (t.to(torch.int64) for t in (pos_from, pos_to, neg_to, neg_from))
        need_grad = ctx.needs_input_grad[0]
        grad_rows = None
        if need_grad:
            grad_rows = torch.zeros((default_replicas(*rows_c.shape),) + tuple(rows_c.shape), device=dev)
        loss64, E_pos, E_neg = pairs_grouped_raw(geom, rows_c, aux, D, pos_from, pos_to, neg_to, neg_from, n_neg, K, alpha,
                                                 _f32(w_pos, dev), _f32(w_neg, dev), grad_rows, None, precision)
        if need_grad:
            grad_rows = reduce_replicas(grad_rows)
        ctx.save_for_backward(grad_rows)
        ctx.mark_non_differentiable(E_pos, E_neg)
        return loss64[0].float(), E_pos, E_neg

    @staticmethod
    def backward(ctx, g_loss, _gp, _gn):
        (grad_rows,) = ctx.saved_tensors
        return (grad_rows * g_loss,) + (None,) * 13


def grouped_pair_loss(rows, aux, D, pos_from, pos_to, neg_to, neg_from, n_neg, geom, K, alpha, w_pos=None, w_neg=None,
                      precision=PREC_F64CORE):
    return GroupedPairLoss.apply(rows, aux, D, pos_from, pos_to, neg_to, neg_from, n_neg, w_pos, w_neg, geom, K, alpha,
                                 precision)


def _softmax_loss_forward(ctx, entry, rows, D, pos_from, pos_to, neg_to):
    """forward of PoincareLoss / LorentzLoss: one launch of `entry` (lec_pairs_poincare or lec_pairs_lorentz)."""
    N.require_cuda(rows)
    dev = rows.device
    n, width = rows.shape
    if width < D:
        raise N.LecError("%s_loss: rows have %d columns, D = %d" % (entry[len("lec_pairs_"):], width, D))
    ld = padded_dim(D)
    padded = torch.zeros((n, ld), device=dev, dtype=torch.float32)
    padded[:, :D] = rows.detach()[:, :D]
    pos_from, pos_to, neg_to = _idx(pos_from, dev), _idx(pos_to, dev), _idx(neg_to, dev)
    if not (pos_from.dtype == pos_to.dtype == neg_to.dtype):
        pos_from, pos_to, neg_to = (t.to(torch.int64) for t in (pos_from, pos_to, neg_to))
    B = int(pos_from.numel())
    n_neg = int(neg_to.numel()) // max(B, 1)
    E_pos = torch.empty(B, device=dev, dtype=torch.float32)
    E_neg = torch.empty((B, n_neg), device=dev, dtype=torch.float32)
    loss64 = torch.zeros(1, device=dev, dtype=torch.float64)
    grad_rows = None
    if ctx.needs_input_grad[0]:
        grad_rows = torch.zeros((default_replicas(n, ld), n, ld), device=dev)
    N.check(getattr(N.lib(), entry)(
        PREC_F64CORE, N._p(padded), n, int(D), ld, N._p(pos_from), N._p(pos_to), N._p(neg_to),
        pos_from.element_size(), B, n_neg, N._p(E_pos), N._p(E_neg), N._p(loss64), N._p(grad_rows),
        1 if grad_rows is None else grad_rows.shape[0], N.stream_ptr(dev)), entry)
    grad = None
    if grad_rows is not None:
        grad = torch.zeros_like(rows, dtype=torch.float32)
        grad[:, :D] = reduce_replicas(grad_rows)[:, :D]
    ctx.save_for_backward(grad)
    ctx.mark_non_differentiable(E_pos, E_neg)
    return loss64[0], E_pos, E_neg


class PoincareLoss(torch.autograd.Function):
    """loss, E_pos[B], E_neg[B, N] of Nickel & Kiela's softmax loss on the Poincare distance (lec_pairs_poincare)."""

    @staticmethod
    def forward(ctx, rows, D, pos_from, pos_to, neg_to):
        return _softmax_loss_forward(ctx, "lec_pairs_poincare", rows, D, pos_from, pos_to, neg_to)

    @staticmethod
    def backward(ctx, g_loss, _gp, _gn):
        (grad,) = ctx.saved_tensors
        return (grad * g_loss.float(),) + (None,) * 4


class LorentzLoss(torch.autograd.Function):
    """loss, E_pos[B], E_neg[B, N] of Nickel & Kiela's softmax loss on the Lorentz distance (lec_pairs_lorentz)."""

    @staticmethod
    def forward(ctx, rows, D, pos_from, pos_to, neg_to):
        return _softmax_loss_forward(ctx, "lec_pairs_lorentz", rows, D, pos_from, pos_to, neg_to)

    @staticmethod
    def backward(ctx, g_loss, _gp, _gn):
        (grad,) = ctx.saved_tensors
        return (grad * g_loss.float(),) + (None,) * 4


def poincare_loss(rows, D, pos_from, pos_to, neg_to):
    """Nickel & Kiela's loss sum_i [d(u_i, v_i) + log sum_{w in {v_i} + neg_to[i]} exp(-d(u_i, w))] on the Poincare
    distance, for use outside the step engine.  rows [n, >= D] are points inside the unit ball (fp32 CUDA); pos_from,
    pos_to [B] and neg_to [B, N] are row ids.  Returns (loss as a float64 scalar, E_pos [B], E_neg [B, N]); the loss is
    differentiable with respect to rows (fp64 pair algebra, gradient computed in the forward launch)."""
    return PoincareLoss.apply(rows, D, pos_from, pos_to, neg_to)


def lorentz_loss(rows, D, pos_from, pos_to, neg_to):
    """The loss of poincare_loss on the Lorentz distance d = arcosh(1 + w), w = -<X,Y>_L - 1 (Nickel & Kiela 2018).
    rows [n, >= D] are the spatial parts x of hyperboloid points (sqrt(1 + |x|^2), x) (fp32 CUDA, any values); the
    other arguments and the results are those of poincare_loss."""
    return LorentzLoss.apply(rows, D, pos_from, pos_to, neg_to)


def lorentz_to_ball(W):
    """Lorentz rows (spatial parts x) -> Poincare-ball points x / (1 + sqrt(1 + |x|^2)); the distance is kept
    (d_L(x, y) = d_P of the images).  fp64 inside, fp32 out, on W's device."""
    x = W.detach().to(torch.float64)
    x0 = torch.sqrt(1.0 + (x * x).sum(-1, keepdim=True))
    return (x / (1.0 + x0)).to(torch.float32)


def ball_to_lorentz(P):
    """Poincare-ball points p (|p| < 1) -> Lorentz rows 2p / (1 - |p|^2), the inverse of lorentz_to_ball.  fp64 inside,
    fp32 out, on P's device."""
    p = P.detach().to(torch.float64)
    return (2.0 * p / (1.0 - (p * p).sum(-1, keepdim=True))).to(torch.float32)


def pairs_flat_raw(geom, rows, aux, D, from_idx, to_idx, K, alpha, w=None, is_pos=None, grad_rows=None, loss_out=None,
                   precision=PREC_F64CORE, E_out=None):
    dev = rows.device
    P = int(from_idx.numel())
    if E_out is None:
        E_out = torch.empty(P, device=dev, dtype=torch.float32)
    if loss_out is None:
        loss_out = torch.zeros(1, device=dev, dtype=torch.float64)
    R = 1 if grad_rows is None or grad_rows.dim() == 2 else grad_rows.shape[0]
    N.check(N.lib().lec_pairs_flat(
        GEOM[geom], int(precision), N._p(rows), _aux_ptr(geom, aux), rows.shape[0], int(D), rows.shape[1],
        N._p(from_idx), N._p(to_idx),
        from_idx.element_size(), N._p(w), N._p(is_pos), P, float(K or 0.0), float(alpha), N._p(E_out),
        N._p(loss_out), N._p(grad_rows), R, N.stream_ptr(dev)), "lec_pairs_flat")
    return loss_out, E_out


class FlatPairLoss(torch.autograd.Function):
    """loss, E[P] for an arbitrary list of (from, to) pairs with positive/negative flags."""

    @staticmethod
    def forward(ctx, rows, aux, D, from_idx, to_idx, is_pos, w, geom, K, alpha, precision):
        N.require_cuda(rows)
        dev = rows.device
        rows_c = rows.detach().contiguous()
        from_idx, to_idx = _idx(from_idx, dev), _idx(to_idx, dev)
        if from_idx.dtype != to_idx.dtype:
            from_idx, to_idx = from_idx.to(torch.int64), to_idx.to(torch.int64)
        if is_pos is not None:
            is_pos = torch.as_tensor(is_pos).to(device=dev, dtype=torch.uint8).contiguous()
        need_grad = ctx.needs_input_grad[0]
        grad_rows = None
        if need_grad:
            grad_rows = torch.zeros((default_replicas(*rows_c.shape),) + tuple(rows_c.shape), device=dev)
        loss64, E = pairs_flat_raw(geom, rows_c, aux, D, from_idx, to_idx, K, alpha, _f32(w, dev), is_pos, grad_rows, None,
                                   precision)
        if need_grad:
            grad_rows = reduce_replicas(grad_rows)
        ctx.save_for_backward(grad_rows)
        ctx.mark_non_differentiable(E)
        return loss64[0].float(), E

    @staticmethod
    def backward(ctx, g_loss, _ge):
        (grad_rows,) = ctx.saved_tensors
        return (grad_rows * g_loss,) + (None,) * 10


def flat_pair_loss(rows, aux, D, from_idx, to_idx, geom, K, alpha, is_pos=None, w=None, precision=PREC_F64CORE):
    return FlatPairLoss.apply(rows, aux, D, from_idx, to_idx, is_pos, w, geom, K, alpha, precision)


# --------------------------------------------------------------------------------------------------
# Dense E_operator (no gather)
# --------------------------------------------------------------------------------------------------
class DenseEnergy(torch.autograd.Function):
    """E_operator(x, y) on arbitrary [..., D] CUDA tensors, differentiable in x and y."""

    @staticmethod
    def forward(ctx, x, y, geom, K, precision):
        N.require_cuda(x, y)
        shp = x.shape
        D = shp[-1]
        x2 = x.detach().reshape(-1, D).contiguous().float()
        y2 = y.detach().reshape(-1, D).contiguous().float()
        if x2.shape != y2.shape:
            raise N.LecError("E_operator: x and y must have the same shape, got %s vs %s" % (tuple(x.shape), tuple(y.shape)))
        E = torch.empty(x2.shape[0], device=x.device, dtype=torch.float32)
        N.check(N.lib().lec_energy_dense(GEOM[geom], int(precision), N._p(x2), N._p(y2), x2.shape[0], D,
                                         float(K or 0.0), N._p(E), N.stream_ptr(x.device)), "lec_energy_dense")
        ctx.save_for_backward(x2, y2)
        ctx.meta = (geom, float(K or 0.0), int(precision), shp, y.shape)
        return E.view(shp[:-1])

    @staticmethod
    def backward(ctx, gE):
        x2, y2 = ctx.saved_tensors
        geom, K, precision, xs, ys = ctx.meta
        gE = gE.reshape(-1).contiguous().float()
        gx, gy = torch.empty_like(x2), torch.empty_like(y2)
        N.check(N.lib().lec_energy_dense_bwd(GEOM[geom], precision, N._p(x2), N._p(y2), N._p(gE), x2.shape[0],
                                             x2.shape[1], K, N._p(gx), N._p(gy), N.stream_ptr(x2.device)),
                "lec_energy_dense_bwd")
        return gx.view(xs), gy.view(ys), None, None, None


def energy(x, y, geom, K=None, precision=PREC_F64CORE):
    return DenseEnergy.apply(x, y, geom, K, precision)


# --------------------------------------------------------------------------------------------------
# RSGD
# --------------------------------------------------------------------------------------------------
def rsgd_update_(table, grad, lr, r_in, textbook_lambda=False, write_rescaled_grad=True):
    """In-place Riemannian SGD step on the whole table (lec_rsgd_update).

    `grad` is the Euclidean gradient [n, D] (or [n, ld] padded, or [R, n, ld] replicas).  With write_rescaled_grad the gradient
    buffer is left holding the Riemannian-rescaled gradient, as the reference leaves weight.grad."""
    N.require_cuda(table, grad)
    if not table.is_contiguous() or table.dtype != torch.float32:
        raise N.LecError("rsgd_update_: table must be a contiguous float32 tensor (updated in place)")
    n, D = table.shape
    grad = grad.contiguous()
    R = grad.shape[0] if grad.dim() == 3 else 1
    ld_g = grad.shape[-1]
    grad_out = grad if (write_rescaled_grad and ld_g == D and R == 1) else None
    N.check(N.lib().lec_rsgd_update(N._p(table), N._p(grad), R, n, D, ld_g, float(lr), float(r_in),
                                    1 if textbook_lambda else 0, N._p(grad_out), N.stream_ptr(table.device)),
            "lec_rsgd_update")
    return table


def update_rows_(table, grad_rows, rule, row_mode, geom, K, lr, r_in=0.0, state_m=None, state_v=None, opt_step=1,
                 momentum=0.0, betas=(0.9, 0.999), eps=1e-8, hyp_rescale=False, project_shell=False, rows_out=None,
                 aux_out=None, grad_out=None, loss_acc=None, loss_step=None, exchange=None, lambda_mode=0):
    """The fused table update (lec_update_rows) on caller-owned tensors: replica sum of grad_rows [R, n, ld] (cleared),
    optional peer exchange (a sharding.PeerExchange / LocalExchange; the caller advances its .step), VJP of `row_mode`,
    rule in {"none", "rsgd", "sgd", "adam"} in place on table [n, D], and -- when rows_out / aux_out are given -- the
    transformed rows and aperture terms of the updated table."""
    N.require_cuda(table, grad_rows)
    if not table.is_contiguous() or table.dtype != torch.float32:
        raise N.LecError("update_rows_: table must be a contiguous float32 tensor (updated in place)")
    n, D = table.shape
    if grad_rows.dim() == 2:
        grad_rows = grad_rows.unsqueeze(0)
    u = N.LecUpdate()
    u.rule = {"none": N.UPD_NONE, "rsgd": N.UPD_RSGD, "sgd": N.UPD_SGD, "adam": N.UPD_ADAM}[rule]
    u.row_mode, u.geom, u.lambda_mode = int(row_mode), GEOM[geom] if geom is not None else 0, int(lambda_mode)
    u.hyp_rescale, u.project_shell = int(bool(hyp_rescale)), int(bool(project_shell))
    u.K, u.lr, u.r_in = float(K or 0.0), float(lr), float(r_in)
    u.momentum, u.beta1, u.beta2, u.eps, u.opt_step = float(momentum), float(betas[0]), float(betas[1]), float(eps), int(opt_step)
    u.table, u.n, u.D, u.ld = table.data_ptr(), n, D, grad_rows.shape[-1]
    u.grad_rows, u.grad_replicas = grad_rows.data_ptr(), grad_rows.shape[0]
    for name, tns in (("state_m", state_m), ("state_v", state_v), ("rows_out", rows_out), ("aux_out", aux_out),
                      ("grad_out", grad_out), ("loss_acc", loss_acc), ("loss_step", loss_step)):
        setattr(u, name, tns.data_ptr() if tns is not None else None)
    x = None
    if exchange is not None:
        x = N.LecExchange()
        exchange.fill(x)
    N.check(N.lib().lec_update_rows(ctypes.byref(u), ctypes.byref(x) if x is not None else None,
                                    N.stream_ptr(table.device)), "lec_update_rows")
    return table


# --------------------------------------------------------------------------------------------------
# Scoring
# --------------------------------------------------------------------------------------------------
class CaptionRankingHinge(torch.autograd.Function):
    """S_i = sum_j max(0, alpha + E+_i - E-_ij) (lec_caption_hinge): the image-label loss of the reference's caption-style
    variant, OrderEmbeddingWithImagesLossvCaption.get_image_label_loss (order_embeddings_images.py:533-542).  Forward
    and the energy gradients come out of one launch; backward only scales them."""

    @staticmethod
    def forward(ctx, E_pos, E_neg, alpha):
        N.require_cuda(E_pos)
        N.require_cuda(E_neg)
        ep = E_pos.detach().contiguous().float()
        en = E_neg.detach().contiguous().float()
        B = ep.numel()
        M = en.numel() // B if B else 0
        if en.numel() != B * M:
            raise N.LecError("E_neg must hold M negatives for each of the %d positives" % B)
        S = torch.empty(B, device=ep.device, dtype=torch.float32)
        need = E_pos.requires_grad or E_neg.requires_grad
        gp = torch.empty_like(ep) if need else None
        gn = torch.empty_like(en) if need else None
        N.check(N.lib().lec_caption_hinge(N._p(ep), N._p(en), B, M, float(alpha), N._p(None), N._p(S), N._p(gp), N._p(gn),
                                          N.stream_ptr(ep.device)), "lec_caption_hinge")
        ctx.save_for_backward(gp, gn)
        ctx.shape_neg = E_neg.shape
        return S

    @staticmethod
    def backward(ctx, gS):
        gp, gn = ctx.saved_tensors
        gS = gS.contiguous().float()
        return gp * gS, (gn.view(gS.numel(), -1) * gS[:, None]).view(ctx.shape_neg), None


def caption_ranking_hinge(E_pos, E_neg, alpha):
    """[B], [B, M] -> [B]; differentiable drop-in for get_image_label_loss of order_embeddings_images.py:533-542."""
    return CaptionRankingHinge.apply(E_pos, E_neg, alpha)


_score_ws = {}  # device -> workspace tensor of the tensor-core scoring path (grown on demand, reused)


def _score_workspace(dev, nbytes):
    ws = _score_ws.get(dev)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes) + 128, device=dev, dtype=torch.uint8)
        _score_ws[dev] = ws
    off = (-ws.data_ptr()) % 128
    return ws[off:]


def score_topk_into(labels, images, geom, K, level_start, level_stop, k, idx, val=None, scores=None, scores_layout=1,
                    precision=PREC_F32, engine="auto"):
    """lec_score_topk_tc / lec_score_topk_ex on caller-owned outputs (any of idx / val / scores may be None)."""
    L, D = labels.shape
    n_img = images.shape[0]
    nl = len(level_start)
    ls = (ctypes.c_int32 * max(nl, 1))(*[int(v) for v in level_start])
    le = (ctypes.c_int32 * max(nl, 1))(*[int(v) for v in level_stop])
    dev = labels.device
    # engine: "tc" = tcgen05 tensor-core contraction + fused epilogue (lec_score_topk_tc), "simt" = the packed-FMA
    # tile kernel (lec_score_topk_ex).  "auto" follows the measurements (profiles/r1f_score_bench.log, 1 M x 723):
    # the tensor-core kernel wins every mode it supports since its top-k lists live in registers (top-k 1.40 vs
    # 1.66 ms at D=10, 2.53 vs 4.19 ms at D=50; matrix 0.86 vs 1.04 ms and 1.14 vs 2.68 ms); the SIMT kernel serves the
    # other geometries, the fp64 core and image-major score matrices.
    lib = N.lib()
    tc_ok = scores_layout == 1 and bool(lib.lec_score_tc_supported(GEOM[geom], int(precision), D, L, nl))
    if engine == "tc" and not tc_ok:
        raise N.LecError("tensor-core scoring supports hyperbolic cones, fp32 core, label-major scores, D <= 128")
    if engine == "auto":
        engine = "tc" if tc_ok else "simt"
    if engine == "tc":
        nbytes = int(lib.lec_score_workspace_bytes(L, D, nl))
        ws = _score_workspace(dev, nbytes)
        N.check(lib.lec_score_topk_tc(GEOM[geom], int(precision), N._p(labels), L, N._p(images), n_img, D,
                                      float(K or 0.0), ctypes.cast(ls, ctypes.c_void_p), ctypes.cast(le, ctypes.c_void_p),
                                      nl, int(k), N._p(scores), N._p(idx), N._p(val), N._p(ws), nbytes, N.stream_ptr(dev)),
                "lec_score_topk_tc")
        return
    N.check(lib.lec_score_topk_ex(GEOM[geom], int(precision), N._p(labels), L, N._p(images), n_img, D,
                                  float(K or 0.0), ctypes.cast(ls, ctypes.c_void_p), ctypes.cast(le, ctypes.c_void_p),
                                  nl, int(k), N._p(scores), int(scores_layout), N._p(idx), N._p(val), N.stream_ptr(dev)),
            "lec_score_topk_ex")


def score_topk(labels, images, geom, K, level_start, level_stop, k=5, want_scores=False, want_values=True,
               precision=PREC_F32, scores_layout="label_major", engine="auto"):  # scoring only ranks: fp32 core by default
    """Per image, per level: the k labels of lowest energy E(x=label, y=image) (lec_score_topk_ex).

    Returns (topk_idx int32 [N, n_levels, k], topk_val float32 or None, scores [N, L] or None).  With the
    default scores_layout="label_major" the matrix is stored [L, N] (the layout whose stores coalesce) and
    returned as its transposed view, so it is still indexed scores[i, l]; "image_major" stores [N, L]."""
    N.require_cuda(labels, images)
    labels = labels.detach().contiguous().float()
    images = images.detach().contiguous().float()
    L, D = labels.shape
    n_img = images.shape[0]
    nl = len(level_start)
    dev = labels.device
    idx = torch.empty((n_img, nl, k), device=dev, dtype=torch.int32)
    val = torch.empty((n_img, nl, k), device=dev, dtype=torch.float32) if want_values else None
    layout = {"image_major": 0, "label_major": 1}[scores_layout]
    scores = None
    if want_scores:
        scores = torch.empty((L, n_img) if layout == 1 else (n_img, L), device=dev, dtype=torch.float32)
    score_topk_into(labels, images, geom, K, level_start, level_stop, k, idx, val, scores, layout, precision, engine)
    if scores is not None and layout == 1:
        scores = scores.t()
    return idx, val, scores


class ScorePipeline:
    """Host-to-host scoring of a large image set (the call the reference's calculate_classification_metrics would
    make, oe_h.py:1971-2036): pinned host image embeddings in, per-level top-k label ids (and energies) out in pinned
    host memory.  The set is cut into slices; the upload of slice j+1 and the download of slice j-1 run on their
    own streams while slice j is scored, so the PCIe copies overlap the kernel.  `out_idx_host` may be int32 or int16
    (label ids of any hierarchy below 32 768 labels fit; the narrowing runs on the download stream and halves the
    device->host bytes, which is what bounds this call once the kernel is faster than the PCIe copies)."""

    def __init__(self, labels, geom, K, level_start, level_stop, k=5, slice_images=131072, engine="auto",
                 precision=PREC_F32):
        N.require_cuda(labels)
        self.labels = labels.detach().contiguous().float()
        self.geom, self.K, self.k, self.engine, self.precision = geom, K, int(k), engine, precision
        self.level_start, self.level_stop = list(level_start), list(level_stop)
        dev = self.labels.device
        self.dev, self.slice = dev, int(slice_images)
        D, nl = self.labels.shape[1], len(self.level_start)
        self.s_in, self.s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.img = [torch.empty((self.slice, D), device=dev) for _ in range(2)]
        self.idx = [torch.empty((self.slice, nl, self.k), device=dev, dtype=torch.int32) for _ in range(2)]
        self.val = [torch.empty((self.slice, nl, self.k), device=dev) for _ in range(2)]
        self.ev_in = [torch.cuda.Event() for _ in range(2)]
        self.ev_scored = [torch.cuda.Event() for _ in range(2)]
        self.ev_out = [torch.cuda.Event() for _ in range(2)]
        self.idx16 = None

    def run(self, images_host, out_idx_host, out_val_host=None):
        if images_host.is_cuda or out_idx_host.is_cuda:
            raise N.LecError("ScorePipeline.run takes host tensors (use ops.score_topk for device tensors)")
        main = torch.cuda.current_stream(self.dev)
        n_img = images_host.shape[0]
        narrow = out_idx_host.dtype == torch.int16
        if narrow:
            if self.labels.shape[0] > 32767:
                raise N.LecError("int16 label ids need fewer than 32 768 labels")
            if self.idx16 is None:
                self.idx16 = [torch.empty_like(t, dtype=torch.int16) for t in self.idx]
        elif out_idx_host.dtype != torch.int32:
            raise N.LecError("out_idx_host must be int32 or int16")
        for j, s0 in enumerate(range(0, n_img, self.slice)):
            b, n = j & 1, min(self.slice, n_img - s0)
            with torch.cuda.stream(self.s_in):
                self.s_in.wait_event(self.ev_scored[b])      # the kernel that last read this slot has finished
                self.img[b][:n].copy_(images_host[s0:s0 + n], non_blocking=True)
                self.ev_in[b].record(self.s_in)
            main.wait_event(self.ev_in[b])
            main.wait_event(self.ev_out[b])                  # the download that last read this slot's outputs has finished
            score_topk_into(self.labels, self.img[b][:n], self.geom, self.K, self.level_start, self.level_stop, self.k,
                            self.idx[b][:n], self.val[b][:n] if out_val_host is not None else None, None, 1,
                            self.precision, self.engine)
            self.ev_scored[b].record(main)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_scored[b])
                if narrow:
                    self.idx16[b][:n].copy_(self.idx[b][:n])
                    out_idx_host[s0:s0 + n].copy_(self.idx16[b][:n], non_blocking=True)
                else:
                    out_idx_host[s0:s0 + n].copy_(self.idx[b][:n], non_blocking=True)
                if out_val_host is not None:
                    out_val_host[s0:s0 + n].copy_(self.val[b][:n], non_blocking=True)
                self.ev_out[b].record(self.s_out)
        self.s_out.synchronize()
        return out_idx_host
