"""Evaluation of the cone path on the device: reconstruction F1 sweep and image-classification metrics.

Drop-ins for `EmbeddingMetrics` (order_embeddings.py:250-306 = oe.py:358-414) and for the scoring + bookkeeping
body of `JointEmbeddings.calculate_classification_metrics` (oe.py:1721-1921, oe_h.py:1971-2178).  The arithmetic
that decides results (energies, top-k, counts, the F1 arg-max) runs in the CUDA library; only the final scalar
formulas, which the reference evaluates on Python ints, are evaluated here on Python ints as well, in the
reference's order, so every reported number is the same float.
"""
import ctypes

import numpy as np
import torch

from . import _native as N
from . import ops


def best_f1_sweep(e_pos, e_neg):
    """Row (f1, threshold, accuracy, precision, recall, correct_positives, correct_negatives) of the first threshold
    with maximal F1 over all unique energies (EmbeddingMetrics.calculate_metrics, 'val').  CPU tensors are moved to
    the GPU (the reference's check_graph_embedding builds them on the CPU, order_embeddings.py:540-553)."""
    if not torch.cuda.is_available():
        raise N.LecError("no CUDA device: the F1 sweep has no CPU path")
    dev = e_pos.device if e_pos.is_cuda else torch.device("cuda")
    ep = e_pos.detach().reshape(-1).to(dev, torch.float32)
    en = e_neg.detach().reshape(-1).to(dev, torch.float32)
    n_pos, n_neg = ep.numel(), en.numel()
    if n_pos + n_neg == 0:
        raise ValueError("best_f1_sweep: no energies")
    vals, order = torch.sort(torch.cat([ep, en]))          # ascending, NaN last
    pos_prefix = torch.cumsum((order < n_pos).to(torch.int64), dim=0)
    out = torch.empty(7, device=dev, dtype=torch.float64)
    nb = int(N.lib().lec_f1_workspace_bytes())
    ws = torch.empty(nb, device=dev, dtype=torch.uint8)
    N.check(N.lib().lec_f1_sweep(N._p(vals), N._p(pos_prefix), n_pos + n_neg, n_pos, n_neg, N._p(out), N._p(ws), nb,
                                 N.stream_ptr(dev)), "lec_f1_sweep")
    return out.cpu().numpy()


RECON_OPEN_BINS = 128   # default coarse bins recounted per round of reconstruction_f1 (about 1 MB of workspace each)


def recon_args(rows, tin, tout, geom, K, D, u_begin, u_end, workspace):
    """lec_recon_t for device rows [n, >= D] (fp32, unit column stride), device int32 Euler intervals tin / tout [n]
    and a device workspace tensor; apex rows [u_begin, u_end)."""
    r = N.LecRecon()
    r.geom, r.K = N.GEOM[geom], float(K or 0.0)
    r.rows, r.n, r.D, r.ld = rows.data_ptr(), rows.shape[0], int(D), rows.stride(0)
    r.tin, r.tout = tin.data_ptr(), tout.data_ptr()
    r.u_begin, r.u_end = int(u_begin), int(u_end)
    r.workspace, r.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    return r


def reconstruction_f1(rows, hierarchy, geom, K, D=None, group=None, workspace_bytes=None, stats=None):
    """check_graph_embedding (order_embeddings.py:512-559 = oe.py:1923-1990) without materialising the n (n-1)
    energies: positives are E(x = rows[u], y = rows[v]) for every v below u in `hierarchy` (a hierarchy.Hierarchy),
    negatives every other ordered pair u != v, and the result is best_f1_sweep's numpy row (f1, threshold, accuracy,
    precision, recall, correct_positives, correct_negatives) over those energies, bit for bit, with the energies of
    the fp32 SIMT scoring kernel (lec_recon_pass / lec_recon_finish).

    rows: device fp32 [n, ld] -- a plain [n, D] table or an engine's padded rows (ConeStep.rows with D = ConeStep.D).
    group: a torch.distributed group whose ranks each evaluate a contiguous share of the apex rows on their own GPU
    (every rank passes the same rows); the counters are summed after every round, so every rank returns the row.
    workspace_bytes: device workspace, lec_recon_workspace_bytes(RECON_OPEN_BINS) by default; a smaller one costs
    rounds, not exactness.  stats: a dict that receives the rounds run, the open coarse bins, the numbers of positive
    and negative pairs and the workspace size."""
    N.require_cuda(rows)
    if rows.dim() != 2 or rows.dtype != torch.float32:
        raise N.LecError("reconstruction_f1: rows must be a float32 [n, ld] tensor")
    n = rows.shape[0]
    D = rows.shape[1] if D is None else int(D)
    if n != hierarchy.n:
        raise ValueError("reconstruction_f1: %d rows for a hierarchy of %d nodes" % (n, hierarchy.n))
    if n < 2:
        raise ValueError("reconstruction_f1: no pairs")
    if D > rows.shape[1]:
        raise ValueError("reconstruction_f1: D = %d exceeds the row width %d" % (D, rows.shape[1]))
    rows = rows.detach()
    if rows.stride(1) != 1 or (rows.stride(0) != D and rows.stride(0) % 4 != 0) or rows.data_ptr() % 16 != 0:
        rows = rows[:, :D].contiguous()
    dev = rows.device
    lib = N.lib()
    tin = torch.as_tensor(np.asarray(hierarchy.tin), dtype=torch.int32).to(dev)
    tout = torch.as_tensor(np.asarray(hierarchy.tout), dtype=torch.int32).to(dev)
    nb = int(lib.lec_recon_workspace_bytes(RECON_OPEN_BINS)) if workspace_bytes is None else int(workspace_bytes)
    cb = int(lib.lec_recon_counter_bytes(nb))
    if cb < 0:
        N.check(cb, "lec_recon_counter_bytes")
    ws = torch.zeros(nb, device=dev, dtype=torch.uint8)
    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    r = recon_args(rows, tin, tout, geom, K, D, n * rank // world, n * (rank + 1) // world, ws)
    out = torch.empty(7, device=dev, dtype=torch.float64)
    status = torch.zeros(4, device=dev, dtype=torch.int64)
    stream = N.stream_ptr(dev)
    rounds = 0
    while True:
        N.check(lib.lec_recon_pass(ctypes.byref(r), stream), "lec_recon_pass")
        rounds += 1
        if group is not None:
            dist.all_reduce(ws[:cb].view(torch.int64), group=group)
        N.check(lib.lec_recon_finish(ctypes.byref(r), N._p(out), N._p(status), stream), "lec_recon_finish")
        more, open_bins, n_pos, n_neg = (int(v) for v in status.cpu())
        if not more:
            break
        if rounds > open_bins + 1:   # each fine round retires at least one open bin
            raise N.LecError("lec_recon_finish asks for round %d with %d open bins" % (rounds + 1, open_bins))
    if stats is not None:
        stats.update(rounds=rounds, open_bins=open_bins, n_pos=n_pos, n_neg=n_neg, workspace_bytes=nb)
    return out.cpu().numpy()


class EmbeddingMetrics:
    """Same constructor and `calculate_metrics` contract as the reference's class."""

    def __init__(self, e_for_u_v_positive, e_for_u_v_negative, threshold, phase, n_proc=4):
        self.e_for_u_v_positive = e_for_u_v_positive.view(-1)
        self.e_for_u_v_negative = e_for_u_v_negative.view(-1)
        self.threshold = threshold
        self.phase = phase
        self.n_proc = n_proc  # kept for signature compatibility; there is no process pool

    def calculate_metrics(self):
        if self.phase == "val":
            return best_f1_sweep(self.e_for_u_v_positive, self.e_for_u_v_negative)
        # fixed threshold (order_embeddings.py:289-306)
        if not torch.cuda.is_available():
            raise N.LecError("no CUDA device: the metrics have no CPU path")
        ep, en = self.e_for_u_v_positive.cuda(), self.e_for_u_v_negative.cuda()
        t = float(self.threshold)
        cp = int((ep <= t).sum().item())
        cn = int((en > t).sum().item())
        n_pos, n_neg = ep.shape[0], en.shape[0]
        accuracy = (cp + cn) / (n_pos + n_neg)
        precision = 0.0 if cp + (n_neg - cn) == 0 else cp / (cp + (n_neg - cn))
        recall = cp / n_pos
        f1 = 0.0 if precision + recall == 0 else (2 * precision * recall) / (precision + recall)
        return f1, self.threshold, accuracy, precision, recall, cp, cn


def classification_counts(topk_idx, truth, n_labels, level_start, level_stop, k_vals=(1, 3, 5)):
    """hit@k per true label and tp / fp / tn / fn per label from per-level top-k predictions (lec_classify_counts).

    topk_idx int32 [n_img, n_levels, k] (CUDA, as ops.score_topk returns it); truth [n_img, n_levels] true label ids.
    Returns numpy int64 arrays: hit [len(k_vals), L], tp, fp, tn, fn [L]."""
    N.require_cuda(topk_idx)
    dev = topk_idx.device
    topk_idx = topk_idx.contiguous()
    n_img, nl, k = topk_idx.shape
    truth_d = torch.as_tensor(np.asarray(truth), dtype=torch.int32).to(dev).contiguous()
    if tuple(truth_d.shape) != (n_img, nl):
        raise N.LecError("truth must be [n_img, n_levels]")
    kv = (ctypes.c_int32 * len(k_vals))(*[int(v) for v in k_vals])
    hit = torch.zeros((len(k_vals), n_labels), device=dev, dtype=torch.int64)
    counts = torch.zeros((3, n_labels), device=dev, dtype=torch.int64)
    level_correct = torch.zeros(nl, device=dev, dtype=torch.int64)
    N.check(N.lib().lec_classify_counts(N._p(topk_idx), N._p(truth_d), n_img, nl, k, ctypes.cast(kv, ctypes.c_void_p),
                                        len(k_vals), n_labels, N._p(hit), N._p(counts), N._p(level_correct),
                                        N.stream_ptr(dev)), "lec_classify_counts")
    hit, counts, level_correct = hit.cpu().numpy(), counts.cpu().numpy(), level_correct.cpu().numpy()
    tp, fp, fn = counts[0], counts[1], counts[2]
    tn = np.zeros(n_labels, dtype=np.int64)
    for lvl, (s, e) in enumerate(zip(level_start, level_stop)):
        tn[int(s):int(e)] = level_correct[lvl] - tp[int(s):int(e)]   # oe.py:1789-1793
    return hit, tp, fp, tn, fn


def classification_metrics(label_rep, img_rep, truth, labelmap, geom, K, k=(1, 3, 5), engine="auto"):
    """The scoring loop and metric assembly of calculate_classification_metrics (oe.py:1755-1921) for label
    embeddings `label_rep` [L, D], image embeddings `img_rep` [n_img, D] (as the caller prepared them -- the
    reference's slicing leaves the last row of each zero, SURVEY F9) and the images' true label per level.
    Returns the reference's `calculated_metrics` dict."""
    if not torch.cuda.is_available():
        raise N.LecError("no CUDA device: scoring has no CPU path")
    dev = label_rep.device if label_rep.is_cuda else torch.device("cuda")
    lab = label_rep.detach().reshape(-1, label_rep.shape[-1]).to(dev, torch.float32)
    img = img_rep.detach().reshape(-1, img_rep.shape[-1]).to(dev, torch.float32)
    L, n_img = lab.shape[0], img.shape[0]
    n_levels = len(labelmap.levels)
    ls, le = list(labelmap.level_start)[:n_levels], list(labelmap.level_stop)[:n_levels]
    k = list(k)
    m = {"median_img_norm": torch.median(torch.norm(img, dim=1)).cpu(),
         "median_label_norm": torch.median(torch.norm(lab, dim=1)).cpu()}
    idx, _, _ = ops.score_topk(lab, img, geom, K, ls, le, k=max(k), want_values=False, engine=engine)
    hit, tp, fp, tn, fn = classification_counts(idx, truth, L, ls, le, k)
    tp, fp, tn, fn = (a.tolist() for a in (tp, fp, tn, fn))   # Python ints: the reference divides ints
    hit = hit.tolist()
    prec_l, rec_l, f1_l = [0.0] * L, [0.0] * L, [0.0] * L
    total = {"tp": 0, "fp": 0, "tn": 0, "fn": 0}
    overall_hit = [0] * len(k)
    for l in range(L):
        for j in range(len(k)):
            overall_hit[j] += hit[j][l]
        total["tp"] += tp[l]; total["fp"] += fp[l]; total["tn"] += tn[l]; total["fn"] += fn[l]
        _ = (tp[l] + tn[l]) / (tp[l] + tn[l] + fp[l] + fn[l])   # per-label accuracy; ZeroDivisionError as in oe.py:1809
        prec_l[l] = 0.0 if tp[l] + fp[l] == 0.0 else tp[l] / (tp[l] + fp[l])
        rec_l[l] = 0.0 if tp[l] + fn[l] == 0.0 else tp[l] / (tp[l] + fn[l])
        f1_l[l] = 0.0 if prec_l[l] + rec_l[l] == 0 else (2 * prec_l[l] * rec_l[l]) / (prec_l[l] + rec_l[l])
    accuracy = (total["tp"] + total["tn"]) / (total["tp"] + total["tn"] + total["fp"] + total["fn"])
    precision = total["tp"] / (total["tp"] + total["fp"])
    recall = total["tp"] / (total["tp"] + total["fn"])
    m["accuracy"], m["m-precision"], m["m-recall"] = accuracy, precision, recall
    m["m-f1"] = 0.0 if precision + recall == 0 else (2 * precision * recall) / (precision + recall)
    for j, kv in enumerate(k):
        m["hit@{}".format(kv)] = overall_hit[j] / (n_levels * n_img)
    mp = mr = mf = 0.0
    for l in range(L):
        mp += prec_l[l]; mr += rec_l[l]; mf += f1_l[l]
    m["M-precision"], m["M-recall"], m["M-f1"] = mp / L, mr / L, mf / L
    m["level_metrics"] = {}
    for lvl in range(n_levels):
        s, e = int(ls[lvl]), int(le[lvl])
        ltp = ltn = lfp = lfn = 0
        lmf = 0.0
        lhit = [0] * len(k)
        for l in range(s, e):
            ltp += tp[l]; ltn += tn[l]; lfp += fp[l]; lfn += fn[l]
            lmf += f1_l[l]
            for j in range(len(k)):
                lhit[j] += hit[j][l]
        d = {}
        for j, kv in enumerate(k):
            d["hit@{}".format(kv)] = lhit[j] / n_img
        lmf /= (e - s + 1)   # sic, oe.py:1879
        lp, lr = ltp / (ltp + lfp), ltp / (ltp + lfn)
        d["m-precision"], d["m-recall"] = lp, lr
        d["m-f1"] = 0.0 if lp + lr == 0 else (2 * lp * lr) / (lp + lr)
        d["M-f1"] = lmf
        d["accuracy"] = (ltp + ltn) / (ltp + ltn + lfp + lfn)
        m["level_metrics"][lvl] = d
    return m
