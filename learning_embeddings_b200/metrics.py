"""Evaluation of the cone path on the device: reconstruction F1 sweep and image-classification metrics.

Drop-ins for `EmbeddingMetrics` (order_embeddings.py:250-306 = oe.py:358-414) and for the scoring + bookkeeping
body of `JointEmbeddings.calculate_classification_metrics` (oe.py:1721-1921, oe_h.py:1971-2178).  The arithmetic
that decides results (energies, top-k, counts, the F1 arg-max) runs in the CUDA library; only the final scalar
formulas, which the reference evaluates on Python ints, are evaluated here on Python ints as well, in the
reference's order, so every reported number is the same float.
"""
import ctypes
import math

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


def _eval_rows(rows, hierarchy, D, what, need_pairs=False):
    """(rows, D) of an all-pairs evaluation of `hierarchy`: checked, and copied to a plain [n, D] table unless the
    kernels can read them as they are (16-byte aligned, unit column stride, row stride D or a multiple of 4)"""
    N.require_cuda(rows)
    if rows.dim() != 2 or rows.dtype != torch.float32:
        raise N.LecError("%s: rows must be a float32 [n, ld] tensor" % what)
    n = rows.shape[0]
    D = rows.shape[1] if D is None else int(D)
    if n != hierarchy.n:
        raise ValueError("%s: %d rows for a hierarchy of %d nodes" % (what, n, hierarchy.n))
    if need_pairs and n < 2:
        raise ValueError("%s: no pairs" % what)
    if D > rows.shape[1]:
        raise ValueError("%s: D = %d exceeds the row width %d" % (what, D, rows.shape[1]))
    rows = rows.detach()
    if rows.stride(1) != 1 or (rows.stride(0) != D and rows.stride(0) % 4 != 0) or rows.data_ptr() % 16 != 0:
        rows = rows[:, :D].contiguous()
    return rows, D


class _Cover:
    """The interval cover of a hierarchy on the device: tin, tout and, for a DagHierarchy with extra intervals, the
    LecReconExtra `x` (None otherwise) with the tensors it points into."""

    def __init__(self, hierarchy, dev):
        self.tin = torch.as_tensor(np.asarray(hierarchy.tin), dtype=torch.int32).to(dev)
        self.tout = torch.as_tensor(np.asarray(hierarchy.tout), dtype=torch.int32).to(dev)
        self.n_extra = int(hierarchy.extra_ptr[-1]) if hasattr(hierarchy, "extra_ptr") else 0
        self.x = None
        if self.n_extra:
            self.xs = [torch.as_tensor(np.asarray(a), dtype=torch.int32).to(dev)
                       for a in (hierarchy.extra_ptr, hierarchy.extra_lo, hierarchy.extra_hi)]
            self.x = N.LecReconExtra(self.xs[0].data_ptr(), self.xs[1].data_ptr(), self.xs[2].data_ptr(), self.n_extra)


class _Heldout:
    """hierarchy.heldout_slots(edges) on the device: the LecHeldout `h`, the held-out layout eval_ptr (host and
    device), the held-out slot of each edge (`order`) and the closure layout's size."""

    def __init__(self, hierarchy, edges, dev):
        closure_ptr, _ = hierarchy.rank_slots()
        eval_ptr, slot_map, self.order, xcum = hierarchy.heldout_slots(edges)
        self.eval_ptr_h = eval_ptr
        self.n_closure = int(closure_ptr[-1])
        # one spare entry: a closure without edges still passes a non-NULL slot map
        self.keep = [torch.as_tensor(a).to(dev) for a in (closure_ptr, np.r_[slot_map, np.int32(-1)])]
        self.eval_ptr = torch.as_tensor(eval_ptr).to(dev)
        xc = None
        if xcum is not None and len(xcum):
            xc = torch.as_tensor(xcum).to(dev)
            self.keep.append(xc)
        self.h = N.LecHeldout(self.keep[0].data_ptr(), self.keep[1].data_ptr(), 0 if xc is None else xc.data_ptr(),
                              self.n_closure)


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
    energies: positives are E(x = rows[u], y = rows[v]) for every v below u in `hierarchy` (a hierarchy.Hierarchy or
    DagHierarchy), negatives every other ordered pair u != v, and the result is best_f1_sweep's numpy row (f1,
    threshold, accuracy, precision, recall, correct_positives, correct_negatives) over those energies, bit for bit, with
    the energies of the fp32 SIMT scoring kernel (lec_recon_pass / lec_recon_finish; lec_recon_pass_dag when a
    DagHierarchy has extra intervals).

    rows: device fp32 [n, ld] -- a plain [n, D] table or an engine's padded rows (ConeStep.rows with D = ConeStep.D).
    group: a torch.distributed group whose ranks each evaluate a contiguous share of the apex rows on their own GPU
    (every rank passes the same rows); the counters are summed after every round, so every rank returns the row.
    workspace_bytes: device workspace, lec_recon_workspace_bytes(RECON_OPEN_BINS) by default; a smaller one costs
    rounds, not exactness.  stats: a dict that receives the rounds run, the open coarse bins, the numbers of positive
    and negative pairs, the workspace size and the number of extra intervals (0 for a forest)."""
    rows, D = _eval_rows(rows, hierarchy, D, "reconstruction_f1", need_pairs=True)
    return _recon_rounds(rows, hierarchy, geom, K, D, group, workspace_bytes, stats)


def _recon_rounds(rows, hierarchy, geom, K, D, group, workspace_bytes, stats, held=None, threshold=None):
    """the rounds of reconstruction_f1 (held: a _Heldout, threshold: lec_recon_finish_at's t)"""
    n = rows.shape[0]
    dev = rows.device
    lib = N.lib()
    cov = _Cover(hierarchy, dev)
    n_extra = cov.n_extra
    nb = int(lib.lec_recon_workspace_bytes(RECON_OPEN_BINS)) if workspace_bytes is None else int(workspace_bytes)
    cb = int(lib.lec_recon_counter_bytes(nb))
    if cb < 0:
        N.check(cb, "lec_recon_counter_bytes")
    ws = torch.zeros(nb, device=dev, dtype=torch.uint8)
    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    r = recon_args(rows, cov.tin, cov.tout, geom, K, D, n * rank // world, n * (rank + 1) // world, ws)
    out = torch.empty(7, device=dev, dtype=torch.float64)
    status = torch.zeros(4, device=dev, dtype=torch.int64)
    stream = N.stream_ptr(dev)
    x = None if cov.x is None else ctypes.byref(cov.x)
    h = None if held is None else ctypes.byref(held.h)
    rounds = 0
    while True:
        N.check(lib.lec_recon_pass_heldout(ctypes.byref(r), x, h, stream), "lec_recon_pass_heldout")
        rounds += 1
        if group is not None:
            dist.all_reduce(ws[:cb].view(torch.int64), group=group)
        if threshold is None:
            N.check(lib.lec_recon_finish(ctypes.byref(r), N._p(out), N._p(status), stream), "lec_recon_finish")
        else:
            N.check(lib.lec_recon_finish_at(ctypes.byref(r), float(threshold), N._p(out), N._p(status), stream),
                    "lec_recon_finish_at")
        more, open_bins, n_pos, n_neg = (int(v) for v in status.cpu())
        if not more:
            break
        if rounds > open_bins + 1:   # each fine round retires at least one open bin
            raise N.LecError("lec_recon_finish asks for round %d with %d open bins" % (rounds + 1, open_bins))
    if stats is not None:
        stats.update(rounds=rounds, open_bins=open_bins, n_pos=n_pos, n_neg=n_neg, workspace_bytes=nb,
                     extra_intervals=n_extra)
    return out.cpu().numpy()


RANK_SHARED_BUCKETS = 16384   # kRankShared of csrc/lec_score_fast_impl.cuh: a larger apex counts in global memory


def rank_args(rows, tin, tout, extra, pos_ptr, n_pos, geom, K, D, u_begin, u_end, workspace, stage_ms=None):
    """lec_rank_t for device rows [n, >= D] (fp32, unit column stride), device int32 tin / tout [n], an optional
    LecReconExtra (None: a forest), device int64 pos_ptr [n+1] and a device workspace tensor; apexes [u_begin, u_end)."""
    r = N.LecRank()
    r.geom, r.K = N.GEOM[geom], float(K or 0.0)
    r.rows, r.n, r.D, r.ld = rows.data_ptr(), rows.shape[0], int(D), rows.stride(0)
    r.tin, r.tout = tin.data_ptr(), tout.data_ptr()
    if extra is not None:
        r.extra = ctypes.pointer(extra)
    r.pos_ptr, r.n_pos = pos_ptr.data_ptr(), int(n_pos)
    r.u_begin, r.u_end = int(u_begin), int(u_end)
    r.workspace, r.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    if stage_ms is not None:
        r.stage_ms = stage_ms
    return r


def reconstruction_ranks(rows, hierarchy, geom, K, D=None, group=None, return_ranks=False, stats=None,
                         time_stages=False):
    """Mean rank and mean average precision of the reconstruction check (Nickel & Kiela, Poincaré embeddings; the
    numbers the hyperbolic-embedding literature reports for WordNet nouns) over the pairs of reconstruction_f1, without
    materialising the n (n-1) energies (lec_rank_run).  For each closure edge (u, v) the rank of v among the negatives
    of apex u (every w != u that is not below u) by the fp32 energy of the SIMT scoring kernel; other positives of u
    are not counted ("filtered" ranks).  Ties: rank_opt counts the negatives with a smaller key, rank_pess those with a
    smaller or equal one (key = the energy's fp32 bits, -0 as 0, NaN after +inf); the reference's unstable argsort
    lands in between.  AP_u groups tied keys like sklearn's average_precision_score(labels, -E).

    rows: device fp32 [n, ld] -- a plain [n, D] table or an engine's padded rows (ConeStep.rows with D = ConeStep.D).
    hierarchy: a hierarchy.Hierarchy or DagHierarchy.
    group: a torch.distributed group whose ranks each evaluate a contiguous share of the apexes on their own GPU (every
    rank passes the same rows); the per-apex results are disjoint, so summing them is exact, and every rank returns
    the result.
    Returns a dict: mean_rank (pessimistic ties, the headline: trained cones put many pairs at exactly E = 0),
    mean_rank_optimistic, map (math.fsum of AP_u over the n_apexes apexes with a descendant), n_edges, n_apexes and
    ap (numpy fp64 [n], NaN where u has no descendant); with return_ranks also ranks, device int32 [n_edges, 2]
    (optimistic, pessimistic) in hierarchy.closure_edges() order.  Without edges the three means are NaN.
    stats: a dict that receives the workspace size, the negatives at or below their apex's largest positive key (the
    ones that reach the count) and, with time_stages (which synchronises after each call), the four stage times in ms."""
    rows, D = _eval_rows(rows, hierarchy, D, "reconstruction_ranks")
    pos_ptr_h, slot_of_edge = hierarchy.rank_slots()
    return _rank_run(rows, hierarchy, geom, K, D, group, return_ranks, stats, time_stages, pos_ptr_h, slot_of_edge)


def _rank_run(rows, hierarchy, geom, K, D, group, return_ranks, stats, time_stages, pos_ptr_h, slot_of, held=None):
    """lec_rank_run(_heldout) of reconstruction_ranks over the layout pos_ptr_h; slot_of: the slot of each returned
    rank's edge"""
    n = rows.shape[0]
    dev = rows.device
    lib = N.lib()
    n_edges = int(pos_ptr_h[-1])
    has = np.diff(pos_ptr_h) > 0
    n_apexes = int(has.sum())
    cov = _Cover(hierarchy, dev)
    pos_ptr = torch.as_tensor(pos_ptr_h, dtype=torch.int64).to(dev)
    nb = int(lib.lec_rank_workspace_bytes(n, n_edges))
    if nb < 0:
        N.check(int(nb), "lec_rank_workspace_bytes")
    ws = torch.empty(nb, device=dev, dtype=torch.uint8)
    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    stage_ms = (ctypes.c_float * 4)() if time_stages else None
    r = rank_args(rows, cov.tin, cov.tout, cov.x, pos_ptr, n_edges, geom, K, D, n * rank // world,
                  n * (rank + 1) // world, ws, stage_ms)
    sums = torch.zeros(3, device=dev, dtype=torch.int64)
    ap = torch.zeros(n, device=dev, dtype=torch.float64)
    ranks = torch.zeros((n_edges, 2), device=dev, dtype=torch.int32) if return_ranks else None
    N.check(lib.lec_rank_run_heldout(ctypes.byref(r), None if held is None else ctypes.byref(held.h), N._p(sums),
                                     N._p(ap), N._p(ranks), N.stream_ptr(dev)), "lec_rank_run_heldout")
    if group is not None:
        for t in (sums, ap) if ranks is None else (sums, ap, ranks):
            dist.all_reduce(t, group=group)
    s_opt, s_pess, counted = (int(v) for v in sums.cpu())
    ap = ap.cpu().numpy()
    ap[~has] = np.nan
    if n_edges:
        out = {"mean_rank": s_pess / n_edges, "mean_rank_optimistic": s_opt / n_edges,
               "map": math.fsum(ap[has].tolist()) / n_apexes}
    else:
        out = {"mean_rank": math.nan, "mean_rank_optimistic": math.nan, "map": math.nan}
    out.update(n_edges=n_edges, n_apexes=n_apexes, ap=ap)
    if ranks is not None:
        out["ranks"] = ranks[torch.as_tensor(slot_of, device=dev)]
    if stats is not None:
        stats.update(workspace_bytes=nb, counted_negatives=counted)
        if time_stages:
            stats["stage_ms"] = dict(zip(("keys", "sort", "count", "finish"), (float(v) for v in stage_ms)))
    return out


def link_prediction_ranks(rows, hierarchy, edges, geom, K, D=None, group=None, return_ranks=False, stats=None,
                          time_stages=False):
    """Mean rank and MAP of link prediction on the held-out closure edges `edges` [m, 2] (Nickel & Kiela's "link
    prediction" column; hierarchy.split_edges makes a split): reconstruction_ranks with the held-out pairs as the
    positives, every ordered pair u != w with w not below u in the full closure as the negatives, and the other closure
    pairs (the training pairs) skipped; same keys, ties and energies, without materialising them (lec_rank_run_heldout).
    With edges = hierarchy.closure_edges() the result is reconstruction_ranks', bit for bit.
    Returns reconstruction_ranks' dict: n_edges = m, n_apexes = the apexes with a held-out edge, ap NaN at every other
    node, and with return_ranks the ranks in `edges` order."""
    rows, D = _eval_rows(rows, hierarchy, D, "link_prediction_ranks")
    held = _Heldout(hierarchy, edges, rows.device)
    return _rank_run(rows, hierarchy, geom, K, D, group, return_ranks, stats, time_stages, held.eval_ptr_h, held.order,
                     held)


def link_prediction_f1(rows, hierarchy, edges, geom, K, D=None, threshold=None, group=None, workspace_bytes=None,
                       stats=None):
    """F1 of link prediction on the held-out closure edges `edges` [m, 2] (Ganea et al.'s transitive closure
    completion) over the pairs of link_prediction_ranks: positives the held-out pairs, negatives every ordered pair
    u != w with w not below u in the full closure, training pairs skipped (lec_recon_pass_heldout).
    Without threshold: reconstruction_f1's best-F1 row over those pairs ('val' phase).  With threshold=t: the row of
    EmbeddingMetrics(..., t, 'test').calculate_metrics() over them (lec_recon_finish_at: E <= t is a predicted
    positive, a NaN energy never is; t is compared in fp32 like the reference's float32 energies), with t itself in
    slot 1 -- pick t on a "val" split, report it on "test".  stats as reconstruction_f1's, plus skipped_pairs."""
    rows, D = _eval_rows(rows, hierarchy, D, "link_prediction_f1", need_pairs=True)
    held = _Heldout(hierarchy, edges, rows.device)
    out = _recon_rounds(rows, hierarchy, geom, K, D, group, workspace_bytes, stats, held, threshold)
    if threshold is not None:
        out[1] = threshold
    if stats is not None:
        stats["skipped_pairs"] = held.n_closure - int(held.eval_ptr_h[-1])
    return out


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
