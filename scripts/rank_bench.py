"""Reconstruction mean rank and MAP over all node pairs (metrics.reconstruction_ranks / lec_rank_run): time per call,
the time of each stage (positive keys, sort, count, finish; events around them in separate calls), the negatives that
reached the count, and, on the same rows in the same run, reconstruction_f1's time per call.  At n = 20 000 also the
materialised path (SIMT score matrix + a per-row torch.sort), with equal results asserted.

    python scripts/rank_bench.py [--reps 5] [--warmup 2] [--cfg4-steps 2000] [--out FILE]

Workloads: ETHEC hyp D = 10 after 1 000 steps, random tree n = 20 000 D = 50 (A/B), and the cfg4 tree and cfg4-sized
DAG random_dag(82 115, 1.0831, 0.02), D = 50 after 2 000 ConeStep steps (the size at which no matrix fits).  One JSON
line per workload, with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from learning_embeddings_b200 import hierarchy as H, metrics, ops  # noqa: E402
from recon_bench import DEV, K, gpu_info, hyp_rows, timed, trained  # noqa: E402


def materialised(rows, h, D):
    """score matrix, the rank keys, a per-row torch.sort with the positives and the diagonal moved last, then every
    positive's lower and upper bound among its row's negatives (one flat search over rows offset by 2^32)"""
    n = h.n
    x = rows[:, :D].contiguous()
    S = torch.empty((n, n), device=DEV, dtype=torch.float32)
    ops.score_topk_into(x, x, "hyp", K, [], [], 1, None, None, S, 1, engine="simt")
    bits = S.view(torch.int32)
    key = torch.where(torch.isnan(S), 0x7FC00000, torch.where(bits == -0x80000000, 0, bits))
    del S, bits
    e = torch.as_tensor(h.closure_edges(), device=DEV)
    pk = key[e[:, 0], e[:, 1]].to(torch.int64) + (e[:, 0] << 32)
    key[e[:, 0], e[:, 1]] = 0x7FFFFFFF
    key.fill_diagonal_(0x7FFFFFFF)
    key, _ = torch.sort(key, dim=1)
    flat = (key.to(torch.int64) + (torch.arange(n, device=DEV, dtype=torch.int64)[:, None] << 32)).reshape(-1)
    del key
    start = e[:, 0] * n
    r_opt = 1 + torch.searchsorted(flat, pk) - start
    r_pess = 1 + torch.searchsorted(flat, pk, right=True) - start
    return torch.stack([r_opt, r_pess], 1).to(torch.int32)


def workload(name, h, rows, D, args, info, ab=False):
    n = h.n
    stats = {}
    out, t = timed(lambda: metrics.reconstruction_ranks(rows, h, "hyp", K, D=D, stats=stats), args.reps, args.warmup)
    _, tf = timed(lambda: metrics.reconstruction_f1(rows, h, "hyp", K, D=D), args.reps, args.warmup)
    stage = []
    for _ in range(args.reps):
        st = {}
        metrics.reconstruction_ranks(rows, h, "hyp", K, D=D, stats=st, time_stages=True)
        stage.append(st["stage_ms"])
    rec = {"workload": name, "n": n, "D": D, "pairs": n * (n - 1), **info, **t,
           "f1_median_ms": tf["median_ms"], "ranks_over_f1": t["median_ms"] / tf["median_ms"],
           "stage_median_ms": {k: float(np.median([s[k] for s in stage])) for k in stage[0]},
           "n_edges": out["n_edges"], "n_apexes": out["n_apexes"], "counted_negatives": stats["counted_negatives"],
           "negatives": n * (n - 1) - out["n_edges"], "workspace_mb": stats["workspace_bytes"] / 2**20,
           "mean_rank": out["mean_rank"], "mean_rank_optimistic": out["mean_rank_optimistic"], "map": out["map"]}
    if ab:
        got = metrics.reconstruction_ranks(rows, h, "hyp", K, D=D, return_ranks=True)["ranks"]
        torch.cuda.empty_cache()
        ref, tm = timed(lambda: materialised(rows, h, D), args.reps, args.warmup)
        rec["materialised"] = tm
        rec["ranks_equal"] = bool(torch.equal(got, ref))
        assert rec["ranks_equal"], "materialised ranks differ"
        rec["speedup"] = tm["median_ms"] / t["median_ms"]
    assert not math.isnan(rec["mean_rank"])
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cfg4-steps", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_bench needs a CUDA device")
    info = gpu_info()
    out = open(args.out, "w") if args.out else None

    def emit(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    h = H.ethec()
    rows, D = trained(h, 10, 1000)
    emit(workload("ethec_hyp_D10_trained1000", h, rows, D, args, info))
    h = H.random_tree(20000, 1.0831)
    emit(workload("tree20000_hyp_D50_ab", h, hyp_rows(h, 50), 50, args, info, ab=True))
    h = H.random_tree(82115, 1.0831)
    rows, D = trained(h, 50, args.cfg4_steps)
    emit(workload("cfg4_hyp_D50_trained%d" % args.cfg4_steps, h, rows, D, args, info))
    h = H.random_dag(82115, 1.0831, 0.02)
    rows, D = trained(h, 50, args.cfg4_steps)
    emit(workload("cfg4dag002_hyp_D50_trained%d" % args.cfg4_steps, h, rows, D, args, info))


if __name__ == "__main__":
    main()
