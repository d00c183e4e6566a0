"""Link prediction on held-out closure edges (metrics.link_prediction_ranks / link_prediction_f1): time per call of the
ranks (with the time of each stage: keys, sort, count, finish; events around them in separate calls), of the best-F1
row and of the row at a fixed threshold, next to reconstruction_ranks and reconstruction_f1 on the same rows in the same
run.  The held-out set is split_edges' "test" at 5 % + 5 %, the threshold the best one on "val".

    python scripts/linkpred_bench.py [--reps 3] [--warmup 1] [--cfg4-steps 2000] [--out FILE]

Workloads: the cfg4 tree random_tree(82 115, 1.0831) and the cfg4-sized DAG random_dag(82 115, 1.0831, 0.02), hyp,
D = 50 after 2 000 ConeStep steps on the full closure, as scripts/rank_bench.py.  One JSON line per workload, with the
GPU's name and power limit read in the same run.
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
from learning_embeddings_b200 import hierarchy as H, metrics  # noqa: E402
from recon_bench import K, gpu_info, timed, trained  # noqa: E402


def workload(name, h, rows, D, args, info):
    split = H.split_edges(h, val=0.05, test=0.05)
    test, val = split["test"], split["val"]
    stats = {}
    out, t_rank = timed(lambda: metrics.link_prediction_ranks(rows, h, test, "hyp", K, D=D, stats=stats),
                        args.reps, args.warmup)
    t_val = float(metrics.link_prediction_f1(rows, h, val, "hyp", K, D=D)[1])
    f1_stats = {}
    best, t_best = timed(lambda: metrics.link_prediction_f1(rows, h, test, "hyp", K, D=D, stats=f1_stats),
                         args.reps, args.warmup)
    at_stats = {}
    at, t_at = timed(lambda: metrics.link_prediction_f1(rows, h, test, "hyp", K, D=D, threshold=t_val, stats=at_stats),
                     args.reps, args.warmup)
    _, t_rr = timed(lambda: metrics.reconstruction_ranks(rows, h, "hyp", K, D=D), args.reps, args.warmup)
    _, t_rf = timed(lambda: metrics.reconstruction_f1(rows, h, "hyp", K, D=D), args.reps, args.warmup)
    stage = []
    for _ in range(args.reps):
        st = {}
        metrics.link_prediction_ranks(rows, h, test, "hyp", K, D=D, stats=st, time_stages=True)
        stage.append(st["stage_ms"])
    rec = {"workload": name, "n": h.n, "D": D, "closure_edges": int(h.rank_slots()[0][-1]),
           "train": len(split["train"]), "val": len(val), "test": len(test), **info,
           "ranks_median_ms": t_rank["median_ms"], "ranks": t_rank,
           "stage_median_ms": {k: float(np.median([s[k] for s in stage])) for k in stage[0]},
           "f1_best_median_ms": t_best["median_ms"], "f1_best_rounds": f1_stats["rounds"],
           "f1_at_median_ms": t_at["median_ms"], "f1_at_rounds": at_stats["rounds"],
           "reconstruction_ranks_median_ms": t_rr["median_ms"], "reconstruction_f1_median_ms": t_rf["median_ms"],
           "counted_negatives": stats["counted_negatives"], "skipped_pairs": f1_stats["skipped_pairs"],
           "mean_rank": out["mean_rank"], "mean_rank_optimistic": out["mean_rank_optimistic"], "map": out["map"],
           "f1_best": float(best[0]), "threshold_best": float(best[1]), "threshold_val": t_val, "f1_at_val": float(at[0])}
    assert not math.isnan(rec["mean_rank"])
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--cfg4-steps", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("linkpred_bench needs a CUDA device")
    info = gpu_info()
    out = open(args.out, "w") if args.out else None

    def emit(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    h = H.random_tree(82115, 1.0831)
    rows, D = trained(h, 50, args.cfg4_steps)
    emit(workload("cfg4_hyp_D50_trained%d" % args.cfg4_steps, h, rows, D, args, info))
    h = H.random_dag(82115, 1.0831, 0.02)
    rows, D = trained(h, 50, args.cfg4_steps)
    emit(workload("cfg4dag002_hyp_D50_trained%d" % args.cfg4_steps, h, rows, D, args, info))


if __name__ == "__main__":
    main()
