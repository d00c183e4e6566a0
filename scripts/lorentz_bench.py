"""Lorentz-model embeddings (Nickel & Kiela 2018): device time of a ConeStep("lorentz") step and of its pair kernel
alone, the time of reconstruction_ranks on Lorentz rows, and ETHEC's reconstruction MAP / mean rank after a fixed number
of steps against the initial table -- the measurements of poincare_bench.py on the hyperboloid.

    python scripts/lorentz_bench.py [--steps 200] [--warmup 20] [--train-steps 1000] [--out FILE]

Workloads: the cfg4 tree random_tree(82 115, 1.0831) at D = 10 and 50, and ETHEC at D = 10; N = 50 negatives (Philox
draws of the sampler, made before the timed window), B = 2 520 positives, lr 0.3 after 20 burn-in steps at 0.01, from a
uniform(-1e-3, 1e-3) table.  Step times are CUDA events around each step (median after the warm-up); the pair kernel's
are the events lec_cone_step records around it.  One JSON line per workload, with the GPU's name and power limit read in
the same run.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from learning_embeddings_b200 import hierarchy as H, metrics  # noqa: E402
from learning_embeddings_b200.engine import ConeStep  # noqa: E402
from learning_embeddings_b200.sampler import SamplerGraph  # noqa: E402
from poincare_bench import B, LR, N_NEG, batches, time_steps, train  # noqa: E402
from recon_bench import gpu_info, timed  # noqa: E402


def engine(h, D, seed=0):
    g = torch.Generator().manual_seed(seed)
    W0 = (torch.rand(h.n, D, generator=g) * 2 - 1) * 1e-3
    return ConeStep(W0.cuda(), "lorentz", N_NEG, B, lr=LR)


def workload(name, h, D, args, info, rank_timing):
    graph = SamplerGraph.from_hierarchy(h)
    data = batches(h, graph, 16, seed=1)
    eng = engine(h, D)
    init = eng.table.clone()
    step_ms, pair_ms = time_steps(eng, data, args.steps, args.warmup)
    rec = {"workload": name, "n": h.n, "D": D, "B": B, "N": N_NEG, "closure_edges": len(h.closure_edges()), **info,
           "step_median_ms": step_ms, "pair_kernel_median_ms": pair_ms,
           "pairs_per_s": B * (N_NEG + 1) / (step_ms * 1e-3)}
    if rank_timing:
        r, t = timed(lambda: metrics.reconstruction_ranks(eng.rows, h, "lorentz", None, D=D), 3, 1)
        rec.update({"reconstruction_ranks_median_ms": t["median_ms"], "after_steps": args.warmup + args.steps,
                    "map": r["map"], "mean_rank": r["mean_rank"]})
    else:
        r0 = metrics.reconstruction_ranks(init, h, "lorentz", None)
        fresh = engine(h, D)
        train(fresh, data, args.train_steps)
        torch.cuda.synchronize()
        r1 = metrics.reconstruction_ranks(fresh.table, h, "lorentz", None)
        radius = torch.asinh(fresh.table.double().norm(dim=1))
        rec.update({"train_steps": args.train_steps, "map_initial": r0["map"], "mean_rank_initial": r0["mean_rank"],
                    "map_trained": r1["map"], "mean_rank_trained": r1["mean_rank"],
                    "max_radius_trained": float(radius.max())})
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--train-steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lorentz_bench.py measures on a GPU; none is visible")
    info = gpu_info()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    emit(workload("ethec_D10", H.ethec(), 10, args, info, rank_timing=False))
    cfg4 = H.random_tree(82115, 1.0831)
    for D in (10, 50):
        emit(workload("cfg4_D%d" % D, cfg4, D, args, info, rank_timing=True))


if __name__ == "__main__":
    main()
