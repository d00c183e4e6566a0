"""Reconstruction F1 over all node pairs (metrics.reconstruction_f1): time per call, rounds, open coarse bins, pairs/s,
and the issue bound from the pair count and the per-pair instructions of the built pass kernel; at n = 20 000 also the
materialised path (SIMT score matrix + torch.sort + lec_f1_sweep) in the same run, with the two rows compared.

    python scripts/recon_bench.py [--reps 5] [--warmup 2] [--out FILE]

Workloads: ETHEC hyp D = 10 after training (the reference's own size), random tree n = 20 000 D = 50 (A/B), cfg4 tree
n = 82 115 D = 50 after 2 000 ConeStep steps (no other path fits), and the cfg4-sized DAG random_dag(82 115, 1.0831,
0.02) D = 50 after as many steps (WordNet's nouns have several parents per node; lec_recon_pass_dag).  One JSON line
per workload.
"""
import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from learning_embeddings_b200 import _native as N, hierarchy as H, metrics, ops  # noqa: E402
from learning_embeddings_b200.engine import ConeStep, pack_index_block  # noqa: E402
from oracle import cones  # noqa: E402

K = 0.1
DEV = torch.device("cuda")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def pass_kernel_sass(DH, NT, PASS=1):
    """Static instructions of the tile loop of score_fast_kernel<HYP, DH, ., NT, 1, Pass(PASS)> (PASS = 1: Pass::F1,
    2: Pass::F1Dag; unrolled twice: 2 labels x RI images per trip) from cuobjdump -sass of the built object.  With
    Pass::F1Dag the loop holds, per label, the block-uniform branch of apexes with extra intervals and its binary-search loop, summarised separately."""
    obj = os.path.join(ROOT, "learning_embeddings_b200", "csrc", "build", "lec_recon.o")
    sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    sym = "_ZN3lec17score_fast_kernelILi1ELi%dELi" % DH
    blocks = sass.split("Function : ")
    body = next(b for b in blocks if b.startswith(sym) and b.split("\n", 1)[0].endswith("ELi%dELi1ELNS_4PassE%dEEEvNS_8FastArgsE" % (NT, PASS)))
    ins = []
    for line in body.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2)))
    addr = {a: i for i, (a, _) in enumerate(ins)}
    loops = []
    for i, (a, t) in enumerate(ins):
        m = re.search(r"\bBRA\b.*?(0x[0-9a-f]+)", t)
        if m and int(m.group(1), 16) < a and int(m.group(1), 16) in addr:
            loops.append((addr[int(m.group(1), 16)], i))
    ffma2 = lambda se: sum("FFMA2" in ins[k][1] for k in range(se[0], se[1] + 1))  # noqa: E731
    # innermost among the loops that do arithmetic (F1Dag's search loops hold no FFMA2 and sit inside the tile loop)
    inner = [(s, e) for s, e in loops
             if not any(s <= s2 and e2 <= e and (s2, e2) != (s, e) and ffma2((s2, e2)) for s2, e2 in loops)]
    s, e = max(inner, key=ffma2)
    body = [t for _, t in ins[s:e + 1]]
    rec = {"loop_instructions": len(body), "ffma2": sum("FFMA2" in t for t in body),
           "mufu": sum("MUFU" in t for t in body), "atomics": sum(("ATOM" in t or "RED" in t) for t in body)}
    if PASS == 2:
        search = [(s2, e2) for s2, e2 in loops if s <= s2 and e2 <= e and (s2, e2) != (s, e)]
        rec["search_loops"] = len(search)
        rec["search_loop_instructions"] = [e2 - s2 + 1 for s2, e2 in search]
        rec["search_loop_loads"] = [sum("LDG" in ins[k][1] for k in range(s2, e2 + 1)) for s2, e2 in search]
        # the branch that an apex without extra intervals jumps over: the nearest forward BRA before each search loop
        # whose target lies past it; what is left of the loop is the fast path every other apex runs
        skipped = 0
        for s2, e2 in search:
            for b in range(s2 - 1, s - 1, -1):
                m = re.search(r"\bBRA\b.*?(0x[0-9a-f]+)", ins[b][1])
                if m and int(m.group(1), 16) in addr and addr[int(m.group(1), 16)] > e2:
                    skipped += addr[int(m.group(1), 16)] - b - 1
                    break
        rec["branch_instructions"] = skipped
        rec["fast_path_instructions"] = len(body) - skipped
    return rec


def hyp_rows(h, D, seed=0):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(h.n, D, generator=g)
    r_in = cones.inner_radius(K)
    return ((r_in + 0.05 * torch.rand(h.n, 1, generator=g)) * w / w.norm(dim=1, keepdim=True)).to(DEV)


def trained(h, D, steps, B=2048, Nn=5):
    eng = ConeStep(hyp_rows(h, D), "hyp", Nn, B, K=K, alpha=0.05, lr=0.01)
    edges = h.closure_edges()
    rng = np.random.default_rng(0)
    for _ in range(steps):
        sel = rng.integers(0, len(edges), size=B)
        u, v = edges[sel, 0], edges[sel, 1]
        nt, nf = h.sample_negatives(u, v, Nn, rng)
        eng.step_device(*eng._split(pack_index_block(u, v, nt, nf).to(DEV), B))
    torch.cuda.synchronize()
    return eng.rows, eng.D


def timed(fn, reps, warmup):
    for _ in range(warmup):
        out = fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return out, {"median_ms": float(np.median(ms)), "min_ms": min(ms), "max_ms": max(ms), "reps": reps}


def materialised(rows, h, D):
    n = h.n
    x = rows[:, :D].contiguous()
    S = torch.empty((n, n), device=DEV, dtype=torch.float32)
    ops.score_topk_into(x, x, "hyp", K, [], [], 1, None, None, S, 1, engine="simt")
    tin = torch.as_tensor(h.tin, device=DEV)
    tout = torch.as_tensor(h.tout, device=DEV)
    pos = (tin[:, None] < tin[None, :]) & (tin[None, :] <= tout[:, None])
    off = ~torch.eye(n, dtype=torch.bool, device=DEV)
    ep, en = S[pos], S[off & ~pos]
    del S, pos, off
    return metrics.best_f1_sweep(ep, en)


def workload(name, h, rows, D, args, info, sass, ab=False):
    n = h.n
    stats = {}
    row, t = timed(lambda: metrics.reconstruction_f1(rows, h, "hyp", K, D=D, stats=stats), args.reps, args.warmup)
    pairs = n * (n - 1)
    passes = stats["rounds"]
    RI = 4 if (D + 1) // 2 <= 8 else 2
    # one trip: 2 labels x RI images per thread; for a DAG the fast path (apexes with extra intervals, a few percent,
    # also run the skipped branch: the bound leaves that out)
    per_pair = sass.get("fast_path_instructions", sass["loop_instructions"]) / (2 * RI)
    clk = float(info["max_sm_clock"].split()[0]) * 1e6
    bound_ms = passes * pairs * per_pair / 32 / (148 * 4 * clk) * 1e3   # 4 warp instructions per clock per SM
    rec = {"workload": name, "n": n, "D": D, "pairs": pairs, **info, **t, "rounds": passes,
           "open_bins": stats["open_bins"], "n_pos": stats["n_pos"], "n_neg": stats["n_neg"],
           "workspace_mb": stats["workspace_bytes"] / 2**20, "pairs_per_s": pairs / (t["median_ms"] * 1e-3),
           "pair_evals_per_s": passes * pairs / (t["median_ms"] * 1e-3), "pass_loop_sass": sass,
           "sass_instr_per_pair": per_pair, "issue_bound_ms": bound_ms, "extra_intervals": stats["extra_intervals"],
           "row": [float(v) for v in row]}
    if ab:
        torch.cuda.empty_cache()
        ref, tm = timed(lambda: materialised(rows, h, D), args.reps, args.warmup)
        rec["materialised"] = tm
        rec["materialised_row"] = [float(v) for v in ref]
        rec["rows_equal"] = bool(np.array_equal(row, ref, equal_nan=True))
        rec["speedup"] = tm["median_ms"] / t["median_ms"]
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cfg4-steps", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recon_bench needs a CUDA device")
    info = gpu_info()
    sass10, sass50 = pass_kernel_sass(5, 512), pass_kernel_sass(25, 256)
    lines = []
    h = H.ethec()
    rows, D = trained(h, 10, 1000)
    lines.append(workload("ethec_hyp_D10_trained", h, rows, D, args, info, sass10))
    h = H.random_tree(20000, 1.0831)
    lines.append(workload("tree20000_hyp_D50_ab", h, hyp_rows(h, 50), 50, args, info, sass50, ab=True))
    h = H.random_tree(82115, 1.0831)
    rows, D = trained(h, 50, args.cfg4_steps)
    lines.append(workload("cfg4_hyp_D50_trained%d" % args.cfg4_steps, h, rows, D, args, info, sass50))
    h = H.random_dag(82115, 1.0831, 0.02)
    rows, D = trained(h, 50, args.cfg4_steps)
    lines.append(workload("cfg4dag002_hyp_D50_trained%d" % args.cfg4_steps, h, rows, D, args, info,
                          pass_kernel_sass(25, 256, PASS=2)))
    lines[-1]["pair_evals_per_s_vs_cfg4_tree"] = lines[-1]["pair_evals_per_s"] / lines[-2]["pair_evals_per_s"]
    out = open(args.out, "w") if args.out else None
    for rec in lines:
        s = json.dumps(rec)
        print(s)
        if out:
            out.write(s + "\n")


if __name__ == "__main__":
    main()
