#!/usr/bin/env python
"""Benchmark of the entailment-cone hot path (BASELINE.json: cone pairs/s fwd+bwd; image x label scores/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload all|cfg0|cfg1|cfg2|cfg3|cfg4]

Prints ONE JSON line (rank 0).  The headline (metric / value / e2e / roofline / cpu_baseline) is workload cfg1
(BASELINE.json configs[1]: Poincare cones, label-only, ETHEC 723-node hierarchy, D=10, RSGD, 10 negatives per edge; the
1 974 closure edges tiled to --pairs pairs per GPU per step, every step a different pre-sampled batch out of a rotation
larger than L2).  One "step" = one pass of the hot path over one batch: fused cone loss fwd+bwd over B*(1+2N) pairs ->
fused update (replica sum, [gradient exchange over NVLink peer memory], RSGD, next step's row transform).

With --workload all (the default, what the driver runs) the same line carries a "workloads" object with short runs of
the other BASELINE configs at the same GPU count -- cfg0 (Euclidean cones, D=2, Adam), cfg2 (joint image+label step),
cfg3 (all-pairs scoring, D=10 and D=50; matrix / top-k / both), cfg4 (82 K-node tree, D=50) -- each with its own value,
ms_per_step, roofline, e2e and clocks; plus, on the headline, a `sustained` record (>= 1 s of back-to-back steps) and,
at N > 1, a `parity` record (table replicas bit-identical across ranks; one sharded step against the same step on one
GPU).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cone pairs/s fwd+bwd"
UNIT = "pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "cfg0", "cfg1", "cfg2", "cfg3", "cfg4"])
    ap.add_argument("--dim", type=int, default=10, help="cfg3: embedding dimension (10 or 50)")
    ap.add_argument("--images", type=int, default=1000000, help="cfg3: images per GPU per step")
    ap.add_argument("--score-mode", default="both", choices=["both", "matrix", "topk"],
                    help="cfg3: what a step writes: per-level top-5 + the full [L, N] energy matrix, or one of them")
    ap.add_argument("--engine", default="auto", choices=["auto", "tc", "simt"], help="cfg3: scoring engine")
    ap.add_argument("--pairs", type=int, default=0, help="pairs per GPU per step (0 = per workload: 2^21, cfg4 131 040)")
    ap.add_argument("--precision", type=int, default=None, help="0 fp32 core, 1 fp64 core (default: per workload)")
    ap.add_argument("--rotation", type=int, default=0, help="distinct batches to rotate through (0 = enough to exceed L2)")
    ap.add_argument("--comm", default="auto", choices=["auto", "p2p", "nccl"],
                    help="multi-GPU gradient exchange: packet all-reduce over peer memory inside the update kernel, or NCCL")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--step-series", type=int, default=0, help="diagnostic: print the device time of each of N steps")
    ap.add_argument("--burst-ab", action="store_true", help="diagnostic: the timed burst under several launch-queue depths")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32 / float64, at "
                         "most 64 MB in all), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the outputs of --impl b200")
    return args


class Ctx:
    """Rank / device / process group of this process (one process per GPU under torchrun)."""

    def __init__(self, need_gpu):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dev, self.pg = None, None
        if need_gpu:
            if not torch.cuda.is_available():
                raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
            torch.cuda.set_device(self.local_rank)
            self.dev = torch.device("cuda", self.local_rank)
            if self.world > 1:
                import torch.distributed as dist
                dist.init_process_group("nccl", device_id=self.dev)
                self.pg = dist.group.WORLD

    def sync_all(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def align_streams(self):
        """Device-side rendezvous enqueued right before a timed region's start event: the ranks' host threads leave
        barrier() tens of microseconds apart, and with a 1.3 ms region that skew would be charged to the first step.  A
        one-element all-reduce completes on every GPU at (nearly) the same moment, so the streams start the region
        together; the host has the region's launches queued behind it."""
        if self.world > 1:
            if getattr(self, "_tok", None) is None:
                self._tok = torch.zeros(1, device=self.dev)
            torch.distributed.all_reduce(self._tok)

    def warm(self, dev_step, eng, kev, warmup):
        """Untimed warm-up: at least 40 steps whatever --warmup says (r2w8: at 8 GPUs the first ~25 steps of a process ran
        ~20 % slow -- peer mappings, lazily loaded modules, first use of the event path -- and a 5-step warm-up put them
        inside the 20-step timed region: 88.7 us/step against 72.7 for the same region a moment later), including one
        rehearsal of the timed loop itself (kernel events, rendezvous, spin kernel)."""
        for i in range(max(3, warmup, 40)):
            dev_step(i)
        self.sync_all()
        self.align_streams()
        self.prequeue()
        for i in range(len(kev)):
            eng.kernel_events = kev[i] if i % 4 == 0 else None
            dev_step(i)
        eng.kernel_events = None
        self.sync_all()

    def prequeue(self):
        """~0.5 ms spin kernel in front of a timed region's start event: by the time the GPU reaches the event the host has
        the region's launches queued, so a 20-step (1.3 ms) region times the device back to back and not the host's
        launch jitter -- with 8 lock-stepped ranks ANY rank's hiccup in an empty launch queue stalls all of them (r2u8:
        20 steps 80.9 us/step, 200 steps 75.4, one second sustained 71.8).  The host side is what `e2e` measures."""
        if os.environ.get("LEC_BENCH_PREQUEUE", "1") != "0":
            torch.cuda._sleep(1_000_000)

    def max_ranks(self, ms):
        if self.world > 1:
            tt = torch.tensor([ms], device=self.dev, dtype=torch.float64)
            torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
            return float(tt.item())
        return ms

    def close(self):
        if self.world > 1 and self.dev is not None:
            torch.distributed.destroy_process_group()


DUMP_BYTES = 64 << 20


def snapshot(arrays):
    """Host copies of the named device tensors, taken right after a timed region (later regions keep training the same
    table).  Floating-point tensors keep float64 or become float32, integer ones become float64 (exact).  A tensor
    larger than its share of DUMP_BYTES is cut to a sample of its flattened elements: the positions are drawn with a
    fixed seed from its size alone, so two runs with the same arguments sample the same elements."""
    share = (DUMP_BYTES - 4096 * len(arrays)) // len(arrays)   # 4 KB per file for the .npy header
    out = {}
    for name, t in arrays.items():
        t = t.detach()
        dt = torch.float64 if (t.dtype == torch.float64 or not t.is_floating_point()) else torch.float32
        k = share // dt.itemsize
        if t.numel() > k:
            pos = np.sort(np.random.default_rng(0).choice(t.numel(), size=k, replace=False))
            t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
        out[name] = t.to(dt).cpu().numpy()
    return out


def restarter(eng, initial, moments):
    """With --dump-outputs the last timed step starts from the seeded initial state: the step sums its gradients with
    float atomics in no fixed order, and over many steps the hinge thresholds turn those last-bit differences into
    different trajectories, so only a step from a fixed state computes the same outputs in every run.  Returns the
    reset: each (parameter, initial device copy) pair is copied back, optimizer moments and step count restart, and the
    engine re-derives its rows from the table (one copy and one extra launch inside the timed region)."""
    def restart():
        for dst, src in initial:
            dst.copy_(src, non_blocking=True)
        for m in moments:
            m.zero_()
        eng.opt_step = 0
        eng.invalidate_rows()
    return restart


def write_dump(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# workload definitions
# ------------------------------------------------------------------------------------------------
def workload_spec(name):
    if name == "cfg0":
        # BASELINE.json configs[0] (the reference's own CPU case: D=2, Embedder K=3, alpha=0.05, N=5, Adam,
        # order_embeddings.py:1364) with the ETHEC closure edges tiled to the cfg1 batch size, so that the Euclidean
        # pair kernel is measured at a size that fills the GPU
        return dict(name="cfg0: Euclidean cones, label-only, ETHEC 723-node hierarchy, D=2, Adam, 10 negatives/edge",
                    geom="euc", D=2, n_neg=5, K=3.0, alpha=0.05, lr=1e-3, tree="ethec", pairs=1 << 21)
    if name == "cfg1":
        return dict(name="cfg1: Poincare cones, label-only, ETHEC 723-node hierarchy, D=10, RSGD, 10 negatives/edge",
                    geom="hyp", D=10, n_neg=5, K=0.1, alpha=0.05, lr=1e-3, tree="ethec", pairs=1 << 21)
    return dict(name="cfg4: Poincare cones, 82115-node random tree, D=50, RSGD, 50 negatives/edge",
                geom="hyp", D=50, n_neg=25, K=0.1, alpha=0.05, lr=1e-3, tree="random82k", pairs=131040)


def build_hierarchy(spec):
    from learning_embeddings_b200 import hierarchy as H
    if spec["tree"] == "ethec":
        return H.ethec()
    return H.random_tree(82115, 1.0831, seed=0)


def init_table(n, D, K, seed):
    """order_embeddings_h.py:198-203: N(0,1) direction, norm r_in + U[0, 0.05)."""
    from learning_embeddings_b200.criterion import inner_radius
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(n, D, generator=g)
    return (inner_radius(K) + 0.05 * torch.rand(n, 1, generator=g)) * w / w.norm(dim=1, keepdim=True)


def make_batches(h, spec, groups, count, seed, pos_only=False):
    """`count` host index blocks of `groups` positives each (closure edges tiled in shuffled order)."""
    from learning_embeddings_b200.engine import pack_index_block, index_dtype_for
    rng = np.random.default_rng(seed)
    dt = index_dtype_for(h.n)
    edges = h.closure_edges()
    out = []
    for _ in range(count):
        sel = rng.integers(0, len(edges), size=groups)
        u, v = edges[sel, 0], edges[sel, 1]
        if pos_only:
            out.append(pack_index_block(u, v, np.zeros(0, np.int64), np.zeros(0, np.int64), dtype=dt, n_rows=h.n))
            continue
        neg_to, neg_from = h.sample_negatives(u, v, spec["n_neg"], rng)
        out.append(pack_index_block(u, v, neg_to, neg_from, dtype=dt, n_rows=h.n))
    return out


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.active = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        while not self._stop_evt.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                    r = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.0005 if self.active.is_set() else 0.002)

    def stop(self):
        self._stop_evt.set()

    def reset(self):
        self.samples, self.reasons = [], set()

    def summary(self):
        return {"sm_mhz": (float(np.median(self.samples)) if self.samples else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the reference's PyTorch-on-CPU step)
# ------------------------------------------------------------------------------------------------
def cpu_step_runner(spec, table, blk, B):
    """Returns a closure running one full reference-style step on the host cores: gather + row transform
    + E_operator + hinge + backward (autograd) + table update, all in torch fp32 on CPU."""
    from oracle import cones
    Nn = spec["n_neg"]
    b = torch.from_numpy(blk[:B * (2 + 2 * Nn)].numpy().astype(np.int64))
    u, v = b[:B], b[B:2 * B]
    neg_to = b[2 * B:2 * B + B * Nn].view(B, Nn)
    neg_from = b[2 * B + B * Nn:].view(B, Nn)
    nf = torch.cat([u[:, None].expand(B, Nn), neg_from], 1).reshape(-1)
    nt = torch.cat([neg_to, v[:, None].expand(B, Nn)], 1).reshape(-1)
    W = table.clone()
    if spec["geom"] == "euc":
        # order_embeddings.py: Embedder.soft_clip rows, EucConesLoss, torch Adam on the table
        P = torch.nn.Parameter(W, requires_grad=False)
        opt = torch.optim.Adam([P], lr=spec["lr"])

        def run_euc():
            r = cones.label_step("euc", P.data, cones.ROW_EUC_SOFTCLIP, spec["K"], spec["alpha"], u, v, nf, nt)
            P.grad = r["gW"]
            opt.step()
            return float(r["loss"])

        return run_euc
    r_in = cones.inner_radius(spec["K"])

    def run():
        nonlocal W
        r = cones.label_step(spec["geom"], W, cones.ROW_HYP_SHELL, spec["K"], spec["alpha"], u, v, nf, nt)
        _, W = cones.rsgd_step(W, r["gW"], spec["lr"], r_in)
        return float(r["loss"])

    return run


def time_cpu(spec, table, blk, groups, steps, warmup, budget_s=25.0):
    """`groups` positives (x(1+2N) pairs) per CPU step; stops after `steps` steps or budget_s seconds."""
    torch.set_num_threads(os.cpu_count() or 1)
    run = cpu_step_runner(spec, table, blk, groups)
    for _ in range(warmup):
        run()
    times = []
    t_all = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    pairs = groups * (1 + 2 * spec["n_neg"])
    return pairs / float(np.mean(times)), float(np.mean(times)), len(times), pairs


# ------------------------------------------------------------------------------------------------
# label-only training workloads (cfg0, cfg1, cfg4)
# ------------------------------------------------------------------------------------------------
def label_geometry(args, wl):
    spec = workload_spec(wl)
    Nn, D = spec["n_neg"], spec["D"]
    ppg = 1 + 2 * Nn
    groups = max(1, (args.pairs or spec["pairs"]) // ppg)
    return spec, Nn, D, ppg, groups


def run_label_reference(args, ctx, wl):
    """--impl reference: the reference's CPU path (oracle port, torch fp32 on every host core) on the SAME step --
    the same number of pairs per step as the GPU arm."""
    if ctx.rank != 0:
        return None
    spec, Nn, D, ppg, groups = label_geometry(args, wl)
    h = build_hierarchy(spec)
    table0 = init_table(h.n, D, spec["K"], seed=0)
    if spec["geom"] == "euc":
        table0 = torch.randn(h.n, D, generator=torch.Generator().manual_seed(0))
    blk = make_batches(h, spec, groups, 1, seed=1)[0]
    v, mean_s, n_done, pairs = time_cpu(spec, table0, blk, groups, args.steps, min(args.warmup, 3), budget_s=240.0)
    from learning_embeddings_b200.engine import index_dtype_for
    cfg = {"workload": spec["name"], "pairs_per_gpu_per_step": pairs, "positives_per_gpu_per_step": groups, "dim": D,
           "negatives_per_edge": 2 * Nn, "table_rows": int(h.n), "update": "adam" if spec["geom"] == "euc" else "rsgd",
           "scalar_core": "fp32", "index_dtype": np.dtype(index_dtype_for(h.n)).name, "parallelism": "host cores only"}
    cores = os.cpu_count() or 1
    sample = "the full step (%d pairs, %d positives), %d timed steps, torch fp32 on all host threads" % (pairs, groups, n_done)
    return {"metric": METRIC, "value": v, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": n_done,
            "warmup": min(args.warmup, 3), "ms_per_step": mean_s * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def run_label(args, ctx, wl, steps, warmup, headline=False, dump=None):
    from learning_embeddings_b200 import _native
    from learning_embeddings_b200.engine import ConeStep, index_dtype_for, pack_index_block
    from learning_embeddings_b200 import sharding
    spec, Nn, D, ppg, groups = label_geometry(args, wl)
    pairs_per_step = groups * ppg
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    precision = args.precision if args.precision is not None else 1
    h = build_hierarchy(spec)
    idx_dt = index_dtype_for(h.n)
    idx_bytes = np.dtype(idx_dt).itemsize
    cfg = {"workload": spec["name"], "pairs_per_gpu_per_step": pairs_per_step, "positives_per_gpu_per_step": groups,
           "dim": D, "negatives_per_edge": 2 * Nn, "table_rows": int(h.n), "update": "rsgd",
           "scalar_core": "fp64" if precision == 1 else "fp32", "index_dtype": np.dtype(idx_dt).name,
           "parallelism": "dp%d (pairs sharded, table replicated)" % world}
    table0 = init_table(h.n, D, spec["K"], seed=0)
    if spec["geom"] == "euc":
        table0 = torch.randn(h.n, D, generator=torch.Generator().manual_seed(0))   # nn.Embedding default init
        cfg["update"] = "adam (torch.optim.Adam semantics inside the fused update kernel)"
        cfg["scalar_core"] = "fp32"

    bytes_per_batch = groups * (2 + 2 * Nn) * idx_bytes + groups * ppg * 4  # indices in + energies out
    rotation = args.rotation or max(4, int(np.ceil(160e6 / bytes_per_batch)))
    cfg["l2_policy"] = "inputs rotate through %d distinct batches (%.0f MB > 126 MB L2)" % (
        rotation, rotation * bytes_per_batch / 1e6)
    if ctx.world > 1:
        cfg["start_alignment"] = "device-side rendezvous (one-element all-reduce) enqueued right before the start event"
    cfg["launch_queue"] = "a ~0.5 ms spin kernel precedes the start event, so the timed launches are queued before the GPU reaches them"
    cfg["warmup_steps"] = "max(--warmup, 40) steps + one untimed rehearsal of the timed loop"
    host_batches = make_batches(h, spec, groups, rotation, seed=100 + (0 if os.environ.get("LEC_BENCH_SAME_BATCHES") else rank))
    dev_batches = [b.to(dev) for b in host_batches]
    table = table0.to(dev).clone()
    eng = ConeStep(table, spec["geom"], Nn, groups, K=spec["K"], alpha=spec["alpha"], lr=spec["lr"],
                   precision=precision, process_group=ctx.pg, comm=args.comm,
                   update="adam" if spec["geom"] == "euc" else "auto")
    cfg["exchange"] = (eng.comm + (" " + eng.comm_note if eng.comm_note else "")) if world > 1 else "none (1 GPU)"

    def dev_step(i):
        eng.step_device(*eng._split(dev_batches[i % rotation], groups))

    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    ctx.warm(dev_step, eng, kev, warmup)
    restart = None
    if args.dump_outputs:
        restart = restarter(eng, [(table, table0.to(dev))], [m for m in (eng.opt_m, eng.opt_v) if m is not None])
        cfg["dump_outputs"] = "the last timed step starts from the seeded initial table"

    # timed region: inputs resident in HBM
    launches0 = _native.launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active.set()
    ctx.align_streams()   # warm the collective up before the bracket
    ctx.sync_all()
    ctx.align_streams()
    ctx.prequeue()
    t0.record()
    for i in range(steps):
        # the pair kernel is bracketed by CUDA events on every 4th step only: two event records per step sit between
        # back-to-back launches and cost more than they measure
        eng.kernel_events = kev[i] if i % 4 == 0 else None
        if restart is not None and i == steps - 1:
            restart()
        dev_step(i)
    t1.record()
    ctx.sync_all()
    sampler.active.clear()
    eng.kernel_events = None
    lec_launches = _native.launch_count() - launches0
    elapsed_ms = ctx.max_ranks(t0.elapsed_time(t1))
    kernel_ms = float(np.mean([a.elapsed_time(b) for i, (a, b) in enumerate(kev) if i % 4 == 0]))
    last_loss = eng.global_loss()
    final_loss = float(last_loss.item())
    if dump is not None:
        # the step's loss, the table it updated in place, and the pair energies of this rank's share of the batch
        dump.update(snapshot({"loss": last_loss, "table": table, "E_pos": eng.E_pos[:groups], "E_neg": eng.E_neg[:groups]}))
    value = world * pairs_per_step * steps / (elapsed_ms * 1e-3)
    clocks = sampler.summary()

    if args.burst_ab:
        # diagnostic: the 20-step burst under different launch-queue depths, with and without the NVML sampler thread
        for rep in range(3):
            for spin_cycles in (0, 1_000_000, 4_000_000):
                for samp in (True, False):
                    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    if samp:
                        sampler.active.set()
                    ctx.align_streams()
                    ctx.sync_all()
                    ctx.align_streams()
                    if spin_cycles:
                        torch.cuda._sleep(spin_cycles)
                    b0.record()
                    for i in range(steps):
                        eng.kernel_events = kev[i] if i % 4 == 0 else None
                        dev_step(i)
                    b1.record()
                    ctx.sync_all()
                    sampler.active.clear()
                    eng.kernel_events = None
                    ms = ctx.max_ranks(b0.elapsed_time(b1))
                    if rank == 0:
                        print("burst rep %d spin %.1f ms sampler %s: %.1f us/step" % (rep, spin_cycles / 1.965e6, samp, 1e3 * ms / steps),
                              file=sys.stderr, flush=True)

    if args.step_series:
        # diagnostic: device time of every step of a short region (one event per step), rank 0 prints the series
        for tag, pre in (("plain", False), ("prequeued", True)):
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.step_series + 1)]
            ctx.sync_all()
            ctx.align_streams()
            if pre:
                ctx.prequeue()
            evs[0].record()
            for i in range(args.step_series):
                dev_step(i)
                evs[i + 1].record()
            ctx.sync_all()
            if rank == 0:
                print("step series (%s, us): %s" % (tag, " ".join("%.1f" % (1e3 * evs[i].elapsed_time(evs[i + 1]))
                                                                  for i in range(args.step_series))), file=sys.stderr, flush=True)

    if args.step_series:
        # debug builds of the library (-DLEC_STEP_TRACE) stamp the phases of a step with %globaltimer
        import ctypes
        try:
            tracer = _native.lib().lec_debug_step_trace
        except AttributeError:
            tracer = None
        if tracer is not None:
            buf = (ctypes.c_uint64 * 7)()
            tracer(None)
            acc, cnt = np.zeros(6), 0
            for i in range(40):
                ctx.sync_all()
                ctx.align_streams()
                dev_step(i)
                torch.cuda.synchronize()
                tracer(buf)
                t = [int(v) for v in buf]
                if i >= 5:
                    acc += np.array([t[1] - t[0], t[2] - t[1], t[3] - t[2], t[4] - t[3], t[5] - t[4], t[6] - t[5]], dtype=np.float64)
                    cnt += 1
            print("rank %d step phases (us): pair kernel %.1f | pair end -> update past its wait %.1f | update blocks enter over %.1f | "
                  "-> packets pushed %.1f | -> reduced %.1f | -> update end %.1f" % ((rank,) + tuple(acc / cnt / 1e3)),
                  file=sys.stderr, flush=True)

    # sustained: at least a second of back-to-back steps, same rotation (the burst figure above is 20 steps ~ 1.4 ms)
    sustained = None
    if headline and not args.no_sustained:
        n_sus = int(min(60000, max(steps, np.ceil(1.1e3 / max(elapsed_ms / steps, 1e-3)))))
        sampler.reset()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.sync_all()
        sampler.active.set()
        ctx.align_streams()
        s0.record()
        for i in range(n_sus):
            dev_step(i)
        s1.record()
        ctx.sync_all()
        sampler.active.clear()
        sus_ms = ctx.max_ranks(s0.elapsed_time(s1))
        sustained = {"steps": n_sus, "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus,
                     "value": world * pairs_per_step * n_sus / (sus_ms * 1e-3), "unit": UNIT,
                     "vs_burst": (sus_ms / n_sus) / (elapsed_ms / steps), "clocks": sampler.summary()}
        sampler.reset()

    # multi-GPU parity, outside every timed region: replicas bit-identical; one sharded step == the same step on one GPU
    parity = None
    if headline and world > 1:
        import torch.distributed as dist
        ref = table.clone()
        dist.broadcast(ref, 0)
        same = torch.tensor([1.0 if torch.equal(ref, table) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        replicas_identical = bool(same.item() == 1.0)
        vg = min(groups, 32768)
        Bg = vg * world
        vb = make_batches(h, spec, Bg, 1, seed=4242)[0]                  # the same global batch on every rank
        u_, v_, nt_, nf_ = (x.numpy() for x in (vb[:Bg], vb[Bg:2 * Bg], vb[2 * Bg:2 * Bg + Bg * Nn], vb[2 * Bg + Bg * Nn:]))
        nt_, nf_ = nt_.reshape(Bg, Nn), nf_.reshape(Bg, Nn)
        before = table.clone()
        su, sv, snt, snf = sharding.shard_groups(u_, v_, nt_, nf_, rank, world)
        part = pack_index_block(su, sv, snt, snf, dtype=idx_dt, pin=False).to(dev)
        eng.step_device(*eng._split(part, len(su)))
        loss_multi = float(eng.global_loss().item())
        one = ConeStep(before.clone(), spec["geom"], Nn, Bg, K=spec["K"], alpha=spec["alpha"], lr=spec["lr"],
                       precision=precision, update="adam" if spec["geom"] == "euc" else "auto")
        one.opt_step = eng.opt_step - 1
        full = vb.to(dev)
        one.step_device(*one._split(full, Bg))
        torch.cuda.synchronize()
        loss_single = float(one.loss.item())
        parity = {"replicas_identical": replicas_identical,
                  "loss_rel_diff_vs_single_gpu_step": abs(loss_multi - loss_single) / max(abs(loss_single), 1e-30),
                  "table_max_abs_diff_vs_single_gpu_step": float((table - one.table).abs().max()),
                  "positives_in_check": Bg}

    # end to end through the public host API, every step: host index block -> H2D -> step -> loss D2H.
    # "host_negatives": ConeStep.submit_host / drain (the whole index block, negatives drawn by the caller -- the
    # bit-exact reference sampler's mode); "device_sampled": ConeStep.submit_host_sampled (only the positive edges
    # cross PCIe, negatives drawn by the library's Philox sampler on the GPU).  The copy of step i+1 overlaps step i;
    # every step's loss is delivered.  "sync" = ConeStep.step_host (loss returned before the next step is issued).
    e2e = None
    if not args.no_e2e:
        def timed(fn_step, fn_end, n):
            for i in range(3):
                fn_step(i)
            fn_end()
            ctx.sync_all()
            sampler.active.set()
            w0 = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                fn_step(i)
            got = fn_end()
            e1.record()
            ctx.sync_all()
            sampler.active.clear()
            return ctx.max_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3)), got

        sync_ms, _ = timed(lambda i: eng.step_host(host_batches[i % rotation], groups), lambda: None, steps)
        pipe_ms, losses = timed(lambda i: eng.submit_host(host_batches[i % rotation], groups), eng.drain, steps)
        assert len(losses) == steps, "every step's loss must come back to the host"
        host_neg = {"value": world * pairs_per_step * steps / (pipe_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": groups * (2 + 2 * Nn) * idx_bytes, "d2h_bytes_per_step": 8,
                    "ms_per_step": pipe_ms / steps, "api": "ConeStep.submit_host/drain (copy of step i+1 overlaps step i)"}
        e2e = dict(host_neg)
        e2e["mode"] = "host_negatives"
        try:
            from learning_embeddings_b200.sampler import SamplerGraph
            graph = SamplerGraph.from_hierarchy(h)
            pos_blocks = make_batches(h, spec, groups, min(rotation, 8), seed=300 + rank, pos_only=True)
            samp_ms, losses2 = timed(lambda i: eng.submit_host_sampled(graph, pos_blocks[i % len(pos_blocks)], groups, 7),
                                     eng.drain, steps)
            assert len(losses2) == steps and all(np.isfinite(losses2))
            dev_samp = {"value": world * pairs_per_step * steps / (samp_ms * 1e-3), "unit": UNIT,
                        "h2d_bytes_per_step": groups * 2 * idx_bytes, "d2h_bytes_per_step": 8,
                        "ms_per_step": samp_ms / steps,
                        "api": "ConeStep.submit_host_sampled/drain (positive edges in, negatives drawn on the GPU by "
                               "lec_sample_negatives_philox inside the step)"}
            if dev_samp["value"] > e2e["value"]:
                e2e = dict(dev_samp)
                e2e["mode"] = "device_sampled"
            e2e["host_negatives"] = host_neg
            e2e["device_sampled"] = dev_samp
        except Exception as ex:  # noqa: BLE001 -- the sampled mode is an extra; report, do not lose the line
            if world > 1:
                raise
            e2e["device_sampled"] = {"error": "%s: %s" % (type(ex).__name__, str(ex)[:200])}
        e2e["sync"] = {"value": world * pairs_per_step * steps / (sync_ms * 1e-3), "ms_per_step": sync_ms / steps,
                       "api": "ConeStep.step_host (loss returned before the next step is issued)"}
    sampler.stop()
    if rank != 0:
        return None

    # roofline of the dominant kernel (the fused pair kernel): algorithmic bytes model of SURVEY.md 8(d)
    peak, peak_src = hbm_peak()
    bytes_per_pair = 24 + 16 * D
    achieved = pairs_per_step * bytes_per_pair / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic_%s.json" % wl)
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    step_ms = elapsed_ms / steps
    roofline = {"bound": "hbm", "kernel": "pairs_grouped_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "traffic_source": ("ncu --set full capture of this kernel on this workload (profiles/traffic_%s.json), not "
                                   "re-measured in this run" % wl) if traffic is not None else None,
                "algorithmic_bytes_per_pair": bytes_per_pair, "kernel_ms": kernel_ms,
                "kernel_share_of_step": kernel_ms / step_ms,
                "step_frac": pairs_per_step * bytes_per_pair / (step_ms * 1e-3) / 1e9 / peak,
                "update_kernel": {"name": "update_rows_kernel", "ms": max(step_ms - kernel_ms, 0.0),
                                  "algorithmic_bytes": 12 * D * int(h.n),
                                  "note": "step minus pair kernel; 12*D bytes per table row (read w, read g, write w)"},
                "note": "logical-bytes model (24+16*D B per pair); the table is L2/L1-resident so DRAM traffic is far "
                        "below it -- the kernel is bound by FP32/FP64 issue and L2 vector reductions, not HBM"}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        budget = 20.0 if headline else 6.0
        v, mean_s, n_done, pairs = time_cpu(spec, table0, host_batches[0], groups, steps=20, warmup=1, budget_s=budget)
        cpu = {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
               "sample": "%d pairs per CPU step (the same batch 0 the GPU runs), %d steps, torch fp32 on all host "
                         "threads, same step (gather+transform+energy+hinge+backward+update)" % (pairs, n_done)}
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(3, warmup),
           "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e,
           "gpu_launches": int(lec_launches), "roofline": roofline, "cpu_baseline": cpu, "final_loss": final_loss}
    if sustained is not None:
        out["sustained"] = sustained
        if not clocks["samples"]:
            # the burst region (steps x ~65 us) can end before NVML answers once: the sustained region right behind it is
            # the same kernel sequence under the same conditions
            out["clocks"] = dict(sustained["clocks"], note="no NVML sample fell inside the %.1f ms burst region; these are "
                                 "the samples of the sustained region that follows it" % elapsed_ms)
    if parity is not None:
        out["parity"] = parity
    return out


# ------------------------------------------------------------------------------------------------
# cfg2: joint image+label Euclidean cones (BASELINE.json configs[2]; SURVEY 8(d))
# ------------------------------------------------------------------------------------------------
CFG2 = dict(name="cfg2: joint image+label Euclidean cones, 2048-d features -> FeatNet -> D=10, ETHEC labels, "
                 "23831 positives x (1+10) = 262141 pairs/step, 16384 distinct images/step, Adam",
            geom="euc", D=10, n_neg=5, K=3.0, alpha=1.0, lr=1e-3, lr_labels=0.1, B=23831, m=16384, F=2048, pool=65536)


def make_joint_batches(h, leaf_of_img, B, Nn, m, count, rng, idx_dtype):
    """`count` steps of (img_sel int64[m] rows of the feature pool, packed index block).  Positive (u, v): u a
    label; v one of the step's images w.p. 0.99 (u = its leaf label or one of that leaf's ancestors) else a
    child label (closure edge).  Negatives uniform over the step's mixed node set [labels ; images] minus the
    reference's excluded sets (oe.py:846-863: descendants of u when the child is corrupted, ancestors of v
    when the parent is corrupted).  Node ids: < n labels, >= n image slot (id - n) of the step."""
    from learning_embeddings_b200.engine import pack_index_block
    n = h.n
    edges = h.closure_edges()
    out = []
    for _ in range(count):
        sel = rng.choice(len(leaf_of_img), size=m, replace=False)
        leaf = leaf_of_img[sel]                       # leaf label of every image slot
        is_img = rng.random(B) < 0.99
        slot = rng.integers(0, m, size=B)
        up = rng.integers(0, 4, size=B)               # how many levels above the leaf the parent sits
        u = leaf[slot].copy()
        for _k in range(3):
            step_up = (up > _k) & (h.parents[u] >= 0)
            u[step_up] = h.parents[u[step_up]]
        e = edges[rng.integers(0, len(edges), size=B)]
        u = np.where(is_img, u, e[:, 0])
        v = np.where(is_img, n + slot, e[:, 1])
        v_lab = np.where(is_img, leaf[slot], e[:, 1])  # the label whose ancestors are v's ancestors
        uu, vv, vl = (np.repeat(a[:, None], Nn, 1) for a in (u, v, v_lab))
        vimg = np.repeat(is_img[:, None], Nn, 1)

        def lab_of(x):                                 # label a node hangs under (itself for a label)
            return np.where(x >= n, leaf[np.clip(x - n, 0, m - 1)], x)

        neg_to = rng.integers(0, n + m, size=(B, Nn))
        while True:                                    # corrupted child: not u, not below u
            cl = lab_of(neg_to)
            bad = (neg_to == uu) | h.is_descendant(uu, cl) | ((neg_to >= n) & (cl == uu))
            k = int(bad.sum())
            if k == 0:
                break
            neg_to[bad] = rng.integers(0, n + m, size=k)
        neg_from = rng.integers(0, n + m, size=(B, Nn))
        while True:                                    # corrupted parent: not v, not an ancestor of v
            lab = neg_from < n
            bad = (neg_from == vv) | (lab & (h.is_descendant(np.where(lab, neg_from, 0), vl) | (vimg & (neg_from == vl))))
            k = int(bad.sum())
            if k == 0:
                break
            neg_from[bad] = rng.integers(0, n + m, size=k)
        blk = pack_index_block(u, v, neg_to, neg_from, dtype=idx_dtype, n_rows=n + m)
        sel_t = torch.from_numpy(sel.astype(np.int64))
        out.append((sel_t.pin_memory() if torch.cuda.is_available() else sel_t, blk))
    return out


def cfg2_cpu_runner(c, table, fw, fb, feats, sel, blk, B):
    """The same joint step on the host cores with the oracle's torch port (oe.py forward + autograd + Adam)."""
    from oracle import cones
    Nn = c["n_neg"]
    b = torch.from_numpy(blk[:B * (2 + 2 * Nn)].numpy().astype(np.int64))
    u, v = b[:B], b[B:2 * B]
    neg_to = b[2 * B:2 * B + B * Nn].view(B, Nn)
    neg_from = b[2 * B + B * Nn:].view(B, Nn)
    nf = torch.cat([u[:, None].expand(B, Nn), neg_from], 1).reshape(-1)
    nt = torch.cat([neg_to, v[:, None].expand(B, Nn)], 1).reshape(-1)
    W = table.clone().requires_grad_(True)
    w1 = fw.clone().requires_grad_(True)
    b1 = fb.clone().requires_grad_(True)
    opt = torch.optim.Adam([{"params": [W], "lr": c["lr_labels"]}, {"params": [w1, b1]}], lr=c["lr"])   # oe.py:1356-1357, :1714
    X = feats[sel]

    def run():
        opt.zero_grad()
        rows = torch.cat([cones.apply_rows(cones.ROW_EUC_SOFTCLIP, W, c["K"]),
                          cones.apply_rows(cones.ROW_EUC_SOFTCLIP, X @ w1.t() + b1, c["K"])], 0)
        E_pos = cones.energy(c["geom"], rows[u], rows[v], c["K"])
        E_neg = cones.energy(c["geom"], rows[nf], rows[nt], c["K"])
        loss = E_pos.sum() + (c["alpha"] - E_neg).clamp(min=0).sum()
        loss.backward()
        opt.step()
        return float(loss)

    return run


def cfg2_setup(ctx):
    c = CFG2
    from learning_embeddings_b200 import hierarchy as H
    from learning_embeddings_b200.engine import index_dtype_for
    h = H.ethec()
    idx_dt = index_dtype_for(h.n + c["m"])
    g = torch.Generator().manual_seed(0)
    table0 = torch.randn(h.n, c["D"], generator=g)
    torch.manual_seed(0)   # fc1's default init draws from the global generator: the same weights in every run
    lin = torch.nn.Linear(c["F"], c["D"])
    with torch.no_grad():
        fw0, fb0 = lin.weight.detach().clone(), lin.bias.detach().clone()
    rng = np.random.default_rng(7 + ctx.rank)
    leaves = np.arange(h.level_start[-1], h.level_stop[-1])
    leaf_of_img = leaves[rng.integers(0, len(leaves), size=c["pool"])]
    return c, h, idx_dt, g, table0, fw0, fb0, rng, leaf_of_img


def run_cfg2_reference(args, ctx):
    if ctx.rank != 0:
        return None
    c, h, idx_dt, g, table0, fw0, fb0, rng, leaf_of_img = cfg2_setup(ctx)
    Nn, B, m = c["n_neg"], c["B"], c["m"]
    pairs_per_step = B * (1 + 2 * Nn)
    torch.set_num_threads(os.cpu_count() or 1)
    pool_cpu = 4 * m  # a bounded feature pool for the host run
    feats = torch.relu(torch.randn(pool_cpu, c["F"], generator=g))
    sel, blk = make_joint_batches(h, leaf_of_img[:pool_cpu], B, Nn, m, 1, rng, idx_dt)[0]
    run = cfg2_cpu_runner(c, table0, fw0, fb0, feats, sel, blk, B)
    for _ in range(min(2, args.warmup)):
        run()
    ts = []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > 150.0:
            break
    v = pairs_per_step / float(np.mean(ts))
    cfg = {"workload": c["name"], "pairs_per_gpu_per_step": pairs_per_step, "positives_per_gpu_per_step": B,
           "images_per_gpu_per_step": m, "feature_dim": c["F"], "dim": c["D"], "negatives_per_edge": 2 * Nn,
           "table_rows": int(h.n), "parallelism": "host cores only"}
    return {"metric": METRIC, "value": v, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": len(ts),
            "warmup": min(2, args.warmup), "ms_per_step": float(np.mean(ts)) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                             "sample": "the full cfg2 step (%d pairs, %d images), %d timed steps" % (pairs_per_step, m, len(ts))},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def run_cfg2(args, ctx, steps, warmup, dump=None):
    from learning_embeddings_b200 import _native
    from learning_embeddings_b200.engine import JointConeStep
    c, h, idx_dt, g, table0, fw0, fb0, rng, leaf_of_img = cfg2_setup(ctx)
    Nn, D, B, m = c["n_neg"], c["D"], c["B"], c["m"]
    pairs_per_step = B * (1 + 2 * Nn)
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    idx_bytes = np.dtype(idx_dt).itemsize
    cfg = {"workload": c["name"], "pairs_per_gpu_per_step": pairs_per_step, "positives_per_gpu_per_step": B,
           "images_per_gpu_per_step": m, "feature_dim": c["F"], "dim": D, "negatives_per_edge": 2 * Nn,
           "table_rows": int(h.n), "update": "adam on table (lr 0.1) + fc1 (lr 1e-3), inside the fused update kernels",
           "scalar_core": "fp32", "index_dtype": np.dtype(idx_dt).name, "feature_pool_images": c["pool"],
           "parallelism": "dp%d (pairs and images sharded, table + fc1 replicated)" % world}
    gd = torch.Generator(device=dev).manual_seed(1 + rank)
    feats = torch.relu(torch.randn(c["pool"], c["F"], generator=gd, device=dev))   # 537 MB, staged once
    rotation = args.rotation or 8
    batches = make_joint_batches(h, leaf_of_img, B, Nn, m, rotation, rng, idx_dt)
    dev_batches = [(s_.to(dev), b_.to(dev)) for s_, b_ in batches]
    cfg["l2_policy"] = "every step gathers %d of %d feature rows (%.0f MB read twice, > 126 MB L2); %d index batches rotate" % (
        m, c["pool"], m * c["F"] * 4 / 1e6, rotation)
    if ctx.world > 1:
        cfg["start_alignment"] = "device-side rendezvous (one-element all-reduce) enqueued right before the start event"
    cfg["launch_queue"] = "a ~0.5 ms spin kernel precedes the start event, so the timed launches are queued before the GPU reaches them"
    cfg["warmup_steps"] = "max(--warmup, 40) steps + one untimed rehearsal of the timed loop"
    table, fw, fb = table0.to(dev).clone(), fw0.to(dev).clone(), fb0.to(dev).clone()
    eng = JointConeStep(table, fw, fb, feats, c["geom"], Nn, B, m, K=c["K"], alpha=c["alpha"], lr=c["lr_labels"],
                        lr_fc=c["lr"], precision=0, process_group=ctx.pg)
    cfg["exchange"] = ("packet all-reduce over peer memory inside the two update kernels (label table 35 KB, fc1 82 KB)"
                       if world > 1 else "none (1 GPU)")

    def dev_step(i):
        s_, b_ = dev_batches[i % rotation]
        eng.step_device(s_, *eng._split(b_, B))

    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    ctx.warm(dev_step, eng, kev, warmup)
    restart = None
    if args.dump_outputs:
        restart = restarter(eng, [(table, table0.to(dev)), (eng.fc_w, fw0.to(dev)), (eng.fc_b, fb0.to(dev))],
                            list(eng.opt.values()) + list(eng.opt_fc.values()))
        cfg["dump_outputs"] = "the last timed step starts from the seeded initial table and fc1"
    launches0 = _native.launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active.set()
    ctx.align_streams()
    ctx.sync_all()
    ctx.align_streams()
    ctx.prequeue()
    t0.record()
    for i in range(steps):
        eng.kernel_events = kev[i] if i % 4 == 0 else None
        if restart is not None and i == steps - 1:
            restart()
        dev_step(i)
    t1.record()
    ctx.sync_all()
    sampler.active.clear()
    eng.kernel_events = None
    lec_launches = _native.launch_count() - launches0
    elapsed_ms = ctx.max_ranks(t0.elapsed_time(t1))
    kernel_ms = float(np.mean([a.elapsed_time(b) for i, (a, b) in enumerate(kev) if i % 4 == 0]))
    value = world * pairs_per_step * steps / (elapsed_ms * 1e-3)
    clocks = sampler.summary()
    if dump is not None:
        dump.update(snapshot({"loss": eng.loss_global, "table": table, "fc_weight": eng.fc_w, "fc_bias": eng.fc_b,
                              "E_pos": eng.E_pos[:B], "E_neg": eng.E_neg[:B]}))
    e2e = None
    if not args.no_e2e:
        for i in range(3):
            eng.step_host(*batches[i % rotation], B)
        ctx.sync_all()
        sampler.active.set()
        w0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            eng.step_host(*batches[i % rotation], B)
        e1.record()
        ctx.sync_all()
        sampler.active.clear()
        e_ms = ctx.max_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3))
        e2e = {"value": world * pairs_per_step * steps / (e_ms * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": B * (2 + 2 * Nn) * idx_bytes + m * 8, "d2h_bytes_per_step": 8,
               "ms_per_step": e_ms / steps,
               "api": "JointConeStep.step_host (features device-resident; per step: image selection + index block in, loss out)"}
    sampler.stop()
    final_loss = float(eng.loss.item())
    if world > 1:
        eng.check_exchange()
    if rank != 0:
        return None
    peak, peak_src = hbm_peak()
    bytes_per_pair = 24 + 16 * D
    achieved = pairs_per_step * bytes_per_pair / (kernel_ms * 1e-3) / 1e9
    step_ms = elapsed_ms / steps
    x_bytes = m * c["F"] * 4
    roofline = {"bound": "hbm", "kernel": "pairs_grouped_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_pair": bytes_per_pair,
                "kernel_ms": kernel_ms, "kernel_share_of_step": kernel_ms / step_ms,
                "step_algorithmic_bytes": 2 * x_bytes + pairs_per_step * bytes_per_pair,
                "step_floor_ms": 2 * x_bytes / (peak * 1e9) * 1e3,
                "step_hbm_frac": 2 * x_bytes / (peak * 1e9) * 1e3 / step_ms,
                "note": "the step is bound by the two passes over the %d x %d fp32 gathered feature rows (lec_featnet_fwd, "
                        "lec_featnet_wgrad: %.0f MB each); step_floor_ms = those bytes at the measured HBM peak, "
                        "step_hbm_frac = floor / measured step" % (m, c["F"], x_bytes / 1e6)}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        run = cfg2_cpu_runner(c, table0, fw0, fb0, feats[:4 * m].cpu(), torch.from_numpy(np.arange(m)), batches[0][1], B)
        run()
        ts = []
        t_all = time.perf_counter()
        while len(ts) < 20 and time.perf_counter() - t_all < 8.0:
            t0_ = time.perf_counter()
            run()
            ts.append(time.perf_counter() - t0_)
        cpu = {"value": pairs_per_step / float(np.mean(ts)), "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
               "sample": "the full cfg2 step (%d pairs, %d images) x %d, torch fp32 on all host threads" % (pairs_per_step, m, len(ts))}
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": max(3, warmup), "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks,
            "e2e": e2e, "gpu_launches": int(lec_launches), "roofline": roofline, "cpu_baseline": cpu,
            "final_loss": final_loss}


# ------------------------------------------------------------------------------------------------
# cfg3: all-pairs image x label scoring (BASELINE.json metric "image x label scores/s")
# ------------------------------------------------------------------------------------------------
def cfg3_inputs(n_img, D, seed):
    """SURVEY 8(d) cfg3: images uniform direction with |y| ~ U[0.30, 0.95]; ETHEC labels, norm by level
    U[0.10 + 0.2 l, 0.30 + 0.2 l]."""
    from learning_embeddings_b200 import hierarchy as H
    h = H.ethec()
    g = torch.Generator().manual_seed(seed)

    def ball(n, lo, hi):
        d = torch.randn(n, D, generator=g)
        return d / d.norm(dim=1, keepdim=True) * (lo + (hi - lo) * torch.rand(n, 1, generator=g))
    labels = torch.zeros(h.n, D)
    for l in range(len(h.level_start)):
        s, e = h.level_start[l], h.level_stop[l]
        labels[s:e] = ball(e - s, 0.10 + 0.2 * l, 0.30 + 0.2 * l)
    return h, labels, ball(n_img, 0.30, 0.95)


def cfg3_cpu(h, labels, images, K, steps, warmup, budget_s):
    """The reference's scoring (oe_h.py:2018-2036: E(label, image) for every pair, per-level topk(5, smallest)) as
    restated by the oracle, on all host threads, over a bounded sample of the images."""
    from oracle import cones
    torch.set_num_threads(os.cpu_count() or 1)

    def run():
        E = cones.score_matrix("hyp", labels, images, K)
        return cones.topk_per_level(E, h.level_start, h.level_stop, 5)
    for _ in range(min(1, warmup)):
        run()
    ts = []
    t_all = time.perf_counter()
    while len(ts) < steps and (not ts or time.perf_counter() - t_all < budget_s):
        t0 = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t0)
    return images.shape[0] * labels.shape[0] / float(np.mean(ts)), float(np.mean(ts)), len(ts)


def run_cfg3_reference(args, ctx):
    if ctx.rank != 0:
        return None
    D, K = args.dim, 0.1
    sample = min(args.images, 32768)
    h, labels, images = cfg3_inputs(sample, D, seed=0)
    v, mean_s, n_done = cfg3_cpu(h, labels, images, K, args.steps, args.warmup, budget_s=150.0)
    cfg = {"workload": "cfg3: hyperbolic cone inference scoring, %d synthetic image embeddings x 723 ETHEC labels, D=%d, "
                       "per-level top-5 + full energy matrix" % (sample, D),
           "images_per_gpu_per_step": sample, "labels": 723, "dim": D, "levels": 4, "topk": 5, "parallelism": "host cores only"}
    cores = os.cpu_count() or 1
    return {"metric": "image x label scores/s", "value": v, "unit": "scores/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": n_done, "warmup": min(1, args.warmup), "ms_per_step": mean_s * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "scores/s", "cores": cores, "kind": "port",
                             "sample": "%d images x 723 labels per step (energy matrix + per-level top-5), %d timed steps, torch "
                                       "fp32 on all host threads" % (sample, n_done)},
            "e2e": {"value": v, "unit": "scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def run_cfg3(args, ctx, steps, warmup, dim=None, modes=None, with_e2e=True, with_cpu=True, dump=None):
    """Returns one record per score mode in `modes` (default: the one --score-mode names), sharing inputs."""
    import ctypes
    from learning_embeddings_b200 import _native, ops
    metric, unit = "image x label scores/s", "scores/s"
    D, n_img, K, k = (dim or args.dim), args.images, 0.1, 5
    modes = modes or [args.score_mode]
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    h, labels, images0 = cfg3_inputs(n_img, D, seed=rank)
    L = labels.shape[0]
    labels_d = labels.to(dev)
    # rotate through image sets so that no step finds its inputs in L2; a matrix-writing step also streams 2.9 GB out
    rotation = args.rotation or max(2, int(np.ceil(160e6 / (n_img * D * 4))))
    host_sets = [images0.pin_memory()]
    for r in range(1, rotation):
        host_sets.append(images0.roll(shifts=r * 977, dims=0).contiguous().pin_memory())
    dev_sets = [x.to(dev) for x in host_sets]
    nl = len(h.level_start)
    lib = _native.lib()
    ls = (ctypes.c_int32 * nl)(*h.level_start)
    le = (ctypes.c_int32 * nl)(*h.level_stop)
    tc_ok = bool(lib.lec_score_tc_supported(ops.GEOM["hyp"], 0, D, L, nl))
    if args.engine == "tc" and not tc_ok:
        raise SystemExit("tensor-core scoring does not support this case")
    use_tc = tc_ok and args.engine in ("tc", "auto")   # "auto" = what ops.score_topk picks
    ws, nb = None, 0
    if use_tc:
        nb = int(lib.lec_score_workspace_bytes(L, D, nl))
        ws = ops._score_workspace(dev, nb)
    peak, peak_src = hbm_peak()
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    records = {}
    idx_buf = torch.empty((n_img, nl, k), device=dev, dtype=torch.int32)
    val_buf = torch.empty((n_img, nl, k), device=dev, dtype=torch.float32)
    scores_buf = None
    for mode in modes:
        want_matrix, want_topk = mode in ("both", "matrix"), mode in ("both", "topk")
        cfg = {"workload": "cfg3: hyperbolic cone inference scoring, %d synthetic image embeddings x 723 ETHEC labels per GPU, D=%d, "
                           "per-level top-5%s" % (n_img, D, " + full [L, N] fp32 energy matrix" if want_matrix else ""),
               "images_per_gpu_per_step": n_img, "labels": 723, "dim": D, "levels": 4, "topk": k, "writes": mode,
               "parallelism": "dp%d (images sharded by contiguous ranges, labels replicated, no collective)" % world,
               "l2_policy": "inputs rotate through %d image sets (%.0f MB > 126 MB L2)%s" % (
                   rotation, rotation * n_img * D * 4 / 1e6,
                   "; every step also writes the %.2f GB matrix" % (L * n_img * 4 / 1e9) if want_matrix else ""),
               "engine": "tc (tcgen05 kind::tf32 3xTF32 + fused epilogue)" if use_tc else "simt (packed FFMA2 tile kernel)"}
        idx = idx_buf if want_topk else None
        val = val_buf if want_topk else None
        if want_matrix and scores_buf is None:
            scores_buf = torch.empty((L, n_img), device=dev, dtype=torch.float32)
        scores = scores_buf if want_matrix else None

        def score(imgs):
            n = imgs.shape[0]
            if use_tc:
                _native.check(lib.lec_score_topk_tc(ops.GEOM["hyp"], 0, _native._p(labels_d), L, _native._p(imgs), n, D, K,
                                                    ctypes.cast(ls, ctypes.c_void_p), ctypes.cast(le, ctypes.c_void_p), nl, k,
                                                    _native._p(scores), _native._p(idx), _native._p(val), _native._p(ws), nb,
                                                    _native.stream_ptr(dev)), "lec_score_topk_tc")
            else:
                _native.check(lib.lec_score_topk_ex(ops.GEOM["hyp"], 0, _native._p(labels_d), L, _native._p(imgs), n, D, K,
                                                    ctypes.cast(ls, ctypes.c_void_p), ctypes.cast(le, ctypes.c_void_p), nl, k,
                                                    _native._p(scores), 1, _native._p(idx), _native._p(val),
                                                    _native.stream_ptr(dev)), "lec_score_topk_ex")

        W = max(3, warmup)
        for i in range(W):
            score(dev_sets[i % rotation])
        ctx.sync_all()
        launches0 = _native.launch_count()
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.reset()
        sampler.active.set()
        ctx.sync_all()
        t0.record()
        for i in range(steps):
            kev[i][0].record()
            score(dev_sets[i % rotation])
            kev[i][1].record()
        t1.record()
        ctx.sync_all()
        sampler.active.clear()
        lec_launches = _native.launch_count() - launches0
        elapsed_ms = ctx.max_ranks(t0.elapsed_time(t1))
        kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
        value = world * n_img * L * steps / (elapsed_ms * 1e-3)
        clocks = sampler.summary()
        if dump is not None:
            got = {"topk_index": idx, "topk_energy": val, "energy": scores}
            dump.update(snapshot({name: t for name, t in got.items() if t is not None}))

        # end to end: pinned host images -> H2D -> per-level top-5 -> predictions D2H, through ops.ScorePipeline, which
        # cuts the image set into slices and overlaps the copies of neighbouring slices with the kernel (what the
        # reference's caller consumes is the top-5 per level, oe_h.py:2030-2036; the matrix never leaves the device)
        e2e = None
        if with_e2e and not args.no_e2e and want_topk:
            out_idx = torch.empty((n_img, nl, k), dtype=torch.int16).pin_memory()   # 723 label ids fit int16
            pipe = ops.ScorePipeline(labels_d, "hyp", K, h.level_start, h.level_stop, k=k, slice_images=131072,
                                     engine=("tc" if args.engine == "tc" else "auto"))
            for i in range(2):
                pipe.run(host_sets[i % rotation], out_idx)
            ctx.sync_all()
            sampler.active.set()
            w0 = time.perf_counter()
            n_e2e = max(3, min(steps, 20))
            for i in range(n_e2e):
                pipe.run(host_sets[i % rotation], out_idx)   # returns with the predictions in host memory
            e_ms = ctx.max_ranks((time.perf_counter() - w0) * 1e3)
            sampler.active.clear()
            e2e = {"value": world * n_img * L * n_e2e / (e_ms * 1e-3), "unit": unit, "h2d_bytes_per_step": n_img * D * 4,
                   "d2h_bytes_per_step": n_img * nl * k * 2, "ms_per_step": e_ms / n_e2e, "steps": n_e2e,
                   "api": "ops.ScorePipeline.run (host images in, host top-5 label ids per level out as int16; 128K-image slices, "
                          "copies overlap the kernel)"}
            assert int(out_idx.min()) >= -1 and int(out_idx.max()) < L
            del pipe, out_idx
        if rank != 0:
            continue
        # SURVEY 8(d): a matrix-writing step moves 4 B per score + the image rows once (+ 160 B of top-k per image);
        # a top-k-only step moves (4 D + 160) / L per score
        bytes_per_score = ((4.0 if want_matrix else 0.0) + 4.0 * D / L + (160.0 / L if want_topk else 0.0))
        achieved = n_img * L * bytes_per_score / (kernel_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic_cfg3.json")
        if use_tc and os.path.exists(tpath):
            per_score = json.load(open(tpath)).get("dram_bytes_per_score", {}).get("d%d_%s" % (D, mode))
            if per_score is not None:
                traffic = per_score * n_img * L
        roofline = {"bound": "hbm", "kernel": "score_mma_kernel" if use_tc else "score_fast_kernel", "achieved": achieved,
                    "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_score": bytes_per_score, "kernel_ms": kernel_ms,
                    "kernel_share_of_step": kernel_ms / (elapsed_ms / steps),
                    "note": "kernel_ms brackets the whole library call (label repack launch + scoring kernel)"
                            + ("" if want_matrix else "; a top-k-only step is bound by FP32/MUFU issue, not HBM")}
        cpu = None
        if with_cpu and world == 1 and not args.no_cpu_baseline:
            sample = min(n_img, 32768)
            v, mean_s, n_done = cfg3_cpu(h, labels, images0[:sample], K, steps=8, warmup=1, budget_s=8.0)
            cpu = {"value": v, "unit": unit, "cores": os.cpu_count() or 1, "kind": "port",
                   "sample": "%d images x 723 labels per step (energy matrix + per-level top-5), %d steps, torch fp32 on all "
                             "host threads" % (sample, n_done)}
            with_cpu = False   # once per dimension
        records[mode] = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": steps, "warmup": W,
                         "ms_per_step": elapsed_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                         "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e,
                         "gpu_launches": int(lec_launches), "roofline": roofline, "cpu_baseline": cpu}
    sampler.stop()
    del dev_sets, host_sets, scores_buf, idx_buf, val_buf
    torch.cuda.empty_cache()
    return records if rank == 0 else None


# ------------------------------------------------------------------------------------------------
def guarded(name, fn, ctx):
    """A failing side workload must not cost the headline line: report the error under its name."""
    try:
        return fn()
    except Exception as ex:  # noqa: BLE001
        if ctx.world > 1:
            raise   # ranks must stay in lock step: a one-sided failure would hang the others in a collective
        return {"error": "%s: %s" % (type(ex).__name__, str(ex)[:300])}


def main():
    args = parse()
    if args.impl == "reference":
        ctx = Ctx(need_gpu=False)
        wl = "cfg1" if args.workload == "all" else args.workload
        if wl == "cfg2":
            rec = run_cfg2_reference(args, ctx)
        elif wl == "cfg3":
            rec = run_cfg3_reference(args, ctx)
        else:
            rec = run_label_reference(args, ctx, wl)
        if rec is not None:
            print(json.dumps(rec))
        return
    ctx = Ctx(need_gpu=True)
    dump = {} if args.dump_outputs and ctx.rank == 0 else None   # outputs of the headline workload's timed path
    try:
        if args.workload in ("cfg0", "cfg1", "cfg4"):
            rec = run_label(args, ctx, args.workload, args.steps, args.warmup, headline=True, dump=dump)
        elif args.workload == "cfg2":
            rec = run_cfg2(args, ctx, args.steps, args.warmup, dump=dump)
        elif args.workload == "cfg3":
            recs = run_cfg3(args, ctx, args.steps, args.warmup, dump=dump)
            rec = recs[args.score_mode] if recs is not None else None
        else:
            rec = run_label(args, ctx, "cfg1", args.steps, args.warmup, headline=True, dump=dump)
            s_steps, s_warm = max(3, min(args.steps, 20)), max(3, min(args.warmup, 5))
            subs = {}
            sub_args = argparse.Namespace(**vars(args))
            sub_args.pairs, sub_args.rotation, sub_args.dump_outputs = 0, 0, None
            subs["cfg0"] = guarded("cfg0", lambda: run_label(sub_args, ctx, "cfg0", s_steps, s_warm), ctx)
            subs["cfg2"] = guarded("cfg2", lambda: run_cfg2(sub_args, ctx, s_steps, s_warm), ctx)
            for D, modes in ((10, ["matrix", "topk", "both"]), (50, ["matrix", "both"])):
                recs = guarded("cfg3", lambda: run_cfg3(sub_args, ctx, s_steps, s_warm, dim=D, modes=modes), ctx)
                if isinstance(recs, dict) and "error" not in recs:
                    for mode, r in recs.items():
                        subs["cfg3_d%d_%s" % (D, mode)] = r
                elif recs is not None:
                    subs["cfg3_d%d" % D] = recs
            subs["cfg4"] = guarded("cfg4", lambda: run_label(sub_args, ctx, "cfg4", s_steps, s_warm), ctx)
            if rec is not None:
                rec["workloads"] = subs
        if rec is not None:
            print(json.dumps(rec))
        if dump is not None:
            write_dump(args.dump_outputs, dump)
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
