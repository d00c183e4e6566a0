"""Latency of the fused update kernel with and without the peer exchange, in isolation (no pair kernel in between).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29512 scripts/xchg_latency.py

Every rank calls lec_update_rows back to back on a zero gradient: with the exchange the ranks run in lock step (each
call waits for every peer's packets), so time per call = update + one exchange.  Compared with the same kernel without
exchange, and with an NCCL all_reduce of the same gradient in front of it.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from learning_embeddings_b200.engine import ConeStep  # noqa: E402


def timed(fn, n=2000, warm=50):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) / n * 1e3], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    for n, D, geom, upd in ((723, 10, "hyp", "rsgd"), (723, 2, "euc", "adam"), (1281, 16, "oe", "adam"), (8192, 10, "hyp", "rsgd"),
                            (82115, 50, "hyp", "rsgd")):
        w = torch.randn(n, D, generator=torch.Generator().manual_seed(0))
        W0 = (0.1 + 0.05 * torch.rand(n, 1)) * w / w.norm(dim=1, keepdim=True) if geom == "hyp" else w
        res = {}
        for comm in ("none", "p2p", "two_shot", "nccl"):
            from learning_embeddings_b200 import sharding
            mode = {"p2p": sharding.ONE_SHOT, "two_shot": sharding.TWO_SHOT}.get(comm)
            if comm == "p2p" and n * D * 4 > (4 << 20):
                res[comm] = float("nan")
                continue
            eng = ConeStep(W0.to(dev).clone(), geom, 5, 16, lr=1e-3, update=upd,
                           process_group=None if comm == "none" else dist.group.WORLD,
                           comm="auto" if comm == "none" else ("nccl" if comm == "nccl" else "p2p"), exchange_mode=mode)
            eng._rows_fwd()
            eng._rows_valid = True
            res[comm] = timed(eng.reduce_and_update)
            if comm in ("p2p", "two_shot"):
                eng.check_exchange()
        if rank == 0:
            print("world %d  table %5d x %2d %s/%s: update only %.2f us | one-shot packets %.2f us (+%.2f) | two-shot %.2f us | NCCL all_reduce + update %.2f us"
                  % (world, n, D, geom, upd, res["none"], res["p2p"], res["p2p"] - res["none"], res["two_shot"], res["nccl"]), flush=True)
    dist.barrier()
    dist.destroy_process_group()


main()
