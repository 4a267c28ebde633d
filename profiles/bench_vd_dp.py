"""Weak scaling of the data-parallel VDTrainer (variational_dropout.py, 784-1200-1200-1200-10, AdamW).

    python -m torch.distributed.run --nproc-per-node W profiles/bench_vd_dp.py [--steps K] [--warmup N] [--out FILE]

Measured as bench.py's bench_module: a device-resident pool of synthetic batches, CUDA events around K replays of the
captured step, the maximum over ranks.  For each batch per rank (the reference's 100 rows and 1000): the single-GPU
VDTrainer (no group) on every rank, then the data-parallel one over the launch's ranks.  Every line carries the card's name
and power limit (nvidia-smi, read-only) and which exchange ran; rank 0 prints the lines and appends them to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "bayesian-neural-nets_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench import ClockSampler, make_pool  # noqa: E402

NUM_BATCHES, POOL = 600.0, 64
BATCHES = (100, 1000)


def card(index):
    """(name, power limit) as nvidia-smi reports them"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(index), None


def run(B, steps, warmup, pg, world, rank):
    import lbbnn
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    lbbnn.manual_seed(99)
    net = lbbnn.vd.BNN().to(dev)
    tr = lbbnn.vd.VDTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-4, process_group=pg)
    px, py = make_pool(POOL, B, 784, 10, seed=1000 + rank)
    px, py = px.to(dev), py.to(dev)

    def step(i):
        tr.x.copy_(px[i % POOL], non_blocking=True)
        tr.y.copy_(py[i % POOL], non_blocking=True)
        tr.step_device()

    for i in range(warmup):
        step(i)
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    torch.cuda.synchronize()
    if pg is not None:
        dist.barrier(group=pg)
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if pg is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=pg)
    ranks = 1 if pg is None else world
    name, limit = card(torch.cuda.current_device())
    rec = {"workload": "vd_mnist", "world": ranks, "batch_per_rank": B, "steps": steps, "warmup": warmup,
           "ms_per_step": ms.item(), "samples_per_s": B * ranks / (ms.item() * 1e-3),
           "exchange": "single" if pg is None else tr.dp_update, "kernels_per_step": tr.kernels_per_step,
           "exchange_bytes_per_step": 4 * tr.n_flat, "gpu": name, "power_limit": limit,
           "clocks": sampler.summary(t0, t1)}
    tr.graph = None
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    pg = None
    if "LOCAL_RANK" in os.environ:
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
        pg = dist.group.WORLD
    for B in BATCHES:
        for group in ((None, pg) if pg is not None else (None,)):
            rec = run(B, a.steps, a.warmup, group, world, rank)
            if rank == 0:
                line = json.dumps(rec)
                print(line, flush=True)
                if a.out:
                    with open(a.out, "a") as fh:
                        fh.write(line + "\n")
    if pg is not None:
        dist.barrier(group=pg)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
