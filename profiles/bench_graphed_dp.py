"""Weak scaling of the data-parallel GraphedTrainer (MNF and MF networks, 784-400-600-10, 100 rows per rank).

    python -m torch.distributed.run --nproc-per-node W profiles/bench_graphed_dp.py [--steps K] [--warmup N] [--ref-ms MS]

Measured as bench.py's bench_module: a device-resident pool of synthetic batches, CUDA events around K replays of the
captured step, here the maximum over ranks.  mnf_mnist at lr 1e-3; mf_mnist with the reference's 33 parameter groups at
lr 1e-4.  Rank 0 prints one JSON line per workload; --ref-ms (JSON {workload: ms at world 1}) gives the efficiency."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "bayesian-neural-nets_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench import ClockSampler, make_pool  # noqa: E402

NUM_BATCHES, B, POOL = 600, 100, 256


def power_limit_w(index):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:  # noqa: BLE001
        return None


def run(kind, steps, warmup, pg, world, rank):
    import lbbnn
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    lbbnn.manual_seed(99)
    net = (lbbnn.mnf.BayesianNetwork() if kind == "mnf_mnist" else lbbnn.mf.BayesianNetwork()).to(dev)
    if kind == "mf_mnist":
        tr = lbbnn.GraphedTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-4, objective="elbo",
                                  param_groups=lbbnn.mf.reference_param_groups(net), process_group=pg)
    else:
        tr = lbbnn.GraphedTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-3, objective="kl", process_group=pg)
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
    import time
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
    mode = "single" if pg is None else tr.opt.dp["mode"]
    tr.graph = None
    return {"workload": kind, "world": world, "batch_per_rank": B, "steps": steps, "warmup": warmup,
            "ms_per_step": ms.item(), "samples_per_s": B * world / (ms.item() * 1e-3), "exchange": mode,
            "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(torch.cuda.current_device()),
            "clocks": sampler.summary(t0, t1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--ref-ms", default=None)
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    pg = None
    if "LOCAL_RANK" in os.environ:
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
        pg = dist.group.WORLD
    ref = json.loads(a.ref_ms) if a.ref_ms else {}
    for kind in ("mnf_mnist", "mf_mnist"):
        rec = run(kind, a.steps, a.warmup, pg, world, rank)
        rec["efficiency_vs_world1"] = (ref[kind] / rec["ms_per_step"]) if kind in ref else None
        if rank == 0:
            print(json.dumps(rec), flush=True)
    if pg is not None:
        dist.barrier(group=pg)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
