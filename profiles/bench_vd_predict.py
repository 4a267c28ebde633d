"""MC posterior predictive of the variational-dropout network (the evaluation branch of run_epoch, VD:148-157) at
784-1200-1200-1200-10, test batch 1000, 100 samples: the eager loop (lbbnn.vd.predict_ensemble, one full forward per
sample) against lbbnn.vd.EnsemblePredictor with gemm="simt" and with gemm="tc".

    python profiles/bench_vd_predict.py [--reps R] [--out FILE]
    python -m torch.distributed.run --nproc-per-node W profiles/bench_vd_predict.py [--reps R] [--out FILE]

Every arm is warmed up first, then R timed repetitions alternate the three arms in the same process.  A repetition is one
whole predict_ensemble call over the 100 samples, timed with CUDA events; under torch.distributed.run the predictor arms run
this rank's shard plus the one all-reduce (the maximum over ranks counts), while the eager loop, which cannot be sharded,
runs all samples on every rank.  FLOPs are computed from the shapes: layer 1's two products (x theta, x^2 theta^2) once per
run, since its input is the same for every sample, every other layer's two products once per sample -- the same
algorithmic count for every arm.  Every line carries the card name, its power limit and the SM clock sampled during the
timed window; rank 0 prints the lines and appends them to --out."""
import argparse
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "profiles"), os.path.join(ROOT, "bayesian-neural-nets_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench import ClockSampler  # noqa: E402
from bench_ensemble import card  # noqa: E402

SIZES, B, S, SPL = (784, 1200, 1200, 1200, 10), 1000, 100, 10


def layer_flops():
    """algorithmic FLOPs of one run: 2 B in out per product, two products per layer"""
    return [2 * 2 * B * k * o * (1 if i == 0 else S) for i, (k, o) in enumerate(zip(SIZES[:-1], SIZES[1:]))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import lbbnn
    world, rank, pg = 1, 0, None
    if "LOCAL_RANK" in os.environ:
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
        pg, world, rank = dist.group.WORLD, dist.get_world_size(), dist.get_rank()
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    lbbnn.manual_seed(99)
    net = lbbnn.vd.BNN(SIZES).to(dev).eval()
    x = torch.randn(B, SIZES[0], device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    arms = {"eager": (lambda: lbbnn.vd.predict_ensemble(net, x, S), None)}
    for gemm in ("simt", "tc"):
        p = lbbnn.vd.EnsemblePredictor(net, batch=B, samples_per_launch=SPL, seed=5, gemm=gemm, process_group=pg)
        arms[gemm] = ((lambda p=p: p.predict_ensemble(x, S)), p)
    for f, _ in arms.values():                                  # warm-up: every arm before any timing
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(a.reps):
        for k, (f, _) in arms.items():                          # alternate the arms inside every repetition
            if pg is not None:
                dist.barrier(group=pg)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    t1 = time.perf_counter()
    sampler.stop()
    name, limit = card(torch.cuda.current_device())
    clocks = sampler.summary(t0, t1)
    fl = layer_flops()
    for k, ts in times.items():
        ms = torch.tensor(sorted(ts)[len(ts) // 2], device=dev)
        if pg is not None and k != "eager":
            dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=pg)
        ms = ms.item()
        p = arms[k][1]
        rec = {"workload": "vd_predict", "arm": k, "sizes": list(SIZES), "world": world if k != "eager" else 1, "batch": B,
               "samples": S, "samples_per_launch": SPL if p else 1, "reps": a.reps, "ms_per_run_median": ms,
               "ms_per_run_min": min(ts), "weight_samples_per_s": S / (ms * 1e-3), "tflops": sum(fl) / (ms * 1e-3) / 1e12,
               "layer_gflop_per_run": [f / 1e9 for f in fl], "tc_layers": p.tc if p else None,
               "kernels_per_launch": p.kernels_per_launch if p else None,
               "gpu": name, "power_limit": limit, "clocks": clocks}
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
