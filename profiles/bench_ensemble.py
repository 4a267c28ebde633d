"""MC posterior predictive of the LRT network (lbbnn.EnsemblePredictor): CUDA-core (gemm="simt") against tensor-core
(gemm="tc") layers, at 784-64-64-10, 784-400-600-10, 1024-1024-1024-10 and 4096-4096-4096-10 with test batch 1000.

    python profiles/bench_ensemble.py [--reps R] [--out FILE]
    python -m torch.distributed.run --nproc-per-node W profiles/bench_ensemble.py [--reps R] [--out FILE]

Per shape and path: one predictor (samples_per_launch 10), every shape and path warmed up first, then R timed repetitions
that alternate simt and tc in the same process.  A repetition is one whole run() over the shape's sample count (under
torch.distributed.run: this rank's shard of it plus the one all-reduce of the accumulators), timed with CUDA events; the
maximum over ranks counts.  FLOPs are computed from the shapes: layer 1's two products once per run (its input is the same for
every sample), every other layer's two products once per sample.  The whole run's algorithmic TFLOP/s comes from those
timings.  A second, separate pass times the same work piece by piece, with CUDA events around the per-run prologue
(`_prepare_batch`: layer 1's products, and M, V of the tensor-core layers) and around every layer of every launch
(`_layer`), and reports algorithmic TFLOP/s per layer.  Every line carries the card name, its power limit and the SM clock
sampled during the timed windows; rank 0 prints the lines and appends them to --out."""
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

from bench import ClockSampler  # noqa: E402

B, SPL = 1000, 10
# sizes, MC samples per run(): below, at and above the 1024 width of gemm="auto"
SHAPES = {"lrt_narrow": ((784, 64, 64, 10), 400), "lrt_mnist": ((784, 400, 600, 10), 200),
          "lrt_1024": ((1024, 1024, 1024, 10), 100), "lrt_wide": ((4096, 4096, 4096, 10), 40)}


def card(index):
    """(name, power limit) as nvidia-smi reports them"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(index), None


def layer_flops(sizes, samples):
    """algorithmic FLOPs of one run(): 2 B in out per product, two products (E and S) per layer"""
    out = []
    for i, (k, o) in enumerate(zip(sizes[:-1], sizes[1:])):
        out.append(2 * 2 * B * k * o * (1 if i == 0 else samples))
    return out


def per_layer(p, sizes, count, first, reps):
    """median ms per run of the per-run prologue and of each layer (summed over the launches of one run), events around each"""
    import lbbnn._capi as K
    st = K.current_stream()
    pro, lay = [], [[] for _ in p.layers]
    for _ in range(reps):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        p._prepare_batch(st)
        e[1].record()
        marks = []
        s = first
        while s < first + count:
            n = min(p.SB, first + count - s)
            h = None
            for li in range(len(p.layers)):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                h, _ = p._layer(li, s, s - first, n, None, h, st)
                b.record()
                marks.append((li, a, b))
            s += n
        torch.cuda.synchronize()
        pro.append(e[0].elapsed_time(e[1]))
        per = [0.0] * len(p.layers)
        for li, a, b in marks:
            per[li] += a.elapsed_time(b)
        for li, v in enumerate(per):
            lay[li].append(v)
    med = lambda v: sorted(v)[len(v) // 2]
    k0, o0 = sizes[0], sizes[1]
    pro_fl = 2 * 2 * B * k0 * o0
    out = {"prologue": {"ms_per_run": med(pro), "gflop_per_run": pro_fl / 1e9, "tflops": pro_fl / (med(pro) * 1e-3) / 1e12}}
    layers = []
    for li, (k, o) in enumerate(zip(sizes[:-1], sizes[1:])):
        fl = 0 if li == 0 else 2 * 2 * B * k * o * count     # layer 1's products are in the prologue
        ms = med(lay[li])
        layers.append({"layer": li + 1, "in": k, "out": o, "tensor_cores": p.tc[li], "ms_per_run": ms, "gflop_per_run": fl / 1e9,
                       "tflops": fl / (ms * 1e-3) / 1e12 if fl else None})
    out["layers"] = layers
    return out


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
    runs = {}
    for shape, (sizes, S) in SHAPES.items():
        net = lbbnn.BayesianNetwork(sizes).to(dev).eval()
        with torch.no_grad():
            for l in net.layers:
                l.weight_mu.mul_(784.0 / l.in_features)
        x = torch.rand(B, sizes[0], device=dev, generator=torch.Generator(device=dev).manual_seed(1))
        for gemm in ("simt", "tc"):
            p = lbbnn.EnsemblePredictor(net, batch=B, samples_per_launch=SPL, seed=5, gemm=gemm, process_group=pg)
            first, count = p._shard(S)

            def call(p=p, x=x, first=first, count=count, S=S):
                p.run(x, count, first_sample=first, global_samples=S if pg is not None else None)
                p._sums()
            call()                                  # warm-up: every shape and path before any timing
            runs[(shape, gemm)] = (call, p, net)
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(a.reps):
        for key in runs:                            # alternate the paths inside every repetition
            if pg is not None:
                dist.barrier(group=pg)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            runs[key][0]()
            e1.record()
            torch.cuda.synchronize()
            times[key].append(e0.elapsed_time(e1))
    t1 = time.perf_counter()
    sampler.stop()
    name, limit = card(torch.cuda.current_device())
    clocks = sampler.summary(t0, t1)
    pieces = {}
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    t2 = time.perf_counter()
    for (shape, gemm), (_, p, _) in runs.items():
        sizes, S = SHAPES[shape]
        first, count = p._shard(S)
        pieces[(shape, gemm)] = per_layer(p, sizes, count, first, a.reps)
    t3 = time.perf_counter()
    sampler.stop()
    piece_clocks = sampler.summary(t2, t3)
    for (shape, gemm), ts in times.items():
        sizes, S = SHAPES[shape]
        ms = torch.tensor(sorted(ts)[len(ts) // 2], device=dev)
        if pg is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=pg)
        ms = ms.item()
        fl = layer_flops(sizes, S)
        p = runs[(shape, gemm)][1]
        rec = {"workload": "ensemble_" + shape, "gemm": gemm, "world": world, "batch": B, "samples": S,
               "samples_per_launch": SPL, "reps": a.reps, "ms_per_run_median": ms, "ms_per_run_min": min(ts),
               "weight_samples_per_s": S / (ms * 1e-3), "tflops": sum(fl) / (ms * 1e-3) / 1e12,
               "layer_gflop_per_run": [f / 1e9 for f in fl], "tc_layers": p.tc, "kernels_per_launch": p.kernels_per_launch,
               "per_layer_pass": dict(pieces[(shape, gemm)], rank=rank, clocks=piece_clocks),
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
