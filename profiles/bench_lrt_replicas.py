"""Cost of training R LRT networks (784-400-600-10, batch 100, Adam: the reference driver's seed loop, LBBNN-GP-MF-LRT.py:354-372)
on one GPU, one JSONL line per R:

  (a) lbbnn.LRTReplicaTrainer: all R networks in one launch of the persistent step kernel per step (graph replays);
  (b) lbbnn.LRTTrainer: one network per launch, R launches back to back (graph replays), i.e. the seeds one after another.

Both are timed by CUDA events over windows of at least 1 s after a warm-up, on the same device-resident minibatches
(per-replica batches for (a)).  `hbm_floor_us` is a bound, not a measurement: per replica the step reads and writes the
parameters, both Adam moments and the gradients once (4 x P floats read + 4 x P written, P = 1.68 M) plus the input batch,
over the data-sheet 7.7 TB/s.  The card's name, power limit and SM clock are read in the same run.

    python profiles/bench_lrt_replicas.py [--replicas 1,2,4,8,10,16,32] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "bayesian-neural-nets_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import torch  # noqa: E402

import lbbnn  # noqa: E402

SIZES, BATCH = (784, 400, 600, 10), 100
HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = (s.strip() for s in q[torch.cuda.current_device()].split(","))
    return {"gpu": name, "power_limit": power, "sm_clock": clock}


def timed(fn, min_s=1.0):
    """(seconds per call, calls) of fn() over a window of at least min_s, by CUDA events."""
    calls = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        s = a.elapsed_time(b) / 1e3
        if s >= min_s:
            return s / calls, calls
        calls = max(calls * 2, int(calls * 1.2 * min_s / max(s, 1e-6)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicas", default="1,2,4,8,10,16,32")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    g = torch.Generator().manual_seed(0)
    lines = []
    for R in [int(v) for v in args.replicas.split(",")]:
        nets = []
        for r in range(R):
            torch.manual_seed(r)                     # the driver's torch.manual_seed(i) per seed
            nets.append(lbbnn.BayesianNetwork(SIZES).cuda())
        singles = []
        for r in range(R):
            torch.manual_seed(r)
            net = lbbnn.BayesianNetwork(SIZES).cuda()
            singles.append(lbbnn.LRTTrainer(net, batch_size=BATCH, num_batches=600, seed=r))
        tr = lbbnn.LRTReplicaTrainer(nets, batch_size=BATCH, num_batches=600, seeds=list(range(R)))
        x = torch.rand(R, BATCH, SIZES[0], generator=g)
        y = torch.randint(0, SIZES[-1], (R, BATCH), generator=g)
        tr.x.copy_(x)
        tr.y.copy_(y)
        for r, s in enumerate(singles):
            s.x.copy_(x[r])
            s.y.copy_(y[r])
        for _ in range(20):                          # warm-up
            tr.step_device()
            for s in singles:
                s.step_device()
        torch.cuda.synchronize()
        t_rep, n_rep = timed(tr.step_device)

        def seq():
            for s in singles:
                s.step_device()
        t_seq, n_seq = timed(seq)
        P = tr.n_flat
        floor = R * (8 * P * 4 + BATCH * SIZES[0] * 4) / HBM_BYTES_PER_S
        line = dict(info, workload="lrt_replicas", sizes=list(SIZES), batch=BATCH, replicas=R, schedule=tr.schedule,
                    replica_step_us=round(t_rep * 1e6, 2), replica_calls=n_rep,
                    sequential_step_us=round(t_seq * 1e6, 2), sequential_calls=n_seq,
                    speedup=round(t_seq / t_rep, 3), us_per_network_step=round(t_rep * 1e6 / R, 2),
                    hbm_floor_us=round(floor * 1e6, 2), share_of_hbm_floor=round(floor / t_rep, 3))
        print(json.dumps(line), flush=True)
        lines.append(line)
        del tr, singles, nets
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
