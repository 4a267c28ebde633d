"""Cost of the MNF simulation study (LBBNN-GP-MF-MNFsim_study.py: 20 -> 1 MNF layer, RNVP flows with hidden sizes [50] * 5,
Adam) on one GPU, one JSONL line:

  (a) lbbnn.mnf.SimStudyEnsemble: all R repetitions in one launch, CUDA events over a window of >= 1 s of 50-epoch launches
      that each restart from the state after a 2-epoch warm-up
  (b) the eager GPU loop of one repetition: SimStudyNetwork.loss + backward + torch.optim.Adam over the 12 groups, per step;
      the R-repetition figure is that step time times the study's steps, labelled as an extrapolation
  (c) the same loop on the host's CPU cores with the float32 oracle port (tests/mnf_sim_ref.mnfsim_loss on the oracle's
      mnf_forward), labelled "port"

    python profiles/bench_mnf_sim_study.py [--replicas 100] [--study-epochs 100] [--out FILE]

All arms run 2000 rows at batch 400 with one learning rate (1e-3) for every group: the study's own rates and stage
boundaries are not recorded in this project.  The card's name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "bayesian-neural-nets_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import cases as C  # noqa: E402
import lbbnn  # noqa: E402
import lbbnn_oracle as O  # noqa: E402
from mnf_sim_ref import mnfsim_loss  # noqa: E402

LR = 1e-3


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
    ap.add_argument("--replicas", type=int, default=100)
    ap.add_argument("--study-epochs", type=int, default=100)
    ap.add_argument("--cpu-steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mnf_sim_study needs a GPU")
    R = args.replicas
    case = C.sim_study_case(seed=0)
    X, y = case["X"].cuda(), case["y"].cuda()
    B, n = case["batch"], case["X"].shape[0]
    steps_per_epoch = n // B
    rec = {"bench": "mnf_sim_study", **gpu_info(), "replicas": R, "rows": n, "batch": B, "in_features": 20,
           "h_sizes": [50] * 5, "n_transforms": 2, "lr": LR, "steps_per_epoch": steps_per_epoch, "study_epochs": args.study_epochs}

    # (a) one launch for every repetition
    nets = []
    for i in range(R):
        torch.manual_seed(i)
        nets.append(lbbnn.mnf.SimStudyNetwork(num_batches=n / B).cuda())
    ens = lbbnn.mnf.SimStudyEnsemble(nets, X, y, batch_size=B, lrs=LR, seed=0)
    finite = lambda: int(torch.isfinite(ens.flat).all(1).sum())   # noqa: E731
    ens.run(2)
    torch.cuda.synchronize()
    rec["replicas_finite_after_warmup"] = finite()
    # every timed launch of EPOCHS epochs starts from the state after the warm-up (parameters, both Adam moments, step
    # counts: a 127 MB device copy per launch, inside the window), so the window times the same 50 epochs of every replica
    # instead of an ever longer run at one fixed rate
    epochs = 50
    state = [t.clone() for t in (ens.flat, ens.exp_avg, ens.exp_avg_sq, ens.step)]

    def launch():
        for dst, src in zip((ens.flat, ens.exp_avg, ens.exp_avg_sq, ens.step), state):
            dst.copy_(src)
        ens.run(epochs)

    per_launch, launches = timed(launch, 1.0)
    t_epoch = per_launch / epochs
    rec["replicas_finite_after_timing"] = finite()
    rec["epochs_trained"] = int(ens.step[0].item()) // steps_per_epoch
    rec["ensemble"] = {"epochs_per_launch": epochs, "launches": launches, "s_per_epoch": t_epoch,
                       "replica_steps_per_s": R * steps_per_epoch / t_epoch, "s_per_study": t_epoch * args.study_epochs}

    # (b) eager GPU loop of one repetition
    torch.manual_seed(0)
    net = lbbnn.mnf.SimStudyNetwork(num_batches=n / B).cuda()
    net.train()
    l1 = net.l1
    groups = [{"params": [getattr(l1, k)], "lr": LR} for k in lbbnn.mnf.SIM_LAYER_NAMES]
    groups += [{"params": list(l1.z_flow.parameters()), "lr": LR}, {"params": list(l1.r_flow.parameters()), "lr": LR}]
    opt = torch.optim.Adam(groups)
    state = {"k": 0}

    def eager_step():
        k = state["k"] % steps_per_epoch
        state["k"] += 1
        opt.zero_grad()
        loss = net.loss(X[k * B:(k + 1) * B], y[k * B:(k + 1) * B])[0]
        loss.backward()
        opt.step()

    for _ in range(20):
        eager_step()
    torch.cuda.synchronize()
    t_step, calls = timed(eager_step, 1.0)
    rec["eager_gpu_finite"] = all(bool(torch.isfinite(v).all()) for v in net.state_dict().values())
    rec["eager_gpu"] = {"s_per_step": t_step, "steps": calls, "replica_steps_per_s": 1.0 / t_step,
                        "s_per_study_extrapolated": t_step * steps_per_epoch * args.study_epochs * R}

    # (c) the float32 oracle port on the host's CPU cores, one repetition
    p = O.init_mnf_params(np.random.default_rng(0), 20, 1, 2, (50,) * 5)
    named = {k: v.clone().requires_grad_(True) for k, v in C.flat_named(p).items()}
    copt = torch.optim.Adam(list(named.values()), lr=LR)
    Xc, yc = case["X"], case["y"]
    pri = O.Priors(mu=0.1, sigma=1.3, alpha=0.3, bias_mu=0.0, bias_sigma=1.3)

    def masks(*shape):
        return [(torch.rand(*shape) < 0.5).float() for _ in range(2)]
    t0 = time.perf_counter()
    for s in range(args.cpu_steps):
        k = s % steps_per_epoch
        nz = {"eps_z": torch.randn(1, 20), "z_masks": masks(1, 20), "eps": torch.randn(B, 1), "eps_z2": torch.randn(1, 20),
              "z_masks2": masks(1, 20), "eps_r": torch.randn(1), "r_masks": masks(20)}
        copt.zero_grad()
        loss = mnfsim_loss(Xc[k * B:(k + 1) * B], yc[k * B:(k + 1) * B], C.unflatten_like(p, named), nz, n / B, pri)[0]
        loss.backward()
        copt.step()
    t_cpu = (time.perf_counter() - t0) / args.cpu_steps
    rec["cpu"] = {"impl": "port", "threads": torch.get_num_threads(), "cores": os.cpu_count(), "s_per_step": t_cpu,
                  "s_per_study_extrapolated": t_cpu * steps_per_epoch * args.study_epochs * R}
    rec["reference_cpu"] = "not measured"
    rec["speedup_vs_eager_gpu"] = rec["eager_gpu"]["s_per_study_extrapolated"] / rec["ensemble"]["s_per_study"]
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
