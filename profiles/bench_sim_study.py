"""Cost of the simulation study (BASELINE.json configs[0], LBBNN-GP-MFsim_study.py:344-429) on one GPU, one JSONL line:

  (a) lbbnn.mf.SimStudyEnsemble: all R repetitions in one launch, CUDA events over a window of >= 1 s after a warm-up
  (b) the eager GPU loop of one repetition: SimStudyNetwork.sample_elbo + backward + the 11-group torch.optim.SGD, per step;
      the 100-repetition figure is that step time times the study's steps, labelled as an extrapolation
  (c) the same loop on the host's CPU cores with the float32 oracle port (oracle/lbbnn_oracle.mfsim_elbo), labelled "port"

    python profiles/bench_sim_study.py [--replicas 100] [--study-epochs 100] [--out FILE]

The card's name, power limit and SM clock are read in the same run.
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

import torch  # noqa: E402

import cases as C  # noqa: E402
import lbbnn  # noqa: E402
import lbbnn_oracle as O  # noqa: E402


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
    ap.add_argument("--cpu-steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sim_study needs a GPU")
    R = args.replicas
    case = C.sim_study_case(seed=0)
    X, y = case["X"].cuda(), case["y"].cuda()
    B, n = case["batch"], case["X"].shape[0]
    steps_per_epoch = n // B
    rec = {"bench": "sim_study", **gpu_info(), "replicas": R, "rows": n, "batch": B, "in_features": 20,
           "steps_per_epoch": steps_per_epoch, "study_epochs": args.study_epochs}

    # (a) one launch for every repetition
    nets = []
    for i in range(R):
        torch.manual_seed(i)
        nets.append(lbbnn.mf.SimStudyNetwork().cuda())
    ens = lbbnn.mf.SimStudyEnsemble(nets, X, y, batch_size=B, seed=0)
    ens.run(2)
    finite = lambda: int(torch.isfinite(ens.flat).all(1).sum())   # noqa: E731
    rec["replicas_finite_after_warmup"] = finite()
    # With native noise the study's SGD rates drive weight_b below zero after ~100-200 epochs on this data (the eager module
    # loop diverges the same way), and NaN parameters would short-cut the work: every launch of EPOCHS epochs starts from the
    # same parameters (one 27 KB copy per launch, inside the window), over as many launches as fill >= 1 s.
    epochs = 50
    snap = ens.flat.clone()

    def launch():
        ens.flat.copy_(snap)
        ens.run(epochs)

    per_launch, launches = timed(launch, 1.0)
    t_epoch = per_launch / epochs
    rec["replicas_finite_after_timing"] = finite()
    rec["ensemble"] = {"epochs_per_launch": epochs, "launches": launches, "s_per_epoch": t_epoch,
                       "replica_steps_per_s": R * steps_per_epoch / t_epoch,
                       "s_per_study": t_epoch * args.study_epochs}

    # (b) eager GPU loop of one repetition
    torch.manual_seed(0)
    net = lbbnn.mf.SimStudyNetwork().cuda()
    net.train()
    names = lbbnn.mf.SIM_PARAM_NAMES
    opt = torch.optim.SGD([{"params": [getattr(net.l1, k)], "lr": lbbnn.mf.SIM_STUDY_LRS[k]} for k in names], lr=0.01)
    state = {"k": 0}

    def eager_step():
        k = state["k"] % steps_per_epoch
        state["k"] += 1
        opt.zero_grad()
        loss = net.sample_elbo(X[k * B:(k + 1) * B], y[k * B:(k + 1) * B])[0]
        loss.backward()
        opt.step()

    snap_e = {k: v.clone() for k, v in net.state_dict().items()}

    def eager_step_fresh():
        # restart from the initial parameters every 50 epochs, as the ensemble arm does (NaN would reach binary_cross_entropy)
        if state["k"] % (50 * steps_per_epoch) == 0:
            net.load_state_dict(snap_e)
        eager_step()

    for _ in range(20):
        eager_step_fresh()
    torch.cuda.synchronize()
    t_step, calls = timed(eager_step_fresh, 1.0)
    assert all(bool(torch.isfinite(v).all()) for v in net.state_dict().values())
    rec["eager_gpu"] = {"s_per_step": t_step, "steps": calls, "replica_steps_per_s": 1.0 / t_step,
                        "s_per_study_extrapolated": t_step * steps_per_epoch * args.study_epochs * R}

    # (c) the float32 oracle port on the host's CPU cores, one repetition
    p = {k: v.clone().requires_grad_(True) for k, v in O.init_mf_params(__import__("numpy").random.default_rng(0), 20, 1,
                                                                         sim=True).items()}
    copt = torch.optim.SGD([{"params": [p[k]], "lr": lbbnn.mf.SIM_STUDY_LRS[k]} for k in names], lr=0.01)
    Xc, yc = case["X"], case["y"]
    t0 = time.perf_counter()
    for s in range(args.cpu_steps):
        k = s % steps_per_epoch
        nz = {"eps_w": torch.randn(1, 20), "eps_b": torch.randn(1),
              "g0_w": torch._standard_gamma(p["weight_a"].detach()), "g0_b": torch._standard_gamma(p["bias_a"].detach())}
        copt.zero_grad()
        loss = O.mfsim_elbo(Xc[k * B:(k + 1) * B], yc[k * B:(k + 1) * B], p, nz, torch.rand(1, 20), n / B)[0]
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
