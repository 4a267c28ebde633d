"""Worker of tests/test_predict_dp_gpu.py: EnsemblePredictor(process_group=) against the single-process predictor.

    python -m torch.distributed.run --nproc-per-node W tests/ensemble_dp_worker.py

Each rank builds the same networks from the same seeds.  Rank 0 first runs the single-process predictor and then restores
the RNG state and flow-key counters it consumed, so that the sharded run draws the same native MNF z.  For every case the
sharded test_ensemble / outofsample must match the single-process run (sums within 1e-6, identical argmax) and be identical
on every rank.  Exits non-zero on a mismatch; rank 0 prints one line per case."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "bayesian-neural-nets_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import cases as C  # noqa: E402
import lbbnn  # noqa: E402

S, B, SPL = 12, 52, 5
KEYS = ("mean_prob", "entropy", "ensemble", "posterior_mean", "oos_entropy", "oos_pred")


def networks(kind):
    case = C.ensemble_case(seed=120 if kind == "lrt" else 121, batch=B, samples=S, kind=kind)
    if kind == "lrt":
        net = lbbnn.BayesianNetwork()
        with torch.no_grad():
            for l, p in zip(net.layers, case["layers"]):
                for k, v in p.items():
                    getattr(l, k).copy_(v)
    else:
        net = lbbnn.mnf.BayesianNetwork()
        for l, p in zip(net.layers, case["layers"]):
            l.load_state_dict(C.flat_named(p))
    return net.cuda().eval(), case


def evaluate(pred, case, inject_z):
    x = case["x"].cuda()
    eps = [e.cuda() for e in case["eps"]]
    z_noise = None
    if inject_z:
        z_noise = [{"eps_z": case["eps_z"][l][:, -1].cuda(), "z_masks": [m[:, -1].cuda() for m in case["z_masks"][l]]}
                   for l in range(3)]
    out = pred.test_ensemble(x, S, eps=eps, z_noise=z_noise)
    oos = pred.outofsample(x, S, eps=eps, z_noise=z_noise)
    out["oos_entropy"], out["oos_pred"] = oos["entropy"], oos["pred"]
    return {k: out[k] for k in KEYS}


def counters(net):
    return [m._calls for m in net.modules() if hasattr(m, "_calls")]


def set_counters(net, values):
    for m, v in zip([m for m in net.modules() if hasattr(m, "_calls")], values):
        m._calls = v


def main():
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    torch.manual_seed(3)
    lbbnn.manual_seed(99)
    failed = 0
    for name, kind, gemm, inject_z in (("lrt_simt", "lrt", "simt", False), ("lrt_tc", "lrt", "tc", False),
                                       ("mnf_injected_z", "mnf", "simt", True), ("mnf_native_z", "mnf", "tc", False)):
        net, case = networks(kind)
        ref = None
        if rank == 0:
            rng, calls = torch.cuda.get_rng_state(), counters(net)
            ref = evaluate(lbbnn.EnsemblePredictor(net, batch=B, samples_per_launch=SPL, seed=11, gemm=gemm), case, inject_z)
            torch.cuda.set_rng_state(rng)
            set_counters(net, calls)
        pred = lbbnn.EnsemblePredictor(net, batch=B, samples_per_launch=SPL, seed=11, gemm=gemm,
                                       process_group=dist.group.WORLD)
        got = evaluate(pred, case, inject_z)
        ok = True
        for k in KEYS:                        # identical on every rank
            allv = [torch.empty_like(got[k]) for _ in range(world)]
            dist.all_gather(allv, got[k])
            ok &= all(torch.equal(a, allv[0]) for a in allv)
        worst = 0.0
        if rank == 0:
            for k in KEYS:
                if got[k].dtype == torch.int64:
                    ok &= torch.equal(got[k], ref[k])
                else:
                    worst = max(worst, C.rel_err(got[k], ref[k]))
            ok &= worst < 1e-6
            print(f"{name}: world {world} rel err {worst:.2e} {'OK' if ok else 'MISMATCH'}, ranks agree", flush=True)
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.all_reduce(flag)
        failed += int(flag.item())
    dist.destroy_process_group()
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
