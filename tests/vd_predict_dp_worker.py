"""Worker of tests/test_vd_predict_dp_gpu.py: lbbnn.vd.EnsemblePredictor(process_group=) against the single-process predictor.

    python -m torch.distributed.run --nproc-per-node W tests/vd_predict_dp_worker.py

Each rank builds the same network from the same seeded case.  Rank 0 first runs the single-process predictor.  For every case
(injected and native zeta, CUDA-core and tensor-core GEMMs) the sharded predict_ensemble and result() must match the
single-process run (within 1e-6, identical argmax) and be identical on every rank.  Exits non-zero on a mismatch; rank 0
prints one line per case."""
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


def network():
    case = C.vd_net_case(seed=82, batch=B)
    net = lbbnn.vd.BNN()
    with torch.no_grad():
        for l, p in zip(net.layers, case["layers"]):
            l.theta.copy_(p["theta"])
            l.alpha.copy_(p["alpha"])
    return net.cuda(), case["x"].cuda()


def evaluate(pred, x, zetas):
    mean = pred.predict_ensemble(x, S, zetas=zetas)
    res = pred.result()
    return {"mean": mean, "mean_logp": res["mean_logp"], "pred": res["pred"]}


def main():
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    torch.manual_seed(3)
    lbbnn.manual_seed(99)
    failed = 0
    for name, gemm, inject in (("injected_simt", "simt", True), ("injected_tc", "tc", True), ("native_simt", "simt", False),
                               ("native_tc", "tc", False)):
        net, x = network()
        zetas = None
        if inject:
            g = torch.Generator(device="cuda").manual_seed(5)
            zetas = [torch.randn(S, B, l.m, device="cuda", generator=g) for l in net.layers]
        ref = None
        if rank == 0:
            ref = evaluate(lbbnn.vd.EnsemblePredictor(net, batch=B, samples_per_launch=SPL, seed=11, gemm=gemm), x, zetas)
        pred = lbbnn.vd.EnsemblePredictor(net, batch=B, samples_per_launch=SPL, seed=11, gemm=gemm,
                                          process_group=dist.group.WORLD)
        got = evaluate(pred, x, zetas)
        ok = True
        for k in got:                         # identical on every rank
            allv = [torch.empty_like(got[k]) for _ in range(world)]
            dist.all_gather(allv, got[k])
            ok &= all(torch.equal(a, allv[0]) for a in allv)
        worst = 0.0
        if rank == 0:
            ok &= torch.equal(got["pred"], ref["pred"]) and torch.equal(got["mean"].argmax(1), ref["mean"].argmax(1))
            worst = max(C.rel_err(got["mean_logp"], ref["mean_logp"]), C.rel_err(got["mean"], ref["mean"]))
            ok &= worst < 1e-6
            print(f"{name}: world {world} rel err {worst:.2e} {'OK' if ok else 'MISMATCH'}, ranks agree", flush=True)
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.all_reduce(flag)
        failed += int(flag.item())
    dist.destroy_process_group()
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
