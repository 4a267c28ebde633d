"""Worker of tests/test_vd_dp_gpu.py: data-parallel VDTrainer against the single-GPU VDTrainer on the concatenated minibatch.

    python tests/vd_dp_worker.py single --world W --out DIR          one process, one GPU: the reference runs
    python -m torch.distributed.run --nproc-per-node W tests/vd_dp_worker.py dp --out DIR

Both phases build the same network with the same seeds.  Injected zeta: each rank feeds its slice of the reference's rows.
Native noise is compared with the reference at one rank only (rank 0 draws from the unshifted seed); at more ranks the
worker checks that the ranks' draws differ.  Exits non-zero on a mismatch; rank 0 prints one line per case."""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "bayesian-neural-nets_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import lbbnn  # noqa: E402

NB, ROWS, STEPS = 600.0, 100, 3
SIZES = (784, 1200, 1200, 1200, 10)          # variational_dropout.py:74-77
# eps well above the gradients' rounding level: the first AdamW steps are ~lr * sign(g), and the shards' partial sums reach
# an element whose gradient is ~0 in another order than the full batch's product does; the sign of such an element is noise
EPS = 1e-3


def cases(world):
    """(name, alpha_trainable, inject, LBBNN_DP_UPDATE)"""
    out = []
    for mode in (("sharded", "nccl") if world > 1 else ("auto", "nccl")):
        for alpha in (False, True):
            for inject in ((True,) if world > 1 else (True, False)):
                out.append((f"{'inject' if inject else 'native'}_alpha{int(alpha)}[{mode}]", alpha, inject, mode))
    return out


def build(alpha, inject, rows, pg, seed=1234):
    torch.manual_seed(7)
    lbbnn.manual_seed(seed)
    net = lbbnn.vd.BNN(SIZES, alpha_trainable=alpha).cuda()
    tr = lbbnn.vd.VDTrainer(net, batch_size=rows, num_batches=NB, lr=1e-4, eps=EPS, inject_noise=inject, process_group=pg)
    return net, tr


def data(step, n):
    g = torch.Generator().manual_seed(50 + step)
    x, y = torch.randn(n, SIZES[0], generator=g), torch.randint(0, SIZES[-1], (n,), generator=g)
    zetas = [torch.randn(n, m, generator=g) for m in SIZES[1:]]
    return x, y, zetas


def params(net, alpha):
    return [getattr(l, k).detach().reshape(-1) for l in net.layers for k in (("theta", "alpha") if alpha else ("theta",))]


def moments(tr, alpha):
    """exp_avg of every trained tensor, in the order of params()"""
    if tr.opt is None:
        flat, offs, off = tr.exp_avg, [], 0
        for p in params(tr.net, alpha):
            offs.append(off)
            off += (p.numel() + 3) // 4 * 4
    else:
        flat, offs = tr.opt.exp_avg, tr.opt.offs
    return [flat[o:o + p.numel()] for p, o in zip(params(tr.net, alpha), offs)]


def run_single(world, out):
    for name, alpha, inject, _ in cases(world):
        B = ROWS * world
        net, tr = build(alpha, inject, B, None)
        rec = []
        for step in range(STEPS):
            x, y, zetas = data(step, B)
            if inject:
                for b, z in zip(tr.buf, zetas):
                    b["zeta"].copy_(z)
            st = tr.step(x, y)
            rec.append({"nll": st["nll"], "kl": st["kl"], "loss": st["loss"],
                        "param": [p.cpu().clone() for p in params(net, alpha)],
                        "exp_avg": [m.cpu().clone() for m in moments(tr, alpha)]})
        torch.save(rec, os.path.join(out, name + ".pt"))
        tr.graph = None
        print(f"single {name}: nll {rec[-1]['nll']:.4f}", flush=True)


def gather(t, world, pg):
    import torch.distributed as dist
    outs = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(outs, t.contiguous(), group=pg)
    return outs


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def arena_params(tr):
    return tr.opt.dp["arena"][:tr.opt.n_flat]


def run_case(name, alpha, inject, mode, rank, world, pg, out):
    import torch.distributed as dist
    os.environ["LBBNN_DP_UPDATE"] = mode
    ref = torch.load(os.path.join(out, name + ".pt"))
    lo, hi = rank * ROWS, (rank + 1) * ROWS
    net, tr = build(alpha, inject, ROWS, pg)
    if mode != "auto":
        assert tr.dp_update == mode, (name, tr.dp_update)
    a0, a1 = tr.opt.dp["arena"].data_ptr(), tr.opt.dp["arena"].data_ptr() + tr.opt.dp["arena"].numel() * 4
    assert all(a0 <= p.data_ptr() < a1 for p in tr.opt.params), (name, "a parameter lives outside the arena")
    worst = 0.0
    for step in range(STEPS):
        x, y, zetas = data(step, ROWS * world)
        if inject:
            for b, z in zip(tr.buf, zetas):
                b["zeta"].copy_(z[lo:hi])
        st = tr.step(x[lo:hi], y[lo:hi])
        r = ref[step]
        tot = torch.tensor([st["nll"], st["loss"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(tot, group=pg)
        assert abs(tot[0].item() - r["nll"]) <= 1e-6 * abs(r["nll"]), (name, step, "sum of nll", tot[0].item(), r["nll"])
        assert abs(tot[1].item() - r["loss"]) <= 1e-6 * abs(r["loss"]), (name, step, "sum of loss", tot[1].item(), r["loss"])
        assert abs(st["kl"] - r["kl"]) <= 1e-6 * abs(r["kl"]), (name, step, "kl", st["kl"], r["kl"])
        kls = gather(torch.tensor([st["kl"]], device="cuda"), world, pg)
        assert all(torch.equal(k, kls[0]) for k in kls), (name, step, "kl differs between ranks")
        for i, (p, m, rp, rm, tp) in enumerate(zip(params(net, alpha), moments(tr, alpha), r["param"], r["exp_avg"],
                                                   tr.opt.params)):
            e = rel(p.cpu(), rp)
            worst = max(worst, e)
            assert e < 1e-6, (name, step, i, "parameters differ from the single-GPU step", e)
            olo, ohi = tr.opt.owned_range(tp)
            if ohi > olo:
                em = rel(m[olo:ohi].cpu(), rm[olo:ohi])
                assert em < 1e-5, (name, step, i, "exp_avg differs from the single-GPU step", em)
    torch.cuda.synchronize()
    flat = arena_params(tr)
    assert all(torch.equal(f, flat) for f in gather(flat, world, pg)), (name, "ranks' parameters differ")
    # the pipelined form per rank: same replay, ranks stay identical
    x, y, _ = data(0, ROWS * world)
    assert tr.step_async(x[lo:hi], y[lo:hi]) is None
    assert tr.step_async(x[lo:hi], y[lo:hi]) is not None and tr.flush() is not None
    torch.cuda.synchronize()
    assert all(torch.equal(f, flat) for f in gather(flat, world, pg)), (name, "ranks diverged under step_async")
    assert tr.kernels_per_step > 0 and int(tr.step_dev) == STEPS + 2 and int(tr.opt.t_dev) == STEPS + 2
    if rank == 0:
        print(f"vd_dp {name}: world {world} OK, worst param rel err {worst:.2e}, update {tr.dp_update}", flush=True)
    tr.graph = None
    return tr.dp_update


def run_dp(out):
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    pg = dist.group.WORLD
    forms = set()
    for name, alpha, inject, mode in cases(world):
        forms.add(run_case(name, alpha, inject, mode, rank, world, pg, out))
    if rank == 0 and world == 1 and "sharded" not in forms:
        print("vd_dp: the fabric reports no multicast for a one-rank group: the sharded form was not exercised", flush=True)
    if world > 1:
        # native noise, the SAME rows on every rank: the rows' zeta is disjoint across ranks, the kl replicated
        os.environ["LBBNN_DP_UPDATE"] = "auto"
        net, tr = build(True, False, ROWS, pg)
        x, y, _ = data(0, ROWS)
        st = tr.step(x, y)
        nlls = gather(torch.tensor([st["nll"], st["kl"]], device="cuda"), world, pg)
        assert not torch.equal(nlls[0][0], nlls[1][0]), "native zeta is the same on every rank"
        assert all(torch.equal(v[1], nlls[0][1]) for v in nlls), "kl differs between ranks"
        tr.graph = None
        del tr, net
        if rank == 0:
            print(f"vd_dp native_noise: world {world} OK, per-rank nll {[round(float(v[0]), 3) for v in nlls]}", flush=True)
        # a rank with another lbbnn.manual_seed: every rank refuses at construction
        try:
            build(False, False, ROWS, pg, seed=1234 if rank else 4321)
        except lbbnn.LbbnnError as e:
            assert "manual_seed" in str(e), e
            if rank == 0:
                print(f"vd_dp mismatched_seed: world {world} OK, refused", flush=True)
        else:
            raise AssertionError("mismatched lbbnn.manual_seed was accepted")
    dist.barrier()
    torch.cuda.synchronize()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("phase", choices=("single", "dp"))
    ap.add_argument("--world", type=int, default=2)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if a.phase == "single":
        run_single(a.world, a.out)
    else:
        run_dp(a.out)


if __name__ == "__main__":
    main()
