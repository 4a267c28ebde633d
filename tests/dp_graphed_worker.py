"""Worker of tests/test_dp_graphed_gpu.py: data-parallel GraphedTrainer (MNF, MF, LRT networks) against the single-GPU
trainer on the concatenated minibatch.

    python tests/dp_graphed_worker.py single --world W --out DIR          one process, one GPU: the reference runs
    python -m torch.distributed.run --nproc-per-node W tests/dp_graphed_worker.py dp --out DIR

Both phases build the same networks in the same order with the same seeds (layer ids and call counts key the native noise,
so the parameter-side draws of the two runs coincide).  The per-row activation noise of the MNF / LRT layers is injected
(the rank's slice of the reference's rows); MF has none.  Exits non-zero on a mismatch; rank 0 prints one line per case."""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "bayesian-neural-nets_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import lbbnn  # noqa: E402

NB = 600
SMALL, LARGE = (72, 40, 24, 10), (784, 400, 600, 10)


class InjectedMNF(lbbnn.mnf.BayesianNetwork):
    """MNF network whose activation noise is the fixed buffers `eps` (rows of this process)."""
    eps = None

    def _logits(self, x, sample=False, noises=None, calculate_log_probs=False):
        if self.eps is not None:
            noises = [{"eps": e} for e in self.eps]
        return super()._logits(x, sample, noises, calculate_log_probs)


class InjectedLRT(lbbnn.BayesianNetwork):
    eps = None

    def forward(self, x, sample=False, eps=None):
        return super().forward(x, sample, eps=self.eps if self.eps is not None else eps)


def cases(world):
    """(name, kind, sizes, rows per rank, trainer kwargs, environment)"""
    out = []
    for mode in (("sharded", "nccl") if world > 1 else ("auto",)):
        env = {"LBBNN_DP_UPDATE": mode}
        out += [(f"mnf_split[{mode}]", "mnf", SMALL, 32, {}, dict(env, LBBNN_ADAM_SPLIT="1")),
                (f"mnf_nosplit[{mode}]", "mnf", SMALL, 32, {}, dict(env, LBBNN_ADAM_SPLIT="0")),
                (f"mnf_torch_objective[{mode}]", "mnf", SMALL, 32, {"fuse_objective": False}, env),
                (f"mf_33_groups[{mode}]", "mf", SMALL, 32, {}, env),
                (f"lrt[{mode}]", "lrt", SMALL, 32, {}, env),
                (f"mnf_784[{mode}]", "mnf", LARGE, 50, {}, env),
                (f"mf_784[{mode}]", "mf", LARGE, 50, {}, env)]
    return out


def build(kind, sizes, rows, eps_rows, kw, pg):
    """Network + trainer; eps_rows: (lo, hi) of the reference rows this process feeds (None: native noise)."""
    torch.manual_seed(7)
    lbbnn.manual_seed(1234)
    dev = torch.device("cuda", torch.cuda.current_device())
    if kind == "mnf":
        net = InjectedMNF(sizes).to(dev)
    elif kind == "lrt":
        net = InjectedLRT(sizes).to(dev)
    else:
        net = lbbnn.mf.BayesianNetwork(sizes, num_batches=NB).to(dev)
    if kind != "mf" and eps_rows is not None:
        g = torch.Generator().manual_seed(99)
        full = [torch.randn(4096, o, generator=g) for o in sizes[1:]]
        net.eps = [e[eps_rows[0]:eps_rows[1]].contiguous().to(dev) for e in full]
    elif kind != "mf":
        net.eps = None
    if kind == "mf":
        tr = lbbnn.GraphedTrainer(net, batch_size=rows, num_batches=NB, lr=1e-4, objective="elbo",
                                  param_groups=lbbnn.mf.reference_param_groups(net), process_group=pg, **kw)
    else:
        tr = lbbnn.GraphedTrainer(net, batch_size=rows, num_batches=NB, lr=1e-3, objective="kl", process_group=pg, **kw)
    return net, tr


def batch(sizes, n):
    g = torch.Generator().manual_seed(5)
    return torch.rand(n, sizes[0], generator=g), torch.randint(0, sizes[-1], (n,), generator=g)


def names(net, tr):
    ids = {id(p): n for n, p in net.named_parameters()}
    return [(ids[id(p)], p, off) for p, off in zip(tr.opt.params, tr.opt.offs)]


def replicated_terms(net, kind):
    if kind == "mf":
        return torch.stack([t.detach().reshape(()) for l in net.layers for t in (l.log_prior, l.log_variational_posterior)])
    return torch.stack([l.kl.detach().reshape(()) for l in net.layers])


def run_single(world, out):
    for name, kind, sizes, rows, kw, env in cases(world):
        os.environ.update(env)
        B = rows * world
        net, tr = build(kind, sizes, B, (0, B), kw, None)
        x, y = batch(sizes, B)
        st = tr.step(x, y)
        torch.cuda.synchronize()
        rec = {"nll": st["nll"], "exp_avg": {}, "param": {}}
        for n, p, off in names(net, tr):
            rec["exp_avg"][n] = tr.opt.exp_avg[off:off + p.numel()].cpu().clone()
            rec["param"][n] = p.detach().reshape(-1).cpu().clone()
        torch.save(rec, os.path.join(out, name + ".pt"))
        tr.graph = None
        print(f"single {name}: nll {st['nll']:.6f}", flush=True)


def gather(t, world, pg):
    import torch.distributed as dist
    outs = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(outs, t.contiguous(), group=pg)
    return outs


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def run_dp(out):
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    pg = dist.group.WORLD
    for name, kind, sizes, rows, kw, env in cases(world):
        os.environ.update(env)
        ref = torch.load(os.path.join(out, name + ".pt"))
        lo, hi = rank * rows, (rank + 1) * rows
        net, tr = build(kind, sizes, rows, (lo, hi), kw, pg)
        D = tr.opt.dp
        a0, a1 = D["arena"].data_ptr(), D["arena"].data_ptr() + D["arena"].numel() * 4
        assert all(a0 <= p.data_ptr() < a1 for p in tr.opt.params), (name, "a parameter lives outside the arena")
        x, y = batch(sizes, rows * world)
        st = tr.step(x[lo:hi], y[lo:hi])
        torch.cuda.synchronize()
        worst, owned = 0.0, 0
        for n, p, off in names(net, tr):
            m = tr.opt.exp_avg[off:off + p.numel()].cpu()
            olo, ohi = tr.opt.owned_range(p)
            owned += ohi - olo
            if ohi > olo:
                err = rel(m[olo:ohi], ref["exp_avg"][n][olo:ohi])
                worst = max(worst, err)
                assert err < 2e-5, (name, n, "exp_avg differs from the single-GPU step", err)
            rest = torch.cat([m[:olo], m[ohi:]])
            assert not rest.numel() or float(rest.abs().max()) == 0.0, (name, n, "moments outside the owned range changed")
            perr = rel(p.detach().reshape(-1).cpu(), ref["param"][n])
            assert perr < 1e-5, (name, n, "parameters after step 1 differ from the single-GPU step", perr)
        cover = torch.tensor([owned], device="cuda")
        dist.all_reduce(cover, group=pg)
        n_all = sum(p.numel() for p in tr.opt.params)
        assert int(cover) == (n_all if D["mode"] == "sharded" else n_all * world), (name, int(cover), n_all)
        nll = torch.tensor([st["nll"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(nll, group=pg)
        assert abs(nll.item() - ref["nll"]) <= 2e-5 * abs(ref["nll"]), (name, nll.item(), ref["nll"])
        terms = gather(replicated_terms(net, kind), world, pg)
        assert all(torch.equal(t, terms[0]) for t in terms), (name, "replicated terms differ between ranks")
        for _ in range(4):
            tr.step(x[lo:hi], y[lo:hi], read_loss=False)
        torch.cuda.synchronize()
        flat = D["arena"][:tr.opt.n_flat]
        assert all(torch.equal(f, flat) for f in gather(flat, world, pg)), (name, "ranks diverged after 5 steps")
        if rank == 0:
            print(f"dp_graphed {name}: world {world} OK, worst exp_avg rel err {worst:.2e}, update {D['mode']}", flush=True)
        tr.graph = None
        del tr, net
    # native noise, the SAME rows on every rank: parameter-side draws shared, per-row activation noise disjoint
    os.environ["LBBNN_DP_UPDATE"] = "auto"
    for kind in ("mnf", "mf"):
        net, tr = build(kind, SMALL, 32, None, {}, pg)
        x, y = batch(SMALL, 32)
        first = tr.step(x, y)
        terms = gather(replicated_terms(net, kind), world, pg)
        assert all(torch.equal(t, terms[0]) for t in terms), (kind, "parameter-side draws differ between ranks")
        nlls = gather(torch.tensor([first["nll"]], device="cuda"), world, pg)
        if kind == "mf":
            assert all(torch.equal(v, nlls[0]) for v in nlls), ("mf", "nll differs on identical rows", nlls)
        elif world > 1:
            assert not torch.equal(nlls[0], nlls[1]), ("mnf", "activation noise is the same on every rank")
        for _ in range(59):
            last = tr.step(x, y)
        assert last["nll"] < first["nll"], (kind, "60 data-parallel steps did not lower the nll", first, last)
        if rank == 0:
            print(f"dp_graphed native_{kind}: world {world} OK, nll {first['nll']:.3f} -> {last['nll']:.3f}", flush=True)
        tr.graph = None
        del tr, net
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
