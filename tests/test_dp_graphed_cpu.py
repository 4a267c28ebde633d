"""The data-parallel rule of GraphedTrainer on the MNF and MF objectives (oracle, CPU, gloo with 2 ranks): rows sharded,
the parameter-side draws (MNF's z draws and masks and KL-branch draws, MF's masks, weight / bias noise and Gamma draws)
identical on every rank, the replicated terms at 1 / world, gradients SUM-reduced -> the full-batch gradient.  And the block
split of the sharded multi-tensor Adam."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, WORLD, NB = 12, 2, 600.0


def _mnf_case():
    import lbbnn_oracle as O
    rng = np.random.default_rng(3)
    sizes = [(10, 8), (8, 4)]
    layers = [O.init_mnf_params(rng, i, o, num_transforms=2, h_sizes=(6, 6)) for i, o in sizes]
    t = lambda *s: torch.from_numpy(rng.standard_normal(size=s)).float()  # noqa: E731
    m = lambda *s: torch.from_numpy((rng.random(size=s) < 0.5).astype(np.float32))  # noqa: E731
    # one z per layer and step for the whole batch (the reference's zs[-1]): the z-side draws do not depend on the rows
    noises = [{"eps_z": t(1, i), "z_masks": [m(1, i) for _ in range(2)], "eps": t(B, o), "eps_z2": t(1, i),
               "z_masks2": [m(1, i) for _ in range(2)], "eps_r": t(o), "r_masks": [m(i) for _ in range(2)]} for i, o in sizes]
    x, y = torch.from_numpy(rng.random((B, sizes[0][0]))).float(), torch.from_numpy(rng.integers(0, 4, B))
    return layers, noises, x, y


def _mf_case():
    import lbbnn_oracle as O
    rng = np.random.default_rng(4)
    sizes = [(10, 8), (8, 4)]
    layers = [O.init_mf_params(rng, i, o) for i, o in sizes]
    t = lambda *s: torch.from_numpy(rng.standard_normal(size=s)).float()  # noqa: E731
    g = lambda *s: torch.from_numpy(rng.gamma(1.05, size=s)).float()  # noqa: E731
    noises = [{"eps_w": t(o, i), "eps_b": t(o), "g0_w": g(1), "g0_b": g(o)} for i, o in sizes]
    us = [torch.from_numpy(rng.random((o, i))).float() for i, o in sizes]
    x, y = torch.from_numpy(rng.random((B, sizes[0][0]))).float(), torch.from_numpy(rng.integers(0, 4, B))
    return layers, noises, us, x, y


def _leaves(layers):
    out = []
    for p in layers:
        for v in p.values():
            if torch.is_tensor(v):
                out.append(v)
            else:                                   # flows: [{"net": [(W, b)...], "t": (W, b), ...}]
                for tp in v:
                    for part in tp.values():
                        for pair in (part if isinstance(part, list) else [part]):
                            out.extend(pair)
    return out


def _clone(layers):
    import copy
    c = copy.deepcopy(layers)
    for t in _leaves(c):
        t.requires_grad_(True)
    return c


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import lbbnn_oracle as O
    rows = slice(rank * B // world, (rank + 1) * B // world)
    res = {}
    # MNF: the rank's rows and ITS rows of the activation eps; z / KL-branch draws shared; kl at 1 / (NB * world)
    layers, noises, x, y = _mnf_case()
    mine = _clone(layers)
    h = x[rows]
    kl = 0
    for i, (p, nz) in enumerate(zip(mine, noises)):
        h, k = O.mnf_forward(h, p, dict(nz, eps=nz["eps"][rows]))
        kl = kl + k
        h = torch.relu(h) if i < len(mine) - 1 else torch.log_softmax(h, dim=1)
    nll = torch.nn.functional.nll_loss(h, y[rows], reduction="sum")
    (nll + kl / (NB * world)).backward()
    g = torch.cat([t.grad.reshape(-1) for t in _leaves(mine)])
    dist.all_reduce(g)
    s = torch.stack([nll.detach(), kl.detach()])
    gs = [torch.empty_like(s) for _ in range(world)]
    dist.all_gather(gs, s)
    res["mnf"] = (g, torch.stack(gs))
    # MF: one sample of masks / weights / precisions for the whole batch; (log q - log prior) at 1 / (NB * world)
    layers, noises, us, x, y = _mf_case()
    mine = _clone(layers)
    _, nll, log_p, log_q, _, _ = O.mf_net_elbo(x[rows], y[rows], mine, noises, us, NB)
    (nll + (log_q - log_p) / (NB * world)).backward()
    g = torch.cat([t.grad.reshape(-1) for t in _leaves(mine)])
    dist.all_reduce(g)
    s = torch.stack([nll.detach(), log_p.detach(), log_q.detach()])
    gs = [torch.empty_like(s) for _ in range(world)]
    dist.all_gather(gs, s)
    res["mf"] = (g, torch.stack(gs))
    if rank == 0:
        ref = {}
        layers, noises, x, y = _mnf_case()
        full = _clone(layers)
        loss, nll, kl, _ = O.mnf_net_loss(x, y, full, noises, NB)
        loss.backward()
        ref["mnf"] = (torch.cat([t.grad.reshape(-1) for t in _leaves(full)]), nll.detach(), kl.detach())
        layers, noises, us, x, y = _mf_case()
        full = _clone(layers)
        loss, nll, log_p, log_q, _, _ = O.mf_net_elbo(x, y, full, noises, us, NB)
        loss.backward()
        ref["mf"] = (torch.cat([t.grad.reshape(-1) for t in _leaves(full)]), nll.detach(), torch.stack([log_p, log_q]).detach())
        torch.save({"dp": res, "single": ref}, out)
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def result(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("dpg") / "dp.pt")
    mp.spawn(_worker, args=(WORLD, 29700 + os.getpid() % 90, out), nprocs=WORLD, join=True)
    return torch.load(out)


@pytest.mark.parametrize("kind", ["mnf", "mf"])
def test_sum_reduced_shard_gradients_equal_the_full_batch_gradient(result, kind):
    g_dp, g_1 = result["dp"][kind][0], result["single"][kind][0]
    assert ((g_dp - g_1).norm() / g_1.norm()).item() <= 2e-6


@pytest.mark.parametrize("kind", ["mnf", "mf"])
def test_rows_are_sharded_and_replicated_terms_are_shared(result, kind):
    stats = result["dp"][kind][1]                  # per rank: [nll, replicated terms...]
    # the parameter-side draws are the same on every rank: the replicated terms agree bitwise
    assert torch.equal(stats[0, 1:], stats[1, 1:])
    # the rows are split: the ranks' nll differ and add up to the full batch's
    assert not torch.equal(stats[0, 0], stats[1, 0])
    assert abs(stats[:, 0].sum().item() - result["single"][kind][1].item()) <= 1e-5 * abs(result["single"][kind][1].item())
    assert torch.allclose(stats[0, 1:], result["single"][kind][2].reshape(-1), rtol=1e-6, atol=0)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("total", [1, 5, 8, 3437, 4099])
def test_owned_blocks_cover_every_block_once(world, total):
    from lbbnn.engine import shard_blocks
    hits = np.zeros(total, dtype=np.int64)
    for r in range(world):
        lo, hi = shard_blocks(total, world, r)
        assert 0 <= lo <= hi <= total
        hits[lo:hi] += 1
    assert (hits == 1).all()
