"""The data-parallel rule of VDTrainer on the float64 variational-dropout oracle (CPU, gloo with 2 ranks): rows and their
zeta sharded, the replicated KL at 1 / (num_batches * world) on every rank, theta and alpha gradients SUM-reduced -> the
full-batch gradient; the ranks' losses add up to the full batch's loss and the KL is the same on every rank."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, WORLD, NB = 12, 2, 600.0
SIZES = [(10, 16), (16, 12), (12, 4)]     # wide enough that no row of a hidden layer is all zero after the relu


def _case():
    import lbbnn_oracle as O
    rng = np.random.default_rng(11)
    layers = [O.init_vd_params(rng, n, m, dtype=torch.float64) for n, m in SIZES]
    for p in layers:                                   # trainable alpha spread over (0.05, 1), as a trained network's
        p["alpha"] = torch.from_numpy(rng.uniform(0.05, 1.0, size=p["alpha"].shape))
    x = torch.from_numpy(rng.standard_normal((B, SIZES[0][0])))
    y = torch.from_numpy(rng.integers(0, SIZES[-1][1], B))
    zetas = [torch.from_numpy(rng.standard_normal((B, m))) for _, m in SIZES]
    return layers, x, y, zetas


def _leaves(layers):
    return [p[k].clone().requires_grad_(True) for p in layers for k in ("theta", "alpha")]


def _as_layers(leaves):
    return [{"theta": leaves[2 * i], "alpha": leaves[2 * i + 1]} for i in range(len(leaves) // 2)]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import lbbnn_oracle as O
    layers, x, y, zetas = _case()
    rows = slice(rank * B // world, (rank + 1) * B // world)
    mine = _leaves(layers)
    _, nll, kl, _ = O.vd_net_loss(x[rows], y[rows], _as_layers(mine), [z[rows] for z in zetas], NB)
    loss = nll + kl / (NB * world)                     # VDTrainer's per-rank objective
    loss.backward()
    g = torch.cat([t.grad.reshape(-1) for t in mine])
    dist.all_reduce(g)
    s = torch.stack([loss.detach(), nll.detach(), kl.detach()])
    gs = [torch.empty_like(s) for _ in range(world)]
    dist.all_gather(gs, s)
    if rank == 0:
        full = _leaves(layers)
        loss1, nll1, kl1, _ = O.vd_net_loss(x, y, _as_layers(full), zetas, NB)
        loss1.backward()
        ref = (torch.cat([t.grad.reshape(-1) for t in full]), torch.stack([loss1, nll1, kl1]).detach())
        torch.save({"dp": (g, torch.stack(gs)), "single": ref}, out)
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def result(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("vddp") / "dp.pt")
    mp.spawn(_worker, args=(WORLD, 29600 + os.getpid() % 90, out), nprocs=WORLD, join=True)
    return torch.load(out)


def test_sum_reduced_shard_gradients_equal_the_full_batch_gradient(result):
    g_dp, g_1 = result["dp"][0], result["single"][0]
    n_alpha = sum(m for _, m in SIZES)
    assert g_dp.numel() == g_1.numel() == sum(n * m for n, m in SIZES) + n_alpha
    assert ((g_dp - g_1).abs().max() / g_1.abs().max()).item() <= 1e-12


def test_alpha_gradient_counts_the_kl_once(result):
    """The alpha gradient has a KL part at 1 / num_batches: summed over ranks at 1 / (num_batches * world) each it is
    counted once; at 1 / num_batches per rank (the single-GPU scale) it would be counted world times."""
    import lbbnn_oracle as O
    layers, _, _, _ = _case()
    leaves = _leaves(layers)
    kl = sum(O.vd_kl(p["alpha"]) for p in _as_layers(leaves))
    (kl / NB).backward()
    g_kl = torch.cat([(t.grad if t.grad is not None else torch.zeros_like(t)).reshape(-1) for t in leaves])
    g_dp, g_1 = result["dp"][0], result["single"][0]
    over = g_dp + (WORLD - 1) * g_kl                    # what a KL at 1 / num_batches on every rank would give
    assert ((over - g_1).abs().max() / g_1.abs().max()).item() > 1e-6


def test_rank_losses_sum_to_the_full_batch_loss_and_kl_is_replicated(result):
    stats = result["dp"][1]                            # per rank: [loss, nll, kl]
    loss1, nll1, kl1 = result["single"][1].tolist()
    assert torch.equal(stats[0, 2], stats[1, 2])
    assert abs(stats[0, 2].item() - kl1) <= 1e-12 * abs(kl1)
    assert not torch.equal(stats[0, 1], stats[1, 1])
    assert abs(stats[:, 1].sum().item() - nll1) <= 1e-12 * abs(nll1)
    assert abs(stats[:, 0].sum().item() - loss1) <= 1e-12 * abs(loss1)
