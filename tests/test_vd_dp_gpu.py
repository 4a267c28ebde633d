"""AdamW in the multi-tensor Adam table (per-group weight_decay) against torch.optim.AdamW, and data-parallel VDTrainer
against the single-GPU VDTrainer on the concatenated minibatch: a one-rank group, and two ranks (skipped below 2 GPUs).
The data-parallel checks live in tests/vd_dp_worker.py: one plain process computes the reference, then one process per GPU
under torch.distributed.run runs the shards."""
import os
import subprocess
import sys

import pytest
import torch

import cases as C

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "vd_dp_worker.py")
SHAPES = [(400, 784), (75,), (1,), (1023,), (1024,), (1025,), (3, 341), (2049,)]


def _groups(ts):
    """three groups: AdamW at two learning rates and decays, and one without weight decay (torch.optim.Adam's update)"""
    return [{"params": ts[0:3], "lr": 1e-3, "weight_decay": 1e-2},
            {"params": ts[3:6], "lr": 2e-2, "weight_decay": 0.3},
            {"params": ts[6:], "lr": 5e-3, "weight_decay": 0.0}]


@pytest.mark.parametrize("captured", [False, True])
def test_multi_tensor_adam_weight_decay_matches_torch_adamw(captured):
    import lbbnn
    torch.manual_seed(11)
    ps = [torch.nn.Parameter(torch.randn(s, device="cuda")) for s in SHAPES]
    qs = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    rs = [torch.nn.Parameter(p.detach().clone()) for p in ps[6:]]
    ours = lbbnn.MultiTensorAdam(_groups(ps), lr=1e-3, weight_decay=0.5)      # every group sets its own decay
    ref = torch.optim.AdamW(_groups(qs), lr=1e-3)
    adam = torch.optim.Adam(rs, lr=5e-3)                                       # the weight_decay=0 group
    assert [g["weight_decay"] for g in ours.param_groups] == [1e-2, 0.3, 0.0]
    grads = [[torch.randn_like(p) * (10.0 ** (step - 2)) for p in ps] for step in range(5)]
    if captured:
        src = [torch.zeros_like(p) for p in ps]
        for p, s in zip(ps, src):
            p.grad = s
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            ours.step()
        ours.finish_capture()
    for step in range(5):
        for i, p in enumerate(ps):
            if captured:
                p.grad.copy_(grads[step][i])
            else:
                p.grad = grads[step][i].clone()
            qs[i].grad = grads[step][i].clone()
        for r, gr in zip(rs, grads[step][6:]):
            r.grad = gr.clone()
        if captured:
            g.replay()
        else:
            ours.step()
        ref.step()
        adam.step()
        torch.cuda.synchronize()
        for i, (p, q) in enumerate(zip(ps, qs)):
            assert C.rel_err(p.detach(), q.detach()) < 1e-6, (step, i)
        for p, r in zip(ps[6:], rs):
            assert C.rel_err(p.detach(), r.detach()) < 1e-6, step
    assert int(ours.t_dev) == 5


def _run(world, tmp_path):
    r = subprocess.run([sys.executable, WORKER, "single", "--world", str(world), "--out", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    port = 29400 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(port), WORKER, "dp", "--out", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    return r.stdout


def test_one_rank_group_equals_the_single_gpu_trainer(tmp_path):
    """injected and native zeta, alpha fixed and trainable, the auto and nccl update forms, 3 steps"""
    out = _run(1, tmp_path)
    assert out.count(" OK, ") == 8
    assert out.count("update nccl") >= 4
    assert "update sharded" in out or "the sharded form was not exercised" in out


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_equal_the_single_gpu_step_on_the_concatenated_batch(tmp_path):
    """injected zeta sharded by rows, sharded and nccl update, alpha fixed and trainable, 3 steps; native zeta differs
    between ranks; a rank with another lbbnn.manual_seed is refused"""
    out = _run(2, tmp_path)
    assert out.count(" OK, ") == 4 + 2
    assert out.count("update sharded") == 2 and out.count("update nccl") == 2
