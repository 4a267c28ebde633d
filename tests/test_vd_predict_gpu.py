"""lbbnn.vd.EnsemblePredictor (the evaluation branch of run_epoch, VD:148-157, batched over MC samples) on both GEMM paths:
against the reference's own network output (tests/golden/vd.npz), against a float64 forward on the GPU at the
784-1200-1200-1200-10 shape, against the eager predict_ensemble loop, on native noise (exported streams, launch width, run
splits, odd shapes), its gemm="auto" selection and launch counts, and parameter updates between runs.  Tolerances as in
test_predict_gpu.py: 1e-5 relative on accumulators, argmax identical except on near-tie rows."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import cases as C
import lbbnn_oracle as O
from test_predict_gpu import _same_argmax
from test_vd_gpu import _load_net

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vd():
    import lbbnn.vd
    return lbbnn.vd


def _net(vd, sizes, seed, **kw):
    torch.manual_seed(seed)
    return vd.BNN(sizes=sizes, **kw).cuda()


def _oracle_logp(net, x, zetas, s):
    """float64 forward of sample s (BNN.forward, VD:79-85) with the injected zeta of every layer"""
    h = x.double().reshape(x.shape[0], -1)
    L = len(net.layers)
    for i, (l, z) in enumerate(zip(net.layers, zetas)):
        h = O.vd_forward(h, l.theta.detach().double(), l.alpha.detach().double(), z[s].double())
        h = F.relu(h) if i < L - 1 else F.log_softmax(h, dim=1)
    return h


def _oracle_sum(net, x, zetas, S):
    return sum(_oracle_logp(net, x, zetas, s) for s in range(S))


def _zetas(net, S, B, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(S, B, l.m, device="cuda", generator=g) for l in net.layers]


@pytest.mark.parametrize("gemm", ["simt", "tc"])
def test_reference_anchor(vd, gemm):
    """One sample with the reference case's zeta reproduces the reference's own BNN output."""
    g = np.load(os.path.join(C.GOLDEN, "vd.npz"))
    case = C.vd_net_case(seed=80, batch=100)
    net = _load_net(vd, case)
    p = vd.EnsemblePredictor(net, batch=100, samples_per_launch=1, seed=1, gemm=gemm)
    assert p.tc == ([True, True, True, False] if gemm == "tc" else [False] * 4)
    p.run(case["x"].cuda(), 1, zetas=[z.cuda()[None] for z in case["zetas"]])
    out = p.result()
    assert C.rel_err(out["mean_logp"], g["net_logp"]) < 1e-5
    assert torch.equal(out["pred"].cpu(), torch.from_numpy(g["net_logp"]).argmax(1))


@pytest.fixture(scope="module")
def wide(vd):
    """784-1200-1200-1200-10 at batch 256, 24 injected samples, and the float64 sum of their log-probabilities"""
    S, B = 24, 256
    net = _net(vd, (784, 1200, 1200, 1200, 10), 21)
    x = torch.randn(B, 784, device="cuda", generator=torch.Generator(device="cuda").manual_seed(22))
    zetas = _zetas(net, S, B, 23)
    with torch.no_grad():
        ref = _oracle_sum(net, x, zetas, S)
    return net, x, zetas, ref, S, B


@pytest.mark.parametrize("gemm", ["simt", "tc"])
@pytest.mark.parametrize("spl", [1, 5, 12])
def test_against_float64(vd, wide, gemm, spl):
    net, x, zetas, ref, S, B = wide
    p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=spl, seed=3, gemm=gemm)
    p.run(x, S, zetas=zetas)
    assert C.rel_err(p.sum_logp, ref) < 1e-5
    assert _same_argmax(p.result()["pred"], ref.cpu())


@pytest.mark.parametrize("gemm", ["simt", "tc"])
def test_same_statistic_as_the_eager_loop(vd, gemm):
    """predict_ensemble's statistic (VD:148-157): the eager loop over model(x, zetas=...) with the same per-sample zeta."""
    S, B = 7, 100
    case = C.vd_net_case(seed=81, batch=B)
    net = _load_net(vd, case)
    x = case["x"].cuda()
    zetas = _zetas(net, S, B, 31)
    with torch.no_grad():
        acc = None
        for s in range(S):
            out = net(x, zetas=[z[s] for z in zetas])
            acc = out if acc is None else acc + out
        loop = acc / S
    p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=3, seed=4, gemm=gemm)
    got = p.predict_ensemble(x, S, zetas=zetas)
    assert got.dtype == torch.float32 and got.shape == (B, 10)
    assert C.rel_err(got, loop) < 1e-5
    assert _same_argmax(got.argmax(1), loop.double().cpu())
    assert vd.predict_ensemble(net, x, samples=2).shape == (B, 10)       # the eager entry point is unchanged


def _exported(vd, p, net, S):
    """The predictor's native zeta, materialised stream by stream: sample g of layer l = stream (0x5E << 56) | (l + g L)"""
    L = len(net.layers)
    return [torch.stack([vd.K.philox_normal((p.B, l.m), p.seed, (0x5E << 56) | (li + g * L)) for g in range(S)])
            for li, l in enumerate(net.layers)]


@pytest.mark.parametrize("gemm", ["simt", "tc"])
def test_native_noise(vd, gemm):
    S, B = 9, 64
    net = _net(vd, (784, 1200, 1200, 1200, 10), 41)
    x = torch.randn(B, 784, device="cuda")
    runs = []
    for spl in (4, 9, 1):
        p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=spl, seed=77, gemm=gemm)
        p.run(x, S)
        runs.append(p.sum_logp.clone())
    for r in runs[1:]:
        assert C.rel_err(r, runs[0]) < 1e-6                  # independent of the launch width
    p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=4, seed=77, gemm=gemm)
    p.run(x, S, zetas=_exported(vd, p, net, S))
    assert C.rel_err(p.sum_logp, runs[0]) < 1e-6             # exactly the exported streams
    with torch.no_grad():
        assert C.rel_err(runs[0], _oracle_sum(net, x, _exported(vd, p, net, S), S)) < 1e-5
    p.run(x, 3)                                              # [0, 3) + [3, 9): the second run starts inside a launch
    part = p.sum_logp.clone()
    p.run(x, 6, first_sample=3)
    assert C.rel_err(part + p.sum_logp, runs[0]) < 1e-6


def test_native_noise_tc_and_simt_agree(vd):
    S, B = 6, 64
    net = _net(vd, (784, 1200, 1200, 1200, 10), 42)
    x = torch.randn(B, 784, device="cuda")
    sums = {}
    for gemm in ("simt", "tc"):
        p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=4, seed=78, gemm=gemm)
        p.run(x, S)
        sums[gemm] = p.sum_logp.clone()
    assert C.rel_err(sums["tc"], sums["simt"]) < 1e-5


@pytest.mark.parametrize("sizes", [(30, 45, 7), (33, 64, 13)])
def test_native_noise_odd_shapes_on_the_cuda_cores(vd, sizes):
    """Odd batch and odd output widths: every element draws from its sample's stream (no vector path), stacked or not."""
    S, B = 5, 13
    net = _net(vd, sizes, 43)
    x = torch.randn(B, sizes[0], device="cuda")
    p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=2, seed=79, gemm="simt")
    assert not any(p.tc)
    p.run(x, S)
    native = p.sum_logp.clone()
    p.run(x, S, zetas=_exported(vd, p, net, S))
    assert C.rel_err(native, p.sum_logp) < 1e-6
    with torch.no_grad():
        assert C.rel_err(native, _oracle_sum(net, x, _exported(vd, p, net, S), S)) < 1e-5
    q = vd.EnsemblePredictor(net, batch=B, samples_per_launch=5, seed=79, gemm="simt")
    q.run(x, S)
    assert C.rel_err(q.sum_logp, native) < 1e-6


def test_auto_selection_and_launch_counts(vd):
    lib = vd.K.lib
    B, spl = 16, 3
    net = _net(vd, (784, 1200, 1200, 1200, 10), 51)
    p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=spl, seed=2)
    assert p.tc == [False, True, True, False]
    p.run(torch.randn(B, 784, device="cuda"), spl)
    # layer 1: epilogue on the per-run moments, writing layer 2's operands; layers 2, 3: two GEMMs + epilogue;
    # head: the CUDA-core forward; one accumulation
    assert p.kernels_per_launch == 1 + 3 + 3 + lib.lbbnn_vd_gemm_launches(spl * B, 10, 1200) + 1
    small = _net(vd, (784, 64, 64, 10), 52)
    p = vd.EnsemblePredictor(small, batch=B, samples_per_launch=spl, seed=2)
    assert p.tc == [False, False, False]
    p.run(torch.randn(B, 784, device="cuda"), spl)
    assert p.kernels_per_launch == (1 + lib.lbbnn_vd_gemm_launches(spl * B, 64, 64) + lib.lbbnn_vd_gemm_launches(spl * B, 10, 64)
                                    + 1)
    # a CUDA-core layer (64 -> 1024) feeding a tensor-core one: its activations are split for the next layer's GEMMs
    mixed = _net(vd, (784, 64, 1024, 1024, 10), 53)
    x = torch.randn(B, 784, device="cuda")
    p = vd.EnsemblePredictor(mixed, batch=B, samples_per_launch=spl, seed=2)
    q = vd.EnsemblePredictor(mixed, batch=B, samples_per_launch=spl, seed=2, gemm="simt")
    assert p.tc == [False, False, True, False]
    p.run(x, 2 * spl)
    q.run(x, 2 * spl)
    assert p.kernels_per_launch == 1 + lib.lbbnn_vd_gemm_launches(spl * B, 1024, 64) + 1 + 3 + \
        lib.lbbnn_vd_gemm_launches(spl * B, 10, 1024) + 1
    assert C.rel_err(p.sum_logp, q.sum_logp) < 1e-5
    with pytest.raises(ValueError):
        vd.EnsemblePredictor(net, batch=B, gemm="bf16")


@pytest.mark.parametrize("gemm", ["simt", "tc"])
def test_parameter_updates_and_bad_inputs(vd, gemm):
    import lbbnn
    S, B = 3, 32
    net = _net(vd, (784, 1024, 1024, 10), 61, alpha_trainable=True)
    x = torch.randn(B, 784, device="cuda")
    zetas = _zetas(net, S, B, 62)
    p = vd.EnsemblePredictor(net, batch=B, samples_per_launch=2, seed=5, gemm=gemm)
    p.run(x, S, zetas=zetas)
    with torch.no_grad():
        assert C.rel_err(p.sum_logp, _oracle_sum(net, x, zetas, S)) < 1e-5
        for l in net.layers:
            l.theta.mul_(-1.3)
        p.run(x, S, zetas=zetas)
        assert C.rel_err(p.sum_logp, _oracle_sum(net, x, zetas, S)) < 1e-5
        for i, l in enumerate(net.layers):
            l.alpha.copy_(torch.linspace(0.05, 0.9, l.m, device="cuda").roll(i))
        p.run(x, S, zetas=zetas)
        assert C.rel_err(p.sum_logp, _oracle_sum(net, x, zetas, S)) < 1e-5
    with pytest.raises(lbbnn.LbbnnError):
        p.run(x.cpu(), S)
    with pytest.raises(lbbnn.LbbnnError):
        p.run(x[:, :700].contiguous(), S)
    with pytest.raises(lbbnn.LbbnnError):
        p.run(x, S, zetas=[z[:, :, :5] for z in zetas])
    with pytest.raises(lbbnn.LbbnnError):
        p.run(x, S + 1, zetas=zetas)
    with pytest.raises(lbbnn.LbbnnError):
        p.run(x, S, zetas=[z.cpu() for z in zetas])
    with pytest.raises(lbbnn.LbbnnError):
        vd.EnsemblePredictor(vd.BNN(sizes=(8, 4, 2)), batch=2)
