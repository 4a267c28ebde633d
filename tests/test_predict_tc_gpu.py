"""lbbnn.EnsemblePredictor with its layers on the tensor cores (gemm="tc": 3xTF32 tcgen05 GEMMs around lbbnn_lrt_mc_epilogue)
against tests/golden/ensemble.npz, against the CUDA-core path on the same native noise, at the 4096-wide shape against a
float64 forward on the GPU, and the gemm="auto" selection.  Tolerances as in test_predict_gpu.py: 1e-5 on accumulators and
probabilities, argmax bit-exact except on near-tie rows."""
import os

import numpy as np
import pytest
import torch

import cases as C
import lbbnn_oracle as O
from test_predict_gpu import G, _load_lrt, _same_argmax

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def _load_mnf(lb, case):
    net = lb.mnf.BayesianNetwork()
    for l, p in zip(net.layers, case["layers"]):
        l.load_state_dict(C.flat_named(p))
    return net.cuda().eval()


@pytest.mark.parametrize("spl", [12, 5, 1])
def test_lrt_tc_predictor_matches_the_reference_loop(lb, spl):
    S, B = 12, 52
    case = C.ensemble_case(seed=120, batch=B, samples=S, kind="lrt")
    net = _load_lrt(lb, case)
    pred = lb.EnsemblePredictor(net, batch=B, samples_per_launch=spl, seed=11, gemm="tc")
    assert pred.tc == [True, True, False]
    eps = [e.cuda() for e in case["eps"]]
    out = pred.test_ensemble(case["x"].cuda(), S, ensemble_first=10, eps=eps)
    outputs = torch.from_numpy(G["lrt_outputs"]).double()
    assert C.rel_err(pred.sum_logp, outputs.sum(0)) < 1e-5
    assert C.rel_err(pred.first_logp, outputs[0:10].sum(0)) < 1e-5
    assert C.rel_err(out["mean_prob"], G["lrt_mean_prob"]) < 1e-5
    assert C.rel_err(out["entropy"], G["lrt_entropy"]) < 1e-5
    assert _same_argmax(out["ensemble"], outputs[0:10].mean(0))
    assert _same_argmax(out["posterior_mean"], G["lrt_posterior_mean_logp"])
    oos = pred.outofsample(case["x"].cuda(), S, eps=eps)
    assert C.rel_err(oos["entropy"], G["lrt_entropy"]) < 1e-5 and C.rel_err(oos["mean_prob"], G["lrt_mean_prob"]) < 1e-5
    assert _same_argmax(oos["pred"], outputs[1:S].mean(0))


@pytest.mark.parametrize("spl", [12, 5, 1])
def test_mnf_tc_predictor_matches_the_reference_loop(lb, spl):
    S, B = 6, 52
    case = C.ensemble_case(seed=121, batch=B, samples=S, kind="mnf")
    net = _load_mnf(lb, case)
    z_noise = [{"eps_z": case["eps_z"][l][:, -1].cuda(), "z_masks": [m[:, -1].cuda() for m in case["z_masks"][l]]} for l in range(3)]
    eps = [e.cuda() for e in case["eps"]]
    outputs = torch.from_numpy(G["mnf_outputs"]).double()
    pred = lb.EnsemblePredictor(net, batch=B, samples_per_launch=spl, seed=5, gemm="tc")
    assert pred.mnf and pred.tc == [True, True, False]
    pred.run(case["x"].cuda(), S, eps=eps, z_noise=z_noise)
    out = pred.result(S)
    assert C.rel_err(pred.sum_logp, outputs.sum(0)) < 1e-5
    assert C.rel_err(out["mean_prob"], G["mnf_mean_prob"]) < 1e-5 and C.rel_err(out["entropy"], G["mnf_entropy"]) < 1e-5
    assert _same_argmax(out["ensemble"], outputs[0:10].mean(0))
    oos = pred.outofsample(case["x"].cuda(), S, eps=eps, z_noise=z_noise)
    assert C.rel_err(oos["entropy"], G["mnf_entropy"]) < 1e-5 and _same_argmax(oos["pred"], outputs[1:S].mean(0))


def test_tc_and_simt_agree_on_native_noise(lb):
    """Same Philox streams on both paths: the tensor-core epilogue draws what lbbnn_lrt_f32_fwd_ex / sample_expand draw.
    MNF: injected z (native z is a fresh draw per call), native eps."""
    S, B = 9, 52
    case = C.ensemble_case(seed=122, batch=B, samples=S, kind="lrt")
    net = _load_lrt(lb, case)
    x = case["x"].cuda()
    sums = {}
    for gemm in ("simt", "tc"):
        p = lb.EnsemblePredictor(net, batch=B, samples_per_launch=4, seed=77, gemm=gemm)
        p.run(x, S)
        sums[gemm] = (p.sum_logp.clone(), p.sum_prob.clone(), p.first_logp.clone())
    for a, b in zip(sums["tc"], sums["simt"]):
        assert C.rel_err(a, b) < 1e-5
    mc = C.ensemble_case(seed=121, batch=B, samples=6, kind="mnf")
    mnet = _load_mnf(lb, mc)
    z_noise = [{"eps_z": mc["eps_z"][l][:, -1].cuda(), "z_masks": [m[:, -1].cuda() for m in mc["z_masks"][l]]} for l in range(3)]
    for gemm in ("simt", "tc"):
        p = lb.EnsemblePredictor(mnet, batch=B, samples_per_launch=4, seed=78, gemm=gemm)
        p.run(mc["x"].cuda(), 6, z_noise=z_noise)
        sums[gemm] = p.sum_logp.clone()
    assert C.rel_err(sums["tc"], sums["simt"]) < 1e-5


def test_tc_predictor_is_launch_width_invariant(lb):
    S, B = 9, 52
    case = C.ensemble_case(seed=122, batch=B, samples=S, kind="lrt")
    net = _load_lrt(lb, case)
    x = case["x"].cuda()
    runs = []
    for spl in (9, 4, 1):
        p = lb.EnsemblePredictor(net, batch=B, samples_per_launch=spl, seed=77, gemm="tc")
        p.run(x, S)
        runs.append((p.sum_logp.clone(), p.sum_prob.clone(), p.first_logp.clone()))
        # layer 1: epilogue only (E1, S1 per batch); layer 2: two GEMMs + epilogue; head: fused fp32 forward; 2 accumulations
        assert p.kernels_per_launch == 1 + 3 + 3 + 2
    for r in runs[1:]:
        for a, b in zip(r, runs[0]):
            assert C.rel_err(a, b) < 1e-6
    p.run(x, 4, first_sample=0)
    part = p.sum_logp.clone()
    p.run(x, 5, first_sample=4)
    assert C.rel_err(part + p.sum_logp, runs[0][0]) < 1e-6


def _params64(net):
    return [{k: getattr(l, k).detach().double() for k in ("weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho")}
            for l in net.layers]


def _rng_and_keys(net):
    """torch's CUDA RNG state and the noise-key counters of the network's modules (the native MNF z draws)"""
    return torch.cuda.get_rng_state(), [m._calls for m in net.modules() if hasattr(m, "_calls")]


def _restore(net, state):
    torch.cuda.set_rng_state(state[0])
    for m, v in zip([m for m in net.modules() if hasattr(m, "_calls")], state[1]):
        m._calls = v


def test_mnf_cuda_core_layer_feeding_a_tensor_core_layer(lb):
    """MNF 30-400-600-10 under gemm="tc": layer 1 (in % 4 != 0) stays on the CUDA cores and its activations are split with the
    next layer's z as the row scale (tf32_split_rows, per-sample stride); against the CUDA-core predictor, same draws."""
    S, B = 6, 52
    sizes = [(30, 400), (400, 600), (600, 10)]
    case = C.ensemble_case(seed=123, batch=B, samples=S, sizes=sizes, kind="mnf")
    net = lb.mnf.BayesianNetwork(sizes=(30, 400, 600, 10))
    for l, p in zip(net.layers, case["layers"]):
        l.load_state_dict(C.flat_named(p))
    net = net.cuda().eval()
    z_noise = [{"eps_z": case["eps_z"][l][:, -1].cuda(), "z_masks": [m[:, -1].cuda() for m in case["z_masks"][l]]} for l in range(3)]
    eps = [e.cuda() for e in case["eps"]]
    sums = {}
    for gemm in ("simt", "tc"):
        p = lb.EnsemblePredictor(net, batch=B, samples_per_launch=4, seed=6, gemm=gemm)
        p.run(case["x"].cuda(), S, eps=eps, z_noise=z_noise)
        sums[gemm] = (p.sum_logp.clone(), p.sum_prob.clone())
        if gemm == "tc":
            assert p.tc == [False, True, False]
            assert p.kernels_per_launch == 3 + 1 + 3 + 3 + 2      # fp32 layer, split, tensor-core layer, head, accumulations
    for a, b in zip(sums["tc"], sums["simt"]):
        assert C.rel_err(a, b) < 1e-5


def test_mnf_shards_starting_inside_a_launch(lb):
    """Shards of a global run whose first sample is not a multiple of samples_per_launch (native z: each run() draws the
    z of the whole global run, launch by launch from sample 0, and takes its own rows) add up to the whole run."""
    S, B = 9, 52
    case = C.ensemble_case(seed=121, batch=B, samples=S, kind="mnf")
    net = _load_mnf(lb, case)
    x = case["x"].cuda()
    p = lb.EnsemblePredictor(net, batch=B, samples_per_launch=4, seed=8, gemm="tc")
    state = _rng_and_keys(net)
    p.run(x, S, global_samples=S)
    full = (p.sum_logp.clone(), p.sum_prob.clone(), p.first_logp.clone())
    assert C.rel_err(p.result()["mean_prob"], full[1] / S) == 0.0
    parts = [torch.zeros_like(t) for t in full]
    for first, count in ((0, 3), (3, 6)):
        _restore(net, state)
        p.run(x, count, first_sample=first, global_samples=S)
        for acc, t in zip(parts, (p.sum_logp, p.sum_prob, p.first_logp)):
            acc += t
    for a, b in zip(parts, full):
        assert C.rel_err(a, b) < 1e-6


def _wide_net(lb, sizes, seed):
    torch.manual_seed(seed)
    net = lb.BayesianNetwork(sizes).cuda().eval()
    with torch.no_grad():
        for l in net.layers:
            l.lambdal.normal_(0.0, 2.0)
            l.weight_mu.mul_(0.05)     # keep the 4096-wide pre-activations O(1)
    return net


def test_wide_lrt_against_float64(lb):
    """4096-4096-4096-10 at batch 512: both GEMM products of both wide layers on the tensor cores; the log-softmax sums and
    the posterior-mean logits against a float64 forward on the GPU with the same injected eps."""
    sizes, B, S = (4096, 4096, 4096, 10), 512, 3
    net = _wide_net(lb, sizes, 3)
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.rand(B, sizes[0], device="cuda", generator=g)
    eps = [torch.randn(S, B, o, device="cuda", generator=g) for o in sizes[1:]]
    pred = lb.EnsemblePredictor(net, batch=B, samples_per_launch=2, seed=1, gemm="tc")
    assert pred.tc == [True, True, False]
    layers = _params64(net)
    # a fresh predictor: mean_logits reads the current parameters without a run() before it
    mean_ref = O.lrt_net_forward(x.double(), layers, sample=False)
    assert C.rel_err(torch.log_softmax(pred.mean_logits(x).double(), 1), mean_ref) < 1e-5
    pred.run(x, S, eps=eps)
    ref = [O.lrt_net_forward(x.double(), layers, [e[s].double() for e in eps]) for s in range(S)]
    ref_sum = torch.stack(ref).sum(0)
    assert C.rel_err(pred.sum_logp, ref_sum) < 1e-5
    assert _same_argmax(pred.result(S)["ensemble"], ref_sum.cpu())
    logits = pred.mean_logits(x)
    assert C.rel_err(torch.log_softmax(logits.double(), 1), mean_ref) < 1e-5
    assert _same_argmax(logits.argmax(1), mean_ref.cpu())
    out = pred.test_ensemble(x, S, eps=eps)
    assert torch.equal(out["posterior_mean"], logits.argmax(1))
    # after a parameter update the next mean_logits follows it, with no run() in between
    with torch.no_grad():
        for l in net.layers:
            l.weight_mu.mul_(-1.5)
    mean_ref = O.lrt_net_forward(x.double(), _params64(net), sample=False)
    assert C.rel_err(torch.log_softmax(pred.mean_logits(x).double(), 1), mean_ref) < 1e-5


def test_auto_selection(lb):
    net = lb.BayesianNetwork().cuda().eval()
    p = lb.EnsemblePredictor(net, batch=16, samples_per_launch=3, seed=2)
    assert p.tc == [False, False, False]
    p.run(torch.rand(16, 784, device="cuda"), 3)
    assert p.kernels_per_launch == 1 + 3 * 2 + 2                 # today's CUDA-core launch sequence
    wide = _wide_net(lb, (4096, 4096, 4096, 10), 4)
    p = lb.EnsemblePredictor(wide, batch=16, samples_per_launch=3, seed=2)
    assert p.tc == [True, True, False]
    p.run(torch.rand(16, 4096, device="cuda"), 3)
    assert p.kernels_per_launch == 1 + 3 + 3 + 2
    # a CUDA-core layer feeding a tensor-core one: its activations are split for the next layer's GEMMs
    mixed = _wide_net(lb, (784, 1024, 1024, 10), 5)
    p = lb.EnsemblePredictor(mixed, batch=16, samples_per_launch=3, seed=2)
    q = lb.EnsemblePredictor(mixed, batch=16, samples_per_launch=3, seed=2, gemm="simt")
    assert p.tc == [False, True, False]
    xm = torch.rand(16, 784, device="cuda")
    p.run(xm, 3)
    q.run(xm, 3)
    assert p.kernels_per_launch == 1 + 1 + 3 + 3 + 2
    assert C.rel_err(p.sum_logp, q.sum_logp) < 1e-5
    with pytest.raises(ValueError):
        lb.EnsemblePredictor(net, batch=16, gemm="bf16")
