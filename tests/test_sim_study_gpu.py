"""GPU tests of the one-launch simulation-study trainer (lbbnn.mf.SimStudyEnsemble, csrc/mf_sim.cu): the trajectory of
every replica against the float64 oracle, the relaxed-gamma gradient against the eager module path, native-noise
determinism, the standard-Gamma sampler and the `.exact` launch flags."""
import copy

import numpy as np
import pytest
import torch

import cases as C
import lbbnn_oracle as O

pytestmark = pytest.mark.gpu
NAMES = ("weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho", "weight_a", "weight_b", "bias_a", "bias_b", "pa", "pb")


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def _net(lb, p):
    net = lb.mf.SimStudyNetwork().cuda()
    with torch.no_grad():
        for k, v in p.items():
            getattr(net.l1, k).copy_(v)
    return net


def _replica_cases(R, steps):
    """R sim_study_case draws with weight_a / bias_a spread over [0.3, 3] (both branches of standard_gamma_grad) and the last
    replica started near the true weights (saturated logits)."""
    spread = np.linspace(0.3, 3.0, R)
    cs = []
    for r in range(R):
        c = C.sim_study_case(seed=200 + r, steps=steps)
        rng = np.random.default_rng(300 + r)
        c["p"]["weight_a"] = torch.tensor([spread[r]], dtype=torch.float32)
        c["p"]["bias_a"] = torch.tensor([spread[R - 1 - r]], dtype=torch.float32)
        for nz in c["noises"]:
            nz["g0_w"] = C.t(rng.gamma(spread[r], size=(1,)))
            nz["g0_b"] = C.t(rng.gamma(spread[R - 1 - r], size=(1,)))
        cs.append(c)
    near = cs[-1]["p"]
    near["weight_mu"] = C.t(C.SIM_TRUE_WEIGHTS[None, :] + 0.01 * np.random.default_rng(7).standard_normal((1, 20)))
    # a broad Gamma prior on the weights' precision: at weight_b ~ 1 the prior term tau * sum ws^2 (~4100 at the true
    # weights) drives weight_a below zero within ten SGD steps, in float64 too, and every gradient after that is NaN
    near["weight_b"] = torch.tensor([100.0], dtype=torch.float32)
    return cs


def _stack_noise(cs, key):
    return torch.stack([torch.stack([nz[key].reshape(-1) for nz in c["noises"]]) for c in cs]).squeeze(-1).cuda()


def test_trajectory_of_every_replica_matches_float64(lb):
    R, E = 6, 2
    cs = _replica_cases(R, steps=10)
    B, nb = cs[0]["batch"], cs[0]["num_batches"]
    steps = E * int(nb)
    gam = torch.stack([torch.stack([O.relaxed_bernoulli_rsample(O.alpha_of(c["p"]["lambdal"]), u).reshape(-1) for u in c["us"]])
                       for c in cs])                                             # constant masks, (R, steps, in)
    # the replica near the true weights keeps every weight, so its logits are the data's own (|logit| up to ~200) and saturate
    # where the labels agree with them.  With masked weights the logits saturate against the labels too: torch's fp32 BCE then
    # clamps log(1 - p) at -100 once p rounds to 1, where float64 keeps -logit (measured: nll 337.8 against 181.3 at step 0)
    gam[-1] = 1.0
    assert (torch.sigmoid(cs[-1]["X"] @ cs[-1]["p"]["weight_mu"].reshape(-1)) == 1.0).sum() > 100
    noise = {"eps_w": _stack_noise(cs, "eps_w"), "eps_b": _stack_noise(cs, "eps_b"), "g0_w": _stack_noise(cs, "g0_w"),
             "g0_b": _stack_noise(cs, "g0_b"), "gamma": gam.cuda()}
    nets = [_net(lb, c["p"]) for c in cs]
    X = torch.stack([c["X"] for c in cs]).cuda()
    y = torch.stack([c["y"] for c in cs]).cuda()
    ens = lb.mf.SimStudyEnsemble(nets, X, y, batch_size=B)
    stats = ens.run(E, noise=noise).cpu()
    torch.cuda.synchronize()
    lrs = lb.mf.SIM_STUDY_LRS
    for r, c in enumerate(cs):
        ref = {k: v.double().clone().requires_grad_(True) for k, v in c["p"].items()}
        opt = torch.optim.SGD([{"params": [ref[k]], "lr": lrs[k]} for k in NAMES], lr=0.01)
        for s in range(steps):
            k = s % int(nb)
            xb, yb = c["X"][k * B:(k + 1) * B].double(), c["y"][k * B:(k + 1) * B]
            nz = {n: v.double() for n, v in c["noises"][s].items()}
            opt.zero_grad()
            loss, nll, lp, lq, _ = O.mfsim_elbo(xb, yb, ref, nz, None, nb, gamma=gam[r, s].reshape(1, -1).double())
            loss.backward()
            for got, want in zip(stats[r, s], (loss, nll, lp, lq)):
                assert abs(got.item() - want.item()) <= 2e-5 * abs(want.item()) + 1e-4, (r, s, stats[r, s], loss, nll, lp, lq)
            if s < steps - 1:
                opt.step()
        for name in NAMES:
            got = getattr(nets[r].l1, name).grad
            if name in ("pa", "pb"):
                # n gp (psi(pa + pb) - psi(1 + pa + pb) - psi(pa | pb)) cancels to ~1e-3 from O(1) digamma terms: fp32 reaches it
                # to 5e-5 of those terms (measured 1.4e-4 of the result for pa, the same in the layer kernels), not of the result
                pa, pb = ref["pa"].detach(), ref["pb"].detach()
                scale = 20 / nb * (torch.digamma(pa + pb).abs() + torch.digamma(1 + pa + pb).abs()
                                   + torch.digamma(pa if name == "pa" else pb).abs())
                assert (got.double().cpu() - ref[name].grad).abs().item() < 5e-5 * scale.item(), (r, name)
            else:
                assert C.rel_err(got, ref[name].grad) < 5e-5, (r, name)
        opt.step()
        for name in NAMES:
            assert C.rel_err(getattr(nets[r].l1, name).data, ref[name].data) < 1e-6, (r, name)
        alpha_ref = O.alpha_of(ref["lambdal"].detach()).reshape(-1)
        assert torch.equal(ens.inclusion_probabilities()[r].cpu() > 0.5, alpha_ref > 0.5)


def test_relaxed_gamma_gradient_matches_the_eager_module(lb):
    R, n, B = 2, 1200, 400
    steps = n // B
    cs = [C.sim_study_case(seed=400 + r, n=n, batch=B, steps=steps) for r in range(R)]
    nets = [_net(lb, c["p"]) for c in cs]
    eager = [copy.deepcopy(m) for m in nets]
    for m in nets + eager:
        m.num_batches = n / B
    X = torch.stack([c["X"] for c in cs]).cuda()
    y = torch.stack([c["y"] for c in cs]).cuda()
    noise = {k: _stack_noise(cs, k) for k in ("eps_w", "eps_b", "g0_w", "g0_b")}
    noise["u"] = torch.stack([torch.stack([u.reshape(-1) for u in c["us"]]) for c in cs]).cuda()
    ens = lb.mf.SimStudyEnsemble(nets, X, y, batch_size=B)
    stats = ens.run(1, noise=noise)
    lrs = lb.mf.SIM_STUDY_LRS
    for r, (m, c) in enumerate(zip(eager, cs)):
        m.train()
        opt = torch.optim.SGD([{"params": [getattr(m.l1, k)], "lr": lrs[k]} for k in NAMES], lr=0.01)
        for s in range(steps):
            opt.zero_grad()
            nz = {k: v.cuda() for k, v in c["noises"][s].items()}
            loss, lp, lq, nll, _ = m.sample_elbo(X[r, s * B:(s + 1) * B], y[r, s * B:(s + 1) * B], noises=[nz],
                                                 us=[c["us"][s].cuda()])
            loss.backward()
            for got, want in zip(stats[r, s].tolist(), (loss.item(), nll.item(), lp.item(), lq.item())):
                assert abs(got - want) <= 1e-5 * abs(want) + 1e-5, (r, s, stats[r, s], loss, nll, lp, lq)
            opt.step()
        for name in NAMES:
            assert C.rel_err(getattr(nets[r].l1, name).data, getattr(m.l1, name).data) < 1e-5, (r, name)
    assert nets[0].l1.lambdal.grad.abs().max() > 0


def test_exact_gamma_draws_the_hard_mask(lb):
    """gamma.exact: the mask is [u < alpha] bit for bit -- the one-step objective equals the float64 oracle fed that mask, and
    a mask with a single flipped bit would move the Bernoulli log q by |log(alpha / (1 - alpha))| >> the bound."""
    c = C.sim_study_case(seed=500, n=400, batch=400, steps=1)
    c["p"]["lambdal"] = C.t(np.random.default_rng(1).uniform(-3, 3, size=(1, 20)))
    net = _net(lb, c["p"])
    net.num_batches = 1.0
    net.l1.gamma.exact = True
    noise = {k: _stack_noise([c], k).reshape(1, 1, -1) if k == "eps_w" else _stack_noise([c], k).reshape(1, 1)
             for k in ("eps_w", "eps_b", "g0_w", "g0_b")}
    noise["u"] = c["us"][0].reshape(1, 1, -1).cuda()
    lam = net.l1.lambdal.detach().clone()
    ens = lb.mf.SimStudyEnsemble([net], c["X"].cuda(), c["y"].cuda(), batch_size=400)
    stats = ens.run(1, noise=noise).cpu()[0, 0]
    mask = (noise["u"].reshape(1, -1) < 1.0 / (1.0 + torch.exp(-lam))).double().cpu()
    ref = {k: v.double() for k, v in c["p"].items()}
    loss, nll, lp, lq, _ = O.mfsim_elbo(c["X"].double(), c["y"], ref, {k: v.double() for k, v in c["noises"][0].items()},
                                        None, 1.0, gamma_exact=True, gamma=mask)
    for got, want in zip(stats.tolist(), (loss.item(), nll.item(), lp.item(), lq.item())):
        assert abs(got - want) <= 2e-5 * abs(want) + 1e-4, (stats, loss, nll, lp, lq)


def _native(lb, R, seed=3, X=None, y=None, n=800):
    cs = [C.sim_study_case(seed=600 + r, n=n, steps=1) for r in range(R)]
    X = cs[0]["X"].cuda() if X is None else X
    y = cs[0]["y"].cuda() if y is None else y
    return lb.mf.SimStudyEnsemble([_net(lb, c["p"]) for c in cs], X, y, batch_size=400, seed=seed)


def test_native_noise_is_keyed_by_replica_and_step(lb):
    a, b = _native(lb, 3), _native(lb, 3)
    sa = a.run(4)
    sb = torch.cat([b.run(2), b.run(2)], dim=1)
    assert torch.equal(sa, sb) and torch.equal(a.flat, b.flat) and torch.equal(a.step, b.step)
    assert torch.isfinite(sa).all() and not torch.equal(sa[0], sa[1])
    big = _native(lb, 16)
    one = _native(lb, 1)
    assert torch.equal(big.flat[0], one.flat[0])
    assert torch.equal(big.run(2)[0], one.run(2)[0]) and torch.equal(big.flat[0], one.flat[0])


@pytest.mark.parametrize("R", [1, 7, 148, 300])
def test_any_number_of_replicas_runs(lb, R):
    ens = _native(lb, R)
    stats = ens.run(3)
    assert stats.shape == (R, 3 * 2, 4) and torch.isfinite(stats).all() and torch.isfinite(ens.flat).all()
    assert torch.equal(ens.step, torch.full((R,), 6, dtype=torch.int64, device="cuda"))


def test_shared_data_equals_the_same_data_per_replica(lb):
    c = C.sim_study_case(seed=700, n=800, steps=1)
    X, y = c["X"].cuda(), c["y"].cuda()
    a = _native(lb, 4, X=X, y=y)
    b = _native(lb, 4, X=X.expand(4, -1, -1).contiguous(), y=y.expand(4, -1).contiguous())
    assert torch.equal(a.run(2), b.run(2)) and torch.equal(a.flat, b.flat)


@pytest.mark.parametrize("a", [0.3, 1.05, 4.0])
def test_std_gamma_sampler_distribution(lb, a):
    from scipy import stats as S
    n = 200_000
    g = lb._capi.philox_std_gamma(a, n, seed=11, stream_id=5).double().cpu().numpy()
    assert np.isfinite(g).all() and (g >= 0).all()
    assert S.kstest(g, S.gamma(a).cdf).pvalue > 1e-3
    assert abs(g.mean() - a) < 4 * np.sqrt(a / n)
    assert abs(g.var() - a) < 4 * np.sqrt((2 * a * a + 6 * a) / n)
    again = lb._capi.philox_std_gamma(a, 1000, seed=11, stream_id=5).double().cpu().numpy()
    assert np.array_equal(again, g[:1000])


def test_exact_prior_flags_are_read_at_every_run(lb):
    c = C.sim_study_case(seed=800, n=400, batch=400, steps=1)
    net = _net(lb, c["p"])
    ens = lb.mf.SimStudyEnsemble([net], c["X"].cuda(), c["y"].cuda(), batch_size=400)
    ens.run(1)                                                   # relaxed priors
    gam = torch.from_numpy(np.random.default_rng(2).uniform(0.2, 0.8, size=(1, 20))).float()   # rounding matters
    noise = {k: _stack_noise([c], k).reshape(1, 1, -1) if k == "eps_w" else _stack_noise([c], k).reshape(1, 1)
             for k in ("eps_w", "eps_b", "g0_w", "g0_b")}
    noise["gamma"] = gam.reshape(1, 1, -1).cuda()
    p = {k: getattr(net.l1, k).detach().double().cpu() for k in NAMES}
    nz = {k: v.double() for k, v in c["noises"][0].items()}
    ref = {}
    for exact in (False, True):
        _, ref[exact], _ = O.mf_forward(c["X"].double(), p, gam.double(), nz, exact=(False, exact, False, exact),
                                        logprob_on_ws=True)
    assert abs(ref[True].item() - ref[False].item()) > 0.1           # >> the bound below
    net.l1.weight_prior.exact = True
    net.l1.gamma_prior.exact = True
    lp = ens.run(1, noise=noise)[0, 0, 2].item()
    assert abs(lp - ref[True].item()) <= 2e-5 * abs(ref[True].item()) + 1e-4, (lp, ref)


def test_mixed_flags_are_rejected(lb):
    ens = _native(lb, 2)
    ens.layers[1].gamma_prior.exact = True
    with pytest.raises(lb.LbbnnError):
        ens.run(1)
