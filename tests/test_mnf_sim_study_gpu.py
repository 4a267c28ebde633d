"""GPU tests of the one-launch MNF simulation-study trainer (lbbnn.mnf.SimStudyEnsemble, csrc/mnf_sim.cu): every replica's
trajectory (stats, last-step gradients, parameters, both Adam moments) against float64 autograd of the oracle's MNF layer
with a float64 Adam, one replica against the eager module + torch.optim.Adam, native-noise reproduction and determinism,
staged learning rates and the .grad views."""
import copy

import numpy as np
import pytest
import torch

import cases as C
import lbbnn_oracle as O
from mnf_sim_ref import mnfsim_loss

pytestmark = pytest.mark.gpu
IN, T, H = 20, 2, (50,) * 5
PRIORS = O.Priors(mu=0.1, sigma=1.3, alpha=0.3, bias_mu=0.0, bias_sigma=1.3)
F32 = lambda v: float(np.float32(v))  # noqa: E731  (the hyperparameters as the kernel receives them)
FLOW_GRAD_BOUND, LAYER_GRAD_BOUND = 5e-5, 1e-5
# Parameters after Adam.  Adam's update lr m^ / (sqrt(v^) + eps) is scale-free per element: an fp32 gradient error of
# GRAD_ERR max|g| (a fraction of the gradient bounds above) changes an element's update by about lr GRAD_ERR max|g| / |g_i|,
# whatever the element's own size -- +-lr at its first nonzero step when g_i is at the rounding level.  So element i is held
# to 2e-6 max|p| plus its own allowance min(ADAM_CAP lr, sum_t lr_t s_i(t)), s_i(t) = min(1, GRAD_ERR max|g_t| / |g_i,t'|)
# at its smallest nonzero gradient up to step t (0 before its first nonzero gradient: elements whose gradient is exactly 0
# throughout, masked conditioner inputs, stay at 2e-6 max|p|).  For an element with |g_i| ~ max|g| the allowance is
# ~1e-5 lr per step; ADAM_CAP keeps every element far inside Adam's own travel.  Each check prints how many elements use it.
GRAD_ERR, ADAM_CAP = 1e-5, 0.05


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def _params(seed, D=IN, T=T, H=H):
    """Sim-study layer parameters with a q0 wide enough for the flows to matter (as tests/cases.py: mnf_layer_case)."""
    rng = np.random.default_rng(seed)
    p = O.init_mnf_params(rng, D, 1, T, H)
    p["lambdal"] = C.t(rng.uniform(1.5, 2.5, size=(1, D)))
    p["q0_log_var"] = C.t(-2.0 + 0.3 * rng.standard_normal(size=(D,)))
    p["q0_mean"] = C.t(1.0 + 0.1 * rng.standard_normal(size=(D,)))
    return p


def _net(lb, p, num_batches):
    D, T, H = p["weight_mu"].shape[1], len(p["z_flow"]), tuple(w.shape[0] for w, _ in p["z_flow"][0]["net"])
    net = lb.mnf.SimStudyNetwork(in_features=D, num_batches=num_batches, num_transforms=T, h_sizes=H).cuda()
    with torch.no_grad():
        for k, v in C.flat_named(p).items():
            net.l1.get_parameter(k).copy_(v)
    return net


def _noise(seed, R, steps, B, IN=IN, T=T):
    rng = np.random.default_rng(seed)
    n = lambda *s: torch.from_numpy(rng.standard_normal(size=s)).float()        # noqa: E731
    m = lambda *s: torch.from_numpy((rng.uniform(size=s) < 0.5).astype(np.float32))  # noqa: E731
    return {"eps_z": n(R, steps, IN), "eps_z2": n(R, steps, IN), "z_masks": m(R, steps, T, IN), "z_masks2": m(R, steps, T, IN),
            "r_masks": m(R, steps, T, IN), "eps": n(R, steps, B), "eps_r": n(R, steps)}


def _oracle_noise(nz, r, s, dtype=torch.float64):
    IN, T = nz["eps_z"].shape[-1], nz["z_masks"].shape[2]
    c = lambda k: nz[k][r, s].to(dtype)  # noqa: E731
    return {"eps_z": c("eps_z").reshape(1, IN), "z_masks": [c("z_masks")[t].reshape(1, IN) for t in range(T)],
            "eps": c("eps").reshape(-1, 1), "eps_z2": c("eps_z2").reshape(1, IN),
            "z_masks2": [c("z_masks2")[t].reshape(1, IN) for t in range(T)], "eps_r": c("eps_r").reshape(1),
            "r_masks": [c("r_masks")[t].reshape(IN) for t in range(T)]}


def _group_of(name):
    return name.split(".")[0] if name.startswith(("z_flow", "r_flow")) else name


class _Ref:
    """float64 autograd of mnfsim_loss + torch.optim.Adam's update in float64 with the kernel's fp32 hyperparameters."""

    def __init__(self, p):
        self.p = p
        self.named = {k: v.double().clone().requires_grad_(True) for k, v in C.flat_named(p).items()}
        self.m = {k: torch.zeros_like(v) for k, v in self.named.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.named.items()}
        self.t = 0
        self.lr_max = {k: 0.0 for k in self.named}
        self.sens = {k: torch.zeros_like(v) for k, v in self.named.items()}        # s_i(t), see GRAD_ERR
        self.allow = {k: torch.zeros_like(v) for k, v in self.named.items()}       # sum_t lr_t s_i(t)

    def step(self, x, y, nz, num_batches, lrs):
        for v in self.named.values():
            v.grad = None
        loss, nll, kl, _ = mnfsim_loss(x.double(), y.double(), C.unflatten_like(self.p, self.named), nz, num_batches, PRIORS)
        loss.backward()
        grads = {k: v.grad.detach().clone() for k, v in self.named.items()}
        self.t += 1
        b1, b2, eps = F32(0.9), F32(0.999), F32(1e-8)
        bc1, bc2 = 1 - b1 ** self.t, 1 - b2 ** self.t
        with torch.no_grad():
            for k, v in self.named.items():
                g = grads[k]
                lr = F32(lrs[_group_of(k)])
                self.lr_max[k] = max(self.lr_max[k], lr)
                nz = g != 0
                s_now = torch.where(nz, (GRAD_ERR * g.abs().max() / g.abs().clamp_min(1e-300)).clamp(max=1.0), torch.zeros_like(g))
                self.sens[k] = torch.maximum(self.sens[k], s_now)
                self.allow[k] += lr * self.sens[k]
                self.m[k] += (1 - b1) * (g - self.m[k])
                self.v[k] = b2 * self.v[k] + (1 - b2) * g * g
                v -= F32(lrs[_group_of(k)]) / bc1 * self.m[k] / (self.v[k].sqrt() / bc2 ** 0.5 + eps)
        return (loss.item(), nll.item(), kl.item()), grads


def _packed_names(net):
    """Parameter names of net.l1 in the packed row order, with their (offset, numel)."""
    l1 = net.l1
    ids = {id(p): n for n, p in l1.named_parameters()}
    out, o = [], 0
    for p in [getattr(l1, k) for k in lb_layer_names()] + l1.z_flow._params() + l1.r_flow._params():
        out.append((ids[id(p)], o, p.numel()))
        o += p.numel()
    return out


def lb_layer_names():
    import lbbnn
    return lbbnn.mnf.SIM_LAYER_NAMES


def _lrs(lb, scale=1.0):
    return {g: scale * 1e-3 * (1 + 0.1 * i) for i, g in enumerate(lb.mnf.SIM_GROUPS)}


def _check_replica(ens, net, r, ref, grads, tag):
    """The last step's gradients (.grad views), the parameters and both Adam moments of replica r against the reference."""
    errs, nused, worst = {}, 0, 0.0
    for name, o, k in _packed_names(net):
        flow = name.startswith(("z_flow", "r_flow"))
        p = net.l1.get_parameter(name)
        ge = C.rel_err(p.grad, grads[name])
        errs[name] = ge
        assert ge < (FLOW_GRAD_BOUND if flow or name.startswith("q0") else LAYER_GRAD_BOUND), (tag, r, name, ge)
        want = ref.named[name].detach()
        dp = (p.data.double().cpu() - want).abs()
        base = 2e-6 * want.abs().max()
        allow = ref.allow[name].clamp(max=ADAM_CAP * ref.lr_max[name])
        over = dp - base
        assert (over <= allow).all(), (tag, r, name, int((over > allow).sum()), over.max().item(), allow[over > allow][:4].tolist())
        used = over > 0
        nused += int(used.sum())
        worst = max(worst, (over[used] / allow[used]).max().item() if used.any() else 0.0)
        assert C.rel_err(ens.exp_avg[r, o:o + k], ref.m[name].reshape(-1)) < FLOW_GRAD_BOUND, (tag, r, name)
        assert C.rel_err(ens.exp_avg_sq[r, o:o + k], ref.v[name].reshape(-1)) < 2 * FLOW_GRAD_BOUND, (tag, r, name)
    print(f"[{tag} r={r}] largest gradient error: layer {max(v for n, v in errs.items() if '.' not in n):.2e}, "
          f"flows {max(v for n, v in errs.items() if '.' in n):.2e}; {nused} parameters past 2e-6 max|p|, "
          f"using at most {worst:.2f} of their Adam allowance")
    return errs


@pytest.mark.parametrize("data", ["shared", "per_replica"])
def test_trajectory_of_every_replica_matches_float64(lb, data):
    R, n, B, E = 4, 800, 400, 5
    steps, nb = E * n // B, n / B
    cases = [C.sim_study_case(seed=900 + r, n=n, batch=B, steps=1) for r in range(R)]
    X = cases[0]["X"] if data == "shared" else torch.stack([c["X"] for c in cases])
    y = cases[0]["y"] if data == "shared" else torch.stack([c["y"] for c in cases])
    ps = [_params(50 + r) for r in range(R)]
    nets = [_net(lb, p, nb) for p in ps]
    lrs = _lrs(lb)
    nz = _noise(7, R, steps, B)
    ens = lb.mnf.SimStudyEnsemble(nets, X.cuda(), y.cuda(), batch_size=B, lrs=lrs)
    stats = ens.run(E, noise={k: v.cuda() for k, v in nz.items()}).cpu()
    worst = 0.0
    for r in range(R):
        ref = _Ref(ps[r])
        Xr, yr = (X if data == "shared" else X[r]), (y if data == "shared" else y[r])
        for s in range(steps):
            k = s % int(nb)
            want, grads = ref.step(Xr[k * B:(k + 1) * B], yr[k * B:(k + 1) * B], _oracle_noise(nz, r, s), nb, lrs)
            for got, w in zip(stats[r, s].tolist(), want):
                worst = max(worst, abs(got - w) / max(abs(w), 1.0))
                assert abs(got - w) <= 1e-5 * max(abs(w), 1.0), (r, s, stats[r, s], want)
        _check_replica(ens, nets[r], r, ref, grads, data)
    assert torch.equal(ens.step.cpu(), torch.full((R,), steps, dtype=torch.int64))
    alpha = ens.inclusion_probabilities()
    assert torch.equal(alpha, torch.sigmoid(ens.flat[:, 2 * IN:3 * IN])) or C.rel_err(alpha, torch.sigmoid(ens.flat[:, 2 * IN:3 * IN])) < 1e-6


def test_staged_learning_rates_match_float64(lb):
    R, n, B = 2, 800, 400
    nb = n / B
    c = C.sim_study_case(seed=950, n=n, batch=B, steps=1)
    ps = [_params(70 + r) for r in range(R)]
    nets = [_net(lb, p, nb) for p in ps]
    A, Bl = _lrs(lb), _lrs(lb, 0.3)
    ens = lb.mnf.SimStudyEnsemble(nets, c["X"].cuda(), c["y"].cuda(), batch_size=B, lrs=0.5)
    nz1, nz2 = _noise(11, R, 4, B), _noise(12, R, 2, B)
    s1 = ens.run(2, lrs=A, noise={k: v.cuda() for k, v in nz1.items()}).cpu()
    s2 = ens.run(1, lrs=Bl, noise={k: v.cuda() for k, v in nz2.items()}).cpu()
    assert ens.lrs == [Bl[g] for g in lb.mnf.SIM_GROUPS]
    for r in range(R):
        ref = _Ref(ps[r])
        for stats, nz, lrs, steps in ((s1, nz1, A, 4), (s2, nz2, Bl, 2)):
            for s in range(steps):
                k = s % int(nb)
                want, grads = ref.step(c["X"][k * B:(k + 1) * B], c["y"][k * B:(k + 1) * B], _oracle_noise(nz, r, s), nb, lrs)
                for got, w in zip(stats[r, s].tolist(), want):
                    assert abs(got - w) <= 1e-5 * max(abs(w), 1.0), (r, s, stats[r, s], want)
        _check_replica(ens, nets[r], r, ref, grads, "staged")


def test_one_replica_matches_the_eager_module_and_torch_adam(lb):
    n, B, E = 800, 400, 2
    steps, nb = E * n // B, n / B
    c = C.sim_study_case(seed=960, n=n, batch=B, steps=1)
    net = _net(lb, _params(80), nb)
    eager = copy.deepcopy(net)
    lrs = _lrs(lb)
    nz = _noise(13, 1, steps, B)
    X, y = c["X"].cuda(), c["y"].cuda()
    ens = lb.mnf.SimStudyEnsemble([net], X, y, batch_size=B, lrs=lrs)
    stats = ens.run(E, noise={k: v.cuda() for k, v in nz.items()}).cpu()
    ref = _Ref(_params(80))
    l1 = eager.l1
    groups = [{"params": [getattr(l1, k)], "lr": F32(lrs[k])} for k in lb.mnf.SIM_LAYER_NAMES]
    groups += [{"params": list(l1.z_flow.parameters()), "lr": F32(lrs["z_flow"])},
               {"params": list(l1.r_flow.parameters()), "lr": F32(lrs["r_flow"])}]
    opt = torch.optim.Adam(groups)
    for s in range(steps):
        k = s % int(nb)
        opt.zero_grad()
        noise = {key: (v.cuda() if torch.is_tensor(v) else [m.cuda() for m in v])
                 for key, v in _oracle_noise(nz, 0, s, torch.float32).items()}
        loss, nll, kl = eager.loss(X[k * B:(k + 1) * B], y[k * B:(k + 1) * B], noise=noise)
        loss.backward()
        ref.step(c["X"][k * B:(k + 1) * B], c["y"][k * B:(k + 1) * B], _oracle_noise(nz, 0, s), nb, lrs)
        for got, w in zip(stats[0, s].tolist(), (loss.item(), nll.item(), kl.item())):
            assert abs(got - w) <= 1e-5 * max(abs(w), 1.0), (s, stats[0, s], loss, nll, kl)
        if s < steps - 1:
            opt.step()
    for name, p in eager.l1.named_parameters():
        bound = FLOW_GRAD_BOUND if name.startswith(("z_flow", "r_flow", "q0")) else LAYER_GRAD_BOUND
        assert C.rel_err(net.l1.get_parameter(name).grad, p.grad) < 2 * bound, name
    opt.step()
    nused = 0
    for name, p in eager.l1.named_parameters():
        # both sides are fp32, each within the float64 bound: twice the base bound and twice the Adam allowance (GRAD_ERR)
        dp = (net.l1.get_parameter(name).data - p.data).abs().double().cpu()
        over = dp - 4e-6 * p.data.abs().max().item()
        allow = 2 * ref.allow[name].clamp(max=ADAM_CAP * ref.lr_max[name])
        assert (over <= allow).all(), (name, int((over > allow).sum()), over.max().item())
        nused += int((over > 0).sum())
    print(f"[eager] {nused} parameters past 4e-6 max|p|")


@pytest.mark.parametrize("D, T_, H_", [(32, 4, (64, 8, 64, 8, 64, 8)), (7, 1, (3,))])
def test_trajectory_at_the_kernel_limits_matches_float64(lb, D, T_, H_):
    """in = 32 (a full warp in phase 3) and T = 4, six hidden layers of mixed widths up to 64; and a small odd shape."""
    R, n, B, E = 2, 600, 200, 2
    steps, nb = E * n // B, n / B
    rng = np.random.default_rng(990 + D)
    X = torch.from_numpy(rng.standard_normal(size=(n, D))).float()
    y = torch.from_numpy((rng.uniform(size=n) < 1 / (1 + np.exp(-X.numpy() @ rng.normal(0, 1, D)))).astype(np.float32))
    ps = [_params(60 + r, D, T_, H_) for r in range(R)]
    nets = [_net(lb, p, nb) for p in ps]
    lrs = _lrs(lb)
    nz = _noise(17, R, steps, B, D, T_)
    ens = lb.mnf.SimStudyEnsemble(nets, X.cuda(), y.cuda(), batch_size=B, lrs=lrs)
    stats = ens.run(E, noise={k: v.cuda() for k, v in nz.items()}).cpu()
    for r in range(R):
        ref = _Ref(ps[r])
        for s in range(steps):
            k = s % int(nb)
            want, grads = ref.step(X[k * B:(k + 1) * B], y[k * B:(k + 1) * B], _oracle_noise(nz, r, s), nb, lrs)
            for got, w in zip(stats[r, s].tolist(), want):
                assert abs(got - w) <= 1e-5 * max(abs(w), 1.0), (r, s, stats[r, s], want)
        _check_replica(ens, nets[r], r, ref, grads, f"limits D={D}")


STREAM = lambda r, s, kind: (r << 40) | (s << 4) | kind  # noqa: E731


def _native(lb, R, seed=5, n=800, nets=None):
    c = C.sim_study_case(seed=970, n=n, batch=400, steps=1)
    nets = nets or [_net(lb, _params(100 + r), n / 400) for r in range(R)]
    return lb.mnf.SimStudyEnsemble(nets, c["X"].cuda(), c["y"].cuda(), batch_size=400, lrs=1e-3, seed=seed)


def test_native_draws_are_the_documented_philox_streams(lb):
    """Replica r's draws of step s, rebuilt with lbbnn_philox_normal / _uniform from the streams include/lbbnn.h documents and
    injected, give the native run bit for bit (and the injected path is held to float64 by the trajectory tests)."""
    K = lb._capi
    R, E, seed = 3, 2, 5
    a = _native(lb, R, seed)
    b = _native(lb, R, seed)
    a.run(1)
    b.run(1)                                              # start at step 2: the step key is the replica's own count
    steps = E * 2
    nz = {k: [] for k in ("eps_z", "eps_z2", "z_masks", "z_masks2", "r_masks", "eps", "eps_r")}
    for r in range(R):
        rows = {k: [] for k in nz}
        for s in range(2, 2 + steps):
            st = lambda kind: STREAM(r, s, kind)  # noqa: E731
            mask = lambda base: torch.stack([K.philox_uniform((IN,), seed, st(base + t)) < 0.5 for t in range(T)]).float()  # noqa: E731
            rows["eps_z"].append(K.philox_normal((IN,), seed, st(K.MNFSIM_DRAW_EPS_Z)))
            rows["eps_z2"].append(K.philox_normal((IN,), seed, st(K.MNFSIM_DRAW_EPS_Z2)))
            rows["eps"].append(K.philox_normal((400,), seed, st(K.MNFSIM_DRAW_EPS)))
            rows["eps_r"].append(K.philox_normal((4,), seed, st(K.MNFSIM_DRAW_EPS_R))[0])
            rows["z_masks"].append(mask(K.MNFSIM_DRAW_Z_MASK))
            rows["z_masks2"].append(mask(K.MNFSIM_DRAW_Z_MASK2))
            rows["r_masks"].append(mask(K.MNFSIM_DRAW_R_MASK))
        for k in nz:
            nz[k].append(torch.stack(rows[k]))
    nz = {k: torch.stack(v) for k, v in nz.items()}
    sa = a.run(E)
    sb = b.run(E, noise=nz)
    assert torch.equal(sa, sb) and torch.equal(a.flat, b.flat) and torch.equal(a.exp_avg_sq, b.exp_avg_sq)
    assert torch.equal(a.grads, b.grads)


def test_native_noise_is_deterministic_and_keyed_by_replica_and_step(lb):
    a, b = _native(lb, 3), _native(lb, 3)
    sa = a.run(4)
    sb = torch.cat([b.run(2), b.run(2)], dim=1)
    assert torch.equal(sa, sb) and torch.equal(a.flat, b.flat) and torch.equal(a.exp_avg, b.exp_avg)
    assert torch.equal(a.exp_avg_sq, b.exp_avg_sq) and torch.equal(a.step, b.step)
    assert torch.isfinite(sa).all() and not torch.equal(sa[0], sa[1])
    c, d = _native(lb, 3), _native(lb, 3)
    assert torch.equal(c.run(2), d.run(2)) and torch.equal(c.flat, d.flat)       # two launches, bit for bit


def test_replica_draws_do_not_depend_on_the_number_of_replicas(lb):
    one = _native(lb, 1)
    net0 = one.nets[0]
    nets = [_net(lb, _params(100), 2.0)] + [_net(lb, _params(200 + r), 2.0) for r in range(299)]
    big = _native(lb, 300, nets=nets)
    assert torch.equal(big.flat[0], one.flat[0])
    assert torch.equal(big.run(2)[0], one.run(2)[0]) and torch.equal(big.flat[0], one.flat[0])
    assert torch.equal(big.exp_avg[0], one.exp_avg[0]) and net0.l1.weight_mu.data_ptr() == one.flat.data_ptr()


@pytest.mark.parametrize("R", [1, 7, 148])
def test_any_number_of_replicas_runs(lb, R):
    ens = _native(lb, R)
    stats = ens.run(3)
    assert stats.shape == (R, 6, 3) and torch.isfinite(stats).all() and torch.isfinite(ens.flat).all()
    assert torch.equal(ens.step, torch.full((R,), 6, dtype=torch.int64, device="cuda"))


def test_grad_views_hold_the_last_step_gradients(lb):
    ens = _native(lb, 2)
    ens.run(1)
    for r, net in enumerate(ens.nets):
        for name, o, k in _packed_names(net):
            p = net.l1.get_parameter(name)
            assert torch.equal(p.grad.reshape(-1), ens.grads[r, o:o + k]) and p.data_ptr() == ens.flat[r, o:].data_ptr()
    assert ens.grads[:, :2 * IN].abs().max() > 0
    lean = lb.mnf.SimStudyEnsemble([_net(lb, _params(100), 2.0)], ens.X, ens.y, lrs=1e-3, seed=5, materialize_grads=False)
    full = _native(lb, 1)
    assert lean.grads is None and torch.equal(lean.run(2), full.run(2)) and torch.equal(lean.flat, full.flat)
    state = ens.nets[0].state_dict()
    assert torch.equal(state["l1.weight_mu"].reshape(-1), ens.flat[0, :IN])
