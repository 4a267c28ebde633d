"""Drop-in LRT layer and network (reference: LBBNN-GP-MF-LRT.py:129-214).

Same constructor, parameter names (= state_dict keys), `forward(input, sample, calculate_log_probs)`
signature and side-effect attributes (`.kl`, `.alpha_q`, `.gamma`, `.weight`, `.bias`) as the
reference's `BayesianLinear` / `BayesianNetwork`; what the reference reads from module globals
(DEVICE, priors) are keyword arguments with the reference's values as defaults.  The compute is the
fused sm_100a kernels of liblbbnn behind a torch.autograd.Function -- CUDA tensors only.
"""
import itertools

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi as K

_seed = 0x5EEDBA5E
_layer_ids = itertools.count(1)


def manual_seed(seed):
    """Seed of the native Philox noise (the eps of LRT:174 when none is injected)."""
    global _seed
    _seed = int(seed)


def current_seed():
    return _seed


class LayerConfig:
    """Per-layer constants the reference keeps as module-level tensors/globals."""

    def __init__(self, mu_prior=0.0, sigma_prior=1.0, alpha_prior=0.05, bias_mu_prior=0.0, bias_sigma_prior=1.0,
                 var_mode="reference"):
        self.priors = K.Priors(mu_prior, sigma_prior, alpha_prior, bias_mu_prior, bias_sigma_prior)
        self.var_mode = {"reference": K.VAR_REFERENCE, "exact": K.VAR_EXACT}[var_mode]


_zero_scalars = {}


def _zero_scalar(dev):
    """A never-written 0-dim zero (the kl output of a call that was not asked for it) -- no fill launch per call."""
    t = _zero_scalars.get(dev.index)
    if t is None:
        if torch.cuda.is_current_stream_capturing():
            raise K.LbbnnError("constant buffer would be created during CUDA-graph capture; run one eager step first")
        t = torch.zeros((), dtype=torch.float32, device=dev)
        _zero_scalars[dev.index] = t
    return t


class _LRTFunction(torch.autograd.Function):
    """activations, kl = f(x, mu, rho, lambda, b_mu, b_rho[, z]); forward LRT:166-196, backward SURVEY §3.5."""

    @staticmethod
    def forward(ctx, x, weight_mu, weight_rho, lambdal, bias_mu, bias_rho, z, eps, cfg, sample, want_kl, noise_key,
                relu=False, mask_dx=False):
        """relu: the activations leave the kernel through F.relu (the layer's gradient input is then d loss / d PRE-relu
        activation: whoever consumes them must mask it -- the next layer's backward with mask_dx does).
        mask_dx: this layer's input x is such a relu output; its input gradient goes through [x > 0]."""
        K.require_device()
        x = x.contiguous()
        B, in_f = x.shape
        out_f = weight_mu.shape[0]
        if weight_mu.shape[1] != in_f:
            raise K.LbbnnError(f"input has {in_f} features, layer expects {weight_mu.shape[1]}")
        params = [t.contiguous() for t in (weight_mu, weight_rho, lambdal, bias_mu, bias_rho)]
        zc = z.contiguous() if z is not None else None
        layer = K.make_layer(*params, zc)
        if eps is not None:
            eps = eps.contiguous()
            if tuple(eps.shape) != (B, out_f):
                raise K.LbbnnError(f"eps must be {(B, out_f)}, got {tuple(eps.shape)}")
        noise = K.make_noise(eps, K.row_noise_seed(noise_key[0]), noise_key[1])    # per-row noise: disjoint across ranks
        flags = (K.FLAG_SAMPLE if sample else 0) | (K.FLAG_KL if want_kl else 0) | (K.FLAG_RELU if relu else 0)
        act = torch.empty(B, out_f, dtype=torch.float32, device=x.device)
        dsf = torch.empty(B, out_f, dtype=torch.float32, device=x.device) if sample else None
        ctx.set_materialize_grads(False)           # an unused output's gradient arrives as None, not as a zero-fill launch
        if want_kl:
            kl = torch.zeros((), dtype=torch.float32, device=x.device)
        else:                                      # not computed (MNF layers: the KL branch is its own node): a shared constant
            kl = _zero_scalar(x.device)
            ctx.mark_non_differentiable(kl)
        # keep M,V for the input-gradient GEMM of the backward (else it recomputes them)
        mv = (torch.empty(K.lrt_mv_bytes(in_f, out_f) // 4, dtype=torch.float32, device=x.device)
              if ctx.needs_input_grad[0] else None)
        ws = K.workspace(K.lrt_workspace_bytes(B, in_f, out_f), x.device)
        K.check(K.lib.lbbnn_lrt_f32_fwd(layer, K.ptr(x), B, noise, cfg.priors, cfg.var_mode, flags, K.ptr(act),
                                        K.ptr(dsf, allow_none=True), K.ptr(kl), K.ptr(mv, allow_none=True),
                                        ws.data_ptr(), ws.numel(), K.current_stream()))
        ctx.save_for_backward(x, *params, zc, dsf, mv)
        ctx.cfg, ctx.sample, ctx.want_kl, ctx.mask_dx = cfg, sample, want_kl, bool(mask_dx)
        return act, kl

    @staticmethod
    def backward(ctx, g_act, g_kl):
        x, wmu, wrho, lam, bmu, brho, z, dsf, mv = ctx.saved_tensors
        cfg = ctx.cfg
        B, in_f = x.shape
        out_f = wmu.shape[0]
        dev = x.device
        g_act = torch.zeros(B, out_f, dtype=torch.float32, device=dev) if g_act is None else g_act.contiguous()
        layer = K.make_layer(wmu, wrho, lam, bmu, brho, z)
        flags = K.FLAG_SAMPLE if ctx.sample else 0
        ws = K.workspace(K.lrt_workspace_bytes(B, in_f, out_f), dev)
        grads = [torch.empty_like(t) for t in (wmu, wrho, lam, bmu, brho)]
        dz = torch.zeros_like(z) if z is not None else None
        use_kl = ctx.want_kl and g_kl is not None
        g_kl_c = g_kl.contiguous().float() if use_kl else None
        K.check(K.lib.lbbnn_lrt_f32_bwd_params(
            layer, K.ptr(x), B, K.ptr(g_act), K.ptr(dsf, allow_none=True), cfg.priors, cfg.var_mode, flags,
            K.ptr(g_kl_c, allow_none=True), 1.0 if use_kl else 0.0,
            K.LayerGrads(*[K.ptr(g) for g in grads], K.ptr(dz, allow_none=True)),
            ws.data_ptr(), ws.numel(), K.current_stream()))
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            K.check(K.lib.lbbnn_lrt_f32_bwd_input(layer, K.ptr(x), B, K.ptr(g_act), K.ptr(dsf, allow_none=True),
                                                  cfg.priors, cfg.var_mode, flags | (K.FLAG_MASK_DX if ctx.mask_dx else 0),
                                                  K.ptr(mv, allow_none=True), K.ptr(dx), ws.data_ptr(), ws.numel(),
                                                  K.current_stream()))
        return (dx, *grads, dz, None, None, None, None, None, None, None)


def lrt_linear(x, weight_mu, weight_rho, lambdal, bias_mu, bias_rho, *, z=None, eps=None, cfg=None, sample=True,
               want_kl=True, noise_key=(0, 0)):
    """Functional form: returns (activations, kl)."""
    cfg = cfg or LayerConfig()
    return _LRTFunction.apply(x, weight_mu, weight_rho, lambdal, bias_mu, bias_rho, z, eps, cfg, sample, want_kl,
                              noise_key)


class GaussianView:
    """Stand-in for the reference's `Gaussian` helper (LRT:73-100): holds references to the
    nn.Parameters; `.sigma` = log1p(exp(rho)) on demand."""

    def __init__(self, mu, rho):
        self.mu, self.rho = mu, rho

    @property
    def sigma(self):
        return torch.log1p(torch.exp(self.rho))


class BernoulliView:
    """Stand-in for the reference's `Bernoulli` helper (LRT:104-127). `.alpha` follows the layer's
    current lambdal; `rsample()` draws hard masks when `exact` (the LRT default, LRT:108)."""

    def __init__(self, layer, temperature=0.001):
        self._layer = layer
        self.exact = True
        self.temperature = temperature
        self._alpha = None

    @property
    def alpha(self):
        return self._alpha if self._alpha is not None else self._layer.alpha_q

    @alpha.setter
    def alpha(self, value):
        self._alpha = value

    def rsample(self):
        a = self.alpha
        if self.exact:
            return torch.bernoulli(a)
        return torch.distributions.RelaxedBernoulli(probs=a, temperature=self.temperature).rsample()


class BayesianLinear(nn.Module):
    """LRT layer, drop-in for LBBNN-GP-MF-LRT.py:129-197.

    Extra (keyword-only) arguments replace the reference's module globals; `eps=` on forward injects
    the N(0,1) noise of LRT:174 (parity tests), otherwise it is drawn natively (Philox) inside the
    kernel and `last_noise_key` tells lbbnn.philox_normal how to reproduce it.
    Parameter initialisation consumes torch's global RNG in the reference's order, so
    `torch.manual_seed(i)` yields the reference's initial parameters.
    """

    def __init__(self, in_features, out_features, *, device=None, mu_prior=0.0, sigma_prior=1.0, alpha_prior=0.05,
                 bias_mu_prior=0.0, bias_sigma_prior=1.0, mu_init=0.2, lambda_init=(0.0, 1.0), var_mode="reference"):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        self.weight_mu = nn.Parameter(torch.empty(out_features, in_features).uniform_(-mu_init, mu_init))
        self.weight_rho = nn.Parameter(torch.empty(out_features, in_features).uniform_(-5, -4))
        self.lambdal = nn.Parameter(torch.empty(out_features, in_features).uniform_(*lambda_init))
        torch.empty(out_features, in_features).uniform_(0.999, 0.9999)  # reference draws alpha_q here (LRT:147)
        self.bias_mu = nn.Parameter(torch.empty(out_features).uniform_(-0.2, 0.2))
        self.bias_rho = nn.Parameter(torch.empty(out_features).uniform_(-5, -4))
        self.cfg = LayerConfig(mu_prior, sigma_prior, alpha_prior, bias_mu_prior, bias_sigma_prior, var_mode)
        self.weight = GaussianView(self.weight_mu, self.weight_rho)
        self.bias = GaussianView(self.bias_mu, self.bias_rho)
        self.gamma = BernoulliView(self)
        self.kl = 0
        self._uid = next(_layer_ids)
        self._calls = 0
        self.last_noise_key = None
        if device is not None:
            self.to(device)

    # the reference materialises these as full tensors every forward; here they are derived on demand
    @property
    def alpha_q(self):
        return 1 / (1 + torch.exp(-self.lambdal.detach()))

    @property
    def mu_prior(self):
        return torch.full_like(self.weight_mu.detach(), self.cfg.priors.mu)

    @property
    def sigma_prior(self):
        return torch.full_like(self.weight_mu.detach(), self.cfg.priors.sigma)

    @property
    def alpha_prior(self):
        return torch.full_like(self.weight_mu.detach(), self.cfg.priors.alpha)

    def _next_noise_key(self):
        self._calls += 1
        self.last_noise_key = (current_seed(), (self._uid << 40) | self._calls)
        return self.last_noise_key

    def forward(self, input, sample=False, calculate_log_probs=False, eps=None, _relu=False, _mask_dx=False):
        """_relu / _mask_dx (internal, set by BayesianNetwork.forward): F.relu fused into this layer's kernel, and the relu
        backward of the layer BELOW fused into this layer's input gradient (see _LRTFunction)."""
        sample_branch = self.training or sample
        want_kl = self.training or calculate_log_probs
        key = self._next_noise_key() if (sample_branch and eps is None) else (0, 0)
        act, kl = _LRTFunction.apply(input, self.weight_mu, self.weight_rho, self.lambdal, self.bias_mu, self.bias_rho,
                                     None, eps, self.cfg, sample_branch, want_kl, key, _relu, _mask_dx)
        self.kl = kl if want_kl else 0
        return act


class BayesianNetwork(nn.Module):
    """784-400-600-10 LRT MLP, drop-in for LBBNN-GP-MF-LRT.py:199-214 (sizes configurable)."""

    def __init__(self, sizes=(28 * 28, 400, 600, 10), **layer_kwargs):
        super().__init__()
        self.sizes = tuple(sizes)
        layers = [BayesianLinear(i, o, **layer_kwargs) for i, o in zip(sizes[:-1], sizes[1:])]
        for n, l in enumerate(layers, 1):
            setattr(self, f"l{n}", l)
        self._names = [f"l{n}" for n in range(1, len(layers) + 1)]

    @property
    def layers(self):
        return [getattr(self, n) for n in self._names]

    def forward(self, x, sample=False, eps=None):
        x = x.view(-1, self.sizes[0])
        ls = self.layers
        for i, l in enumerate(ls):     # F.relu (LRT:208-209) rides in the layer kernels: forward flag here, backward mask in the next layer
            x = l.forward(x, sample, eps=None if eps is None else eps[i], _relu=i < len(ls) - 1, _mask_dx=i > 0)
        return F.log_softmax(x, dim=1)

    def kl(self):
        return sum(l.kl for l in self.layers)


def predict_ensemble(net, x, samples, ensemble_first=10, forward=None):
    """The per-batch body of `test_ensemble` for the LRT / MNF networks (LRT:239-265, MNF:287-318) without its device ->
    host NumPy round trip per MC sample: `samples` stochastic forwards `net(x, sample=True)`, accumulating on the device

      * mean_prob  = mean over samples of the row-normalised expit of the log-probabilities (`mydata_means`, LRT:249-258),
      * ensemble   = argmax of the mean of the FIRST `ensemble_first` outputs (`outputs[0:10].mean(0)`, LRT:262-263),
      * posterior_mean = argmax of `net(x, sample=False)` (LRT:264-265),
      * density    = mean over samples of one Bernoulli(alpha_q) draw per layer (LRT:242-246), when the layers expose
                     `.gamma.rsample()`; None otherwise.

    Sums are kept in fp64 so the argmax does not depend on how the samples are split over calls.  `forward(x, sample)`
    overrides the call (the MNF network draws its own z inside)."""
    call = forward if forward is not None else (lambda inp, sample: net(inp, sample=sample))
    layers = list(getattr(net, "layers", []))
    has_gamma = bool(layers) and all(hasattr(l, "gamma") and hasattr(l.gamma, "rsample") for l in layers)
    was_training = net.training if hasattr(net, "training") else False
    if hasattr(net, "eval"):
        net.eval()
    sum_prob = sum_first = None
    dens = None
    with torch.no_grad():
        for i in range(samples):
            if has_gamma:
                d = torch.cat([l.gamma.rsample().flatten() for l in layers]).mean().to(torch.float64)
                dens = d if dens is None else dens + d
            out = call(x, True).to(torch.float64)
            p = torch.sigmoid(out)
            p = p / p.sum(dim=1, keepdim=True)
            sum_prob = p if sum_prob is None else sum_prob + p
            if i < ensemble_first:
                sum_first = out if sum_first is None else sum_first + out
        mean_out = call(x, False)
    if was_training and hasattr(net, "train"):
        net.train()
    n_first = min(samples, ensemble_first)
    mean_prob = sum_prob / samples
    return {"mean_prob": mean_prob, "ensemble": (sum_first / n_first).argmax(1), "posterior_mean": mean_out.argmax(1),
            "entropy": -(mean_prob * torch.log(mean_prob)).sum(1), "density": None if dens is None else dens / samples}
