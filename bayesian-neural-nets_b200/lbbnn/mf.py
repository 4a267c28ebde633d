"""Drop-in mean-field (full weight sampling) layer and network, reference LBBNN-GP-MF.py:74-319
(and the sim-study variant LBBNN-GP-MFsim_study.py:173-300 via `logprob_on_ws=True`).

The O(out*in) work -- gamma.rsample(), w = gamma (mu + sigma eps), the five element sums behind
log_prior / log_variational_posterior, F.linear and all their gradients -- runs in liblbbnn kernels.
The O(1)/O(out) hyper-prior glue (Gamma(a,b).rsample(), the (a,b,tau) and (pa,pb) constants, the bias
terms) stays in torch on the device, exactly where the reference has it, so autograd reaches
weight_a/weight_b/bias_a/bias_b/pa/pb unchanged.
"""
import ctypes as C
import math
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi as K
from .lrt import GaussianView, current_seed, _layer_ids

_LOG_SQRT_2PI = math.log(math.sqrt(2 * math.pi))


class _GammaSample(torch.autograd.Function):
    """gamma.rsample() for a given alpha tensor (MF:110-117) -- or, from_lambda, for alpha = sigmoid(lambdal) formed inside
    the kernel (forward and backward: no torch.sigmoid node on either side)."""

    @staticmethod
    def forward(ctx, alpha, u, exact, temperature, key, from_lambda=False):
        K.require_device()
        alpha_c = alpha.contiguous()
        gamma = torch.empty_like(alpha_c)
        noise = K.make_noise(u.contiguous() if u is not None else None, key[0], key[1])
        src = (K.ptr(alpha_c), None) if from_lambda else (None, K.ptr(alpha_c))
        K.check(K.lib.lbbnn_mf_gamma_sample(*src, alpha_c.numel(), noise, int(exact), temperature, K.ptr(gamma),
                                            K.current_stream()))
        ctx.save_for_backward(alpha_c, gamma)
        ctx.exact, ctx.t, ctx.from_lambda = exact, temperature, bool(from_lambda)
        if exact:
            ctx.mark_non_differentiable(gamma)
        return gamma

    @staticmethod
    def backward(ctx, dgamma):
        if ctx.exact:
            return None, None, None, None, None, None
        alpha, gamma = ctx.saved_tensors
        dalpha = torch.empty_like(alpha)
        src = (K.ptr(alpha), None) if ctx.from_lambda else (None, K.ptr(alpha))
        K.check(K.lib.lbbnn_mf_gamma_sample_bwd(*src, K.ptr(gamma), K.ptr(dgamma.contiguous()), alpha.numel(), ctx.t,
                                                K.ptr(dalpha), K.current_stream()))
        return dalpha, None, None, None, None, None


# The two Gamma precisions of a layer call drawn outside autograd with their partial derivatives (BayesianLinear._tau_draw)
# instead of torch.distributions.Gamma(...).rsample() + its autograd nodes; False keeps the torch formulation (tests compare).
FUSED_TAU = True


_ticket_bufs = {}


def _tickets(dev):
    """Two device counters (forward, backward) for the last-block reductions of the sampler kernels on the CURRENT stream:
    zero when a launch starts, zero again when it ends; one pair per (device, stream) like the kernel workspace."""
    key = (dev.index, K.current_stream())
    t = _ticket_bufs.get(key)
    if t is None:
        if torch.cuda.is_current_stream_capturing():
            raise K.LbbnnError("ticket buffer would be created during CUDA-graph capture; run one eager step first")
        t = torch.zeros(2, dtype=torch.int32, device=dev)
        _ticket_bufs[key] = t
    return t


class _MFSample(torch.autograd.Function):
    """(w, sums[5]) = f(mu, rho, lambda, gamma, pb): weight sampling + log-prob element sums (csrc/mf.cu)."""

    @staticmethod
    def forward(ctx, mu, rho, lam, gamma, pb, alpha_stale, eps, mode, flags, key):
        K.require_device()
        mu, rho, lam = mu.contiguous(), rho.contiguous(), lam.contiguous()
        gamma = gamma.contiguous() if gamma is not None else None
        n = mu.numel()
        w = torch.empty_like(mu)
        want_lp = bool(flags & K.MF_FLAG_LOGPROBS)
        # with log-probs every sum is written by the launch's last block (ticket): no zero-fill, no second launch
        sums = (torch.empty if want_lp else torch.zeros)(5, dtype=torch.float32, device=mu.device)
        ws = K.workspace(K.lib.lbbnn_mf_workspace_bytes(n), mu.device)
        eps = eps.contiguous() if eps is not None else None
        noise = K.make_noise(eps, key[0], key[1])
        ctx.tickets = tickets = _tickets(mu.device) if want_lp else None
        if want_lp:
            K.check(K.lib.lbbnn_mf_sample_fwd_ticket(K.ptr(mu), K.ptr(rho), K.ptr(lam), K.ptr(gamma, allow_none=True),
                                                     K.ptr(alpha_stale, allow_none=True), K.ptr(pb), n, noise, mode, flags,
                                                     K.ptr(w), K.ptr(sums), ws.data_ptr(), ws.numel(), tickets.data_ptr(),
                                                     K.current_stream()))
        else:
            K.check(K.lib.lbbnn_mf_sample_fwd(K.ptr(mu), K.ptr(rho), K.ptr(lam), K.ptr(gamma, allow_none=True),
                                              K.ptr(alpha_stale, allow_none=True), K.ptr(pb), n, noise, mode, flags,
                                              K.ptr(w), K.ptr(sums), ws.data_ptr(), ws.numel(), K.current_stream()))
        ctx.save_for_backward(mu, rho, lam, gamma, pb, eps)
        ctx.mode, ctx.flags, ctx.key = mode, flags, key
        return w, sums

    @staticmethod
    def backward(ctx, dw, dsums):
        if ctx.mode != K.MF_SAMPLE:
            raise K.LbbnnError("gradients through the medimean / joint-mean forward are not implemented "
                               "(the reference only uses them under no_grad)")
        mu, rho, lam, gamma, pb, eps = ctx.saved_tensors
        n = mu.numel()
        dmu, drho, dlam = torch.empty_like(mu), torch.empty_like(mu), torch.empty_like(mu)
        want_dg = ctx.needs_input_grad[3]
        dgamma = torch.empty_like(mu) if want_dg else None
        ws = K.workspace(K.lib.lbbnn_mf_workspace_bytes(n), mu.device)
        noise = K.make_noise(eps, ctx.key[0], ctx.key[1])
        dw_c = dw.contiguous() if dw is not None else None
        ds_c = dsums.contiguous() if dsums is not None else None
        if ctx.tickets is not None:        # dpb written by the launch's last block: no fill, no reduction / scaling launches
            dpb = torch.empty_like(pb)
            K.check(K.lib.lbbnn_mf_sample_bwd_ticket(K.ptr(mu), K.ptr(rho), K.ptr(lam), K.ptr(gamma), K.ptr(pb), n, noise,
                                                     ctx.flags, K.ptr(dw_c, allow_none=True), K.ptr(ds_c, allow_none=True),
                                                     K.ptr(dmu), K.ptr(drho), K.ptr(dlam), K.ptr(dgamma, allow_none=True),
                                                     K.ptr(dpb), ws.data_ptr(), ws.numel(), ctx.tickets.data_ptr() + 4,
                                                     K.current_stream()))
        else:
            dpb = torch.zeros_like(pb)
            K.check(K.lib.lbbnn_mf_sample_bwd(K.ptr(mu), K.ptr(rho), K.ptr(lam), K.ptr(gamma), K.ptr(pb), n, noise, ctx.flags,
                                              K.ptr(dw_c, allow_none=True), K.ptr(ds_c, allow_none=True), K.ptr(dmu),
                                              K.ptr(drho), K.ptr(dlam), K.ptr(dgamma, allow_none=True), K.ptr(dpb),
                                              ws.data_ptr(), ws.numel(), K.current_stream()))
        return dmu, drho, dlam, dgamma, dpb, None, None, None, None, None


class _Linear(torch.autograd.Function):
    """F.linear(x, W, b) on the fp32 SIMT GEMM kernels (MF:255)."""

    @staticmethod
    def forward(ctx, x, W, b, relu=False, mask_dx=False):
        """relu: the output leaves the kernel through F.relu (MF:268-269); the gradient that comes back is then the one wrt the
        PRE-relu output, which the consumer must have masked -- the next layer's backward with mask_dx does (its input x is this
        relu output, and [x > 0] is the relu's derivative)."""
        K.require_device()
        x, W, b = x.contiguous(), W.contiguous(), b.contiguous()
        B, kf = x.shape
        nf = W.shape[0]
        out = torch.empty(B, nf, dtype=torch.float32, device=x.device)
        ws = K.workspace(K.lrt_workspace_bytes(B, kf, nf), x.device)
        K.check(K.lib.lbbnn_linear_f32_fwd(K.ptr(x), K.ptr(W), K.ptr(b), B, kf, nf, K.FLAG_RELU if relu else 0, K.ptr(out),
                                           ws.data_ptr(), ws.numel(), K.current_stream()))
        ctx.save_for_backward(x, W)
        ctx.mask_dx = bool(mask_dx)
        return out

    @staticmethod
    def backward(ctx, g):
        x, W = ctx.saved_tensors
        g = g.contiguous()
        B, kf = x.shape
        nf = W.shape[0]
        ws = K.workspace(K.lrt_workspace_bytes(B, kf, nf), x.device)
        dW, db = torch.empty_like(W), torch.empty(nf, dtype=torch.float32, device=x.device)
        K.check(K.lib.lbbnn_linear_f32_bwd_params(K.ptr(x), K.ptr(g), B, kf, nf, K.ptr(dW), K.ptr(db), ws.data_ptr(),
                                                  ws.numel(), K.current_stream()))
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            K.check(K.lib.lbbnn_linear_f32_bwd_input(K.ptr(x), K.ptr(W), K.ptr(g), B, kf, nf,
                                                     K.FLAG_MASK_DX if ctx.mask_dx else 0, K.ptr(dx), ws.data_ptr(),
                                                     ws.numel(), K.current_stream()))
        return dx, dW, db, None, None


class _MFLogProbs(torch.autograd.Function):
    """(bias, log_prior, log_variational_posterior) of one MF layer call from the sampler's five sums, the two Gamma draws and
    the hyper-parameters (MF:148-150, 167-173, 246-251) -- the scalar tail of the layer as ONE launch each way
    (lbbnn_mf_prior_fwd / _bwd) instead of ~70 forward and ~140 backward elementwise launches on (1,) and (out,) tensors."""

    @staticmethod
    def forward(ctx, s, a, b, tau_w, ba, bb, tau_b, bias_mu, bias_rho, pa, pb, eps_b, meta):
        K.require_device()
        sample_bias, n, key = meta[:3]
        ctx.tau_grads = meta[3] if len(meta) > 3 else None
        ts = [t.contiguous() for t in (s, a, b, tau_w, pa, pb, ba, bb, tau_b, bias_mu, bias_rho)]
        out_f = bias_mu.numel()
        dev = bias_mu.device
        f32 = dict(dtype=torch.float32, device=dev)
        bias, eps, lp = torch.empty(out_f, **f32), torch.empty(out_f, **f32), torch.empty(2, **f32)
        noise = K.make_noise(eps_b.contiguous() if eps_b is not None else None, key[0], key[1])
        K.check(K.lib.lbbnn_mf_prior_fwd(*[K.ptr(t) for t in ts], noise, int(sample_bias), out_f, float(n), K.ptr(bias), K.ptr(eps),
                                         K.ptr(lp), K.current_stream()))
        ctx.save_for_backward(*ts, bias, eps)
        ctx.meta = (sample_bias, n)
        return bias, lp[0], lp[1]

    @staticmethod
    def backward(ctx, g_bias, g_lp, g_lq):
        *ts, bias, eps = ctx.saved_tensors
        sample_bias, n = ctx.meta
        out_f = bias.numel()
        f32 = dict(dtype=torch.float32, device=bias.device)
        d10 = torch.empty(10, **f32)
        d_ba, d_bb, d_tb, d_mu, d_rho = (torch.empty(out_f, **f32) for _ in range(5))
        cz = lambda t: None if t is None else t.contiguous().float()   # noqa: E731
        g_bias, g_lp, g_lq = cz(g_bias), cz(g_lp), cz(g_lq)
        factors = [None] * 4
        if ctx.tau_grads is not None:
            # the two precisions were drawn outside autograd (BayesianLinear._tau_draw) together with d tau / d a and
            # d tau / d b: their chain rule is four fused multiply-adds inside the kernel instead of ~18 torch nodes per layer
            (ta_w, tb_w), (ta_b, tb_b), factors_ready = ctx.tau_grads
            if factors_ready is not None:
                torch.cuda.current_stream().wait_event(factors_ready)
            factors = [t.contiguous() for t in (ta_w, tb_w, ta_b, tb_b)]
        K.check(K.lib.lbbnn_mf_prior_bwd_tau(*[K.ptr(t) for t in ts], K.ptr(bias), K.ptr(eps), int(sample_bias), out_f, float(n),
                                             K.ptr(g_lp, allow_none=True), K.ptr(g_lq, allow_none=True),
                                             K.ptr(g_bias, allow_none=True), *[K.ptr(t, allow_none=True) for t in factors],
                                             K.ptr(d10), K.ptr(d_ba), K.ptr(d_bb), K.ptr(d_tb), K.ptr(d_mu), K.ptr(d_rho),
                                             K.current_stream()))
        d_a, d_b, d_tw = d10[5:6], d10[6:7], d10[7:8]
        if ctx.tau_grads is not None:
            d_tw = d_tb = None
        #       s        a    b    tau_w ba    bb    tau_b bias_mu bias_rho pa        pb        eps_b meta
        return (d10[:5], d_a, d_b, d_tw, d_ba, d_bb, d_tb, d_mu, d_rho, d10[8:9], d10[9:10], None, None)


class _StdGammaReparam(torch.autograd.Function):
    """Injected standard-gamma draw with torch's implicit reparameterisation gradient (gamma.py:79-87)."""

    @staticmethod
    def forward(ctx, a, g0):
        ctx.save_for_backward(a.detach(), g0)
        return g0.clone()

    @staticmethod
    def backward(ctx, grad):
        a, g0 = ctx.saved_tensors
        return grad * torch._standard_gamma_grad(a, g0), None


class MFBernoulliView:
    """Stand-in for the reference's `Bernoulli` helper (MF:105-128): `.alpha` is a plain tensor attribute the
    caller refreshes (MF:292-297, 369-374); `.exact` False = relaxed at `temperature` (TEMPER_PRIOR, MF:44)."""

    def __init__(self, alpha, temperature=0.001):
        self.alpha = alpha
        self.exact = False
        self.temperature = temperature
        self._uid = next(_layer_ids)
        self._calls = 0
        self.last_noise_key = None

    def rsample(self, u=None, lambdal=None):
        """lambdal: draw for alpha = sigmoid(lambdal) without materialising alpha (the gradient then goes to lambdal)."""
        self._calls += 1
        self.last_noise_key = (current_seed(), (self._uid << 40) | self._calls)
        if lambdal is not None:
            return _GammaSample.apply(lambdal, u, bool(self.exact), float(self.temperature), self.last_noise_key, True)
        return _GammaSample.apply(self.alpha, u, bool(self.exact), float(self.temperature), self.last_noise_key)


class _ExactFlag:
    """The `.exact` switch of GaussGamma / BetaBinomial (MF:137,160), flipped by the driver at epoch 20 (MF:559-569)."""

    def __init__(self, **kw):
        self.exact = False
        self.__dict__.update(kw)


class BayesianLinear(nn.Module):
    """MF layer, drop-in for LBBNN-GP-MF.py:182-255 (ctor `(in_features, out_features, layer_id)`).
    `noise=` on forward injects {"eps_w","eps_b","g0_w","g0_b"} (parity tests)."""

    def __init__(self, in_features, out_features, layer_id=1, *, device=None, temperature=0.001, mu_init=0.2,
                 lambda_init=(0.0, 1.0), logprob_on_ws=False):
        super().__init__()
        self.layer, self.in_features, self.out_features = layer_id, in_features, out_features
        U = lambda *shape: torch.empty(*shape)  # noqa: E731  (same RNG consumption order as the reference ctor)
        self.weight_mu = nn.Parameter(U(out_features, in_features).uniform_(-mu_init, mu_init))
        self.weight_rho = nn.Parameter(U(out_features, in_features).uniform_(-5, -4))
        self.weight_a = nn.Parameter(U(1).uniform_(1, 1.1))
        self.weight_b = nn.Parameter(U(1).uniform_(1, 1.1))
        self.lambdal = nn.Parameter(U(out_features, in_features).uniform_(*lambda_init))
        self.gammas = U(out_features, in_features).uniform_(0.99, 1)
        self.alpha = U(out_features, in_features).uniform_(0.999, 0.9999)
        self.pa = nn.Parameter(U(1).uniform_(1, 1.1))
        self.pb = nn.Parameter(U(1).uniform_(1, 1.1))
        self.bias_mu = nn.Parameter(U(out_features).uniform_(-0.2, 0.2))
        self.bias_rho = nn.Parameter(U(out_features).uniform_(-5, -4))
        self.bias_a = nn.Parameter(U(out_features).uniform_(1, 1.1))
        self.bias_b = nn.Parameter(U(out_features).uniform_(1, 1.1))
        self.weight = GaussianView(self.weight_mu, self.weight_rho)
        self.bias = GaussianView(self.bias_mu, self.bias_rho)
        self.gamma = MFBernoulliView(self.alpha, temperature)
        self.weight_prior = _ExactFlag(a=self.weight_a, b=self.weight_b)
        self.bias_prior = _ExactFlag(a=self.bias_a, b=self.bias_b)
        self.gamma_prior = _ExactFlag(pa=self.pa, pb=self.pb)
        self.logprob_on_ws = logprob_on_ws
        self.log_prior = 0
        self.log_variational_posterior = 0
        self.lagrangian = 0
        self._uid = next(_layer_ids)
        self._calls = 0
        self.last_noise_key = None
        if device is not None:
            self.to(device)

    def _apply(self, fn, *a, **kw):          # keep the non-parameter tensors on the module's device
        super()._apply(fn, *a, **kw)
        self.gammas, self.alpha = fn(self.gammas), fn(self.alpha)
        self.gamma.alpha = self.alpha
        return self

    def _tau(self, a, b, g0):
        if g0 is None:
            return torch.distributions.Gamma(a, b, validate_args=False).rsample()   # no host sync: graph-capturable
        return _StdGammaReparam.apply(a, g0) / b

    @staticmethod
    def _tau_draw(a, b, g0=None, value_ready=None):
        """Gamma(a, b).rsample() (MF:167-173: the precisions of the GaussGamma priors) OUTSIDE autograd, with its two partial
        derivatives: tau = g / b, g ~ standard Gamma(a) (or the injected draw g0); d tau / d a = standard_gamma_grad(a, g) / b
        (torch's implicit reparameterisation, gamma.py:79-87), d tau / d b = -g / b^2.  _MFLogProbs applies them to the
        gradient that reaches tau.  Depends on the hyper-parameters only: the network issues it for every layer on a side
        stream at the start of the step."""
        with torch.no_grad():
            g = torch._standard_gamma(a) if g0 is None else g0
            rb = 1.0 / b
            raw = g * rb
            tau = raw.clamp(min=torch.finfo(raw.dtype).tiny)       # Gamma.rsample's clamp (value only)
            if value_ready is not None:                            # the forward needs tau only: the derivative factors
                value_ready.record(torch.cuda.current_stream())    # (standard_gamma_grad: ~20 us) are the backward's
            d_a = torch._standard_gamma_grad(a, g) * rb
            d_b = -raw * rb
        return tau, (d_a, d_b)

    def forward(self, input, cgamma, sample=False, medimean=False, calculate_log_probs=False, noise=None, _relu=False,
                _mask_dx=False):
        w, bias = self._draw_weights(cgamma, sample, medimean, calculate_log_probs, noise)
        return _Linear.apply(input, w, bias, _relu, _mask_dx)

    def _draw_weights(self, cgamma, sample=False, medimean=False, calculate_log_probs=False, noise=None):
        """Everything of forward() that does not depend on the input batch: the weights and bias of this call (MF:228-245)
        and, training / calculate_log_probs, log_prior and log_variational_posterior (MF:246-251).  Returns (w, bias)."""
        noise = noise or {}
        sample_branch = self.training or sample
        want_lp = self.training or calculate_log_probs
        alpha_stale = None
        eb = noise.get("eps_b")
        if sample_branch:
            self.gammas = cgamma
            mode = K.MF_SAMPLE
        elif medimean:
            mode = K.MF_MEDIMEAN
        else:
            mode = K.MF_JOINTMEAN
            alpha_stale = self.alpha.detach().contiguous()
        flags = (K.MF_FLAG_LOGPROBS if want_lp else 0) | (K.MF_FLAG_LP_ON_WS if self.logprob_on_ws else 0) \
            | (K.MF_FLAG_EXACT_GAMMA if self.gamma.exact else 0) | (K.MF_FLAG_EXACT_WPRIOR if self.weight_prior.exact else 0) \
            | (K.MF_FLAG_EXACT_GPRIOR if self.gamma_prior.exact else 0)
        self._calls += 1
        self.last_noise_key = (current_seed(), (self._uid << 40) | self._calls)
        w, s = _MFSample.apply(self.weight_mu, self.weight_rho, self.lambdal, cgamma, self.pb, alpha_stale,
                               noise.get("eps_w"), mode, flags, self.last_noise_key)
        if want_lp:
            if not self.__dict__.pop("_alpha_fresh", False):
                self.alpha = torch.sigmoid(self.lambdal)                                      # MF:246: 1 / (1 + exp(-lambda)), one kernel
            n = float(self.weight_mu.numel())
            # bias draw (stream + 2 of the call's noise key), GaussGamma / BetaBinomial / Gaussian log-probabilities: one launch
            bias_key = (self.last_noise_key[0], self.last_noise_key[1] + (2 << 32))
            if FUSED_TAU:
                pre = self.__dict__.pop("_tau_pre", None)
                if pre is not None:
                    torch.cuda.current_stream().wait_event(pre[2])       # the values; the backward waits for the factors
                if pre is None or "g0_w" in noise or "g0_b" in noise:
                    pre = (self._tau_draw(self.weight_a, self.weight_b, noise.get("g0_w")),
                           self._tau_draw(self.bias_a, self.bias_b, noise.get("g0_b")), None, None)
                (tau_w, tgw), (tau_b, tgb) = pre[:2]
                meta = (sample_branch, n, bias_key, (tgw, tgb, pre[3]))
            else:
                tau_w = self._tau(self.weight_a, self.weight_b, noise.get("g0_w"))
                tau_b = self._tau(self.bias_a, self.bias_b, noise.get("g0_b"))
                meta = (sample_branch, n, bias_key)
            bias, self.log_prior, self.log_variational_posterior = _MFLogProbs.apply(
                s, self.weight_a, self.weight_b, tau_w, self.bias_a, self.bias_b, tau_b, self.bias_mu, self.bias_rho, self.pa,
                self.pb, eb, meta)
        else:
            self.log_prior, self.log_variational_posterior = 0, 0
            if sample_branch:
                sb = self.bias.sigma
                bias = self.bias_mu + sb * (eb if eb is not None else torch.randn_like(sb))
            else:
                bias = self.bias_mu
        return w, bias


class BayesianNetwork(nn.Module):
    """784-400-600-10 MF network, drop-in for LBBNN-GP-MF.py:259-319 (sizes configurable)."""

    def __init__(self, sizes=(28 * 28, 400, 600, 10), num_batches=600, **layer_kwargs):
        super().__init__()
        self.sizes, self.num_batches = tuple(sizes), num_batches
        for n, (i, o) in enumerate(zip(sizes[:-1], sizes[1:]), 1):
            setattr(self, f"l{n}", BayesianLinear(i, o, 1, **layer_kwargs))
        self._names = [f"l{n}" for n in range(1, len(sizes))]

    @property
    def layers(self):
        return [getattr(self, n) for n in self._names]

    def forward(self, x, *gammas, sample=False, medimean=False, noises=None, **named):
        return F.log_softmax(self._logits(x, *gammas, sample=sample, medimean=medimean, noises=noises, **named), dim=1)

    def _logits(self, x, *gammas, sample=False, medimean=False, noises=None, **named):
        """forward() without the closing log_softmax (GraphedTrainer fuses it with the loss)."""
        gs = list(gammas) + [named[f"g{i}"] for i in range(len(gammas) + 1, len(self._names) + 1) if f"g{i}" in named]
        x = x.view(-1, self.sizes[0])
        ls = self.layers
        for i, l in enumerate(ls):          # F.relu (MF:268-269) rides in the layer kernels: forward flag, next layer's dx mask
            x = l.forward(x, gs[i], sample, medimean, noise=None if noises is None else noises[i], _relu=i < len(ls) - 1,
                          _mask_dx=i > 0)
        return x

    def _elbo_terms(self, input):
        """One sample of sample_elbo (MF:285-319, samples = 1) up to the logits: (logits, the layers' log q and log prior
        terms, their signs in loss = nll + (log q - log prior) / num_batches)."""
        fork = None
        if FUSED_TAU and input.is_cuda:
            cur = torch.cuda.current_stream()
            if getattr(self, "_tau_stream", None) is None or self._tau_stream.device != input.device:
                self._tau_stream = torch.cuda.Stream(device=input.device)
            fork = torch.cuda.Event()
            fork.record(cur)
        ls = self.layers
        if fork is not None and (getattr(self, "_layer_streams", None) is None or
                                 self._layer_streams[0].device != input.device):
            self._layer_streams = [torch.cuda.Stream(device=input.device) for _ in ls]
        gs = []
        for i, l in enumerate(ls):
            if fork is not None:              # alpha = sigmoid(lambda) inside the mask kernels; the attribute on the side stream
                self._layer_streams[i].wait_event(fork)
                with torch.cuda.stream(self._layer_streams[i]):
                    gs.append(l.gamma.rsample(None, lambdal=l.lambdal))
            else:
                l.alpha = torch.sigmoid(l.lambdal)
                l.gamma.alpha = l.alpha
                gs.append(l.gamma.rsample(None))
            l._alpha_fresh = True             # the layer call's own alpha (MF:246) is this very value: no second launch
        if fork is not None:                  # the layers' precisions depend on hyper-parameters only: side stream
            # (issued here, after the gamma launches, but forked from the start of the step: a captured graph issues its
            # nodes in capture order, and ten side-stream launches in front of the main path delayed it by ~12 us)
            self._tau_stream.wait_event(fork)
            with torch.cuda.stream(self._tau_stream), torch.no_grad():
                for l in self.layers:         # the reference's alpha attributes (MF:290-297): values only, nobody waits for them
                    l.alpha = torch.sigmoid(l.lambdal)
                    l.alpha.record_stream(cur)
                    l.gamma.alpha = l.alpha
                # ALL layers' weight and bias precisions as one batch: one standard-gamma draw, one standard_gamma_grad and a
                # handful of elementwise launches over ~10^3 elements instead of nine launches per precision and layer
                hp = [(l.weight_a, l.weight_b) for l in self.layers] + [(l.bias_a, l.bias_b) for l in self.layers]
                a_all = torch.cat([a.reshape(-1) for a, _ in hp])
                b_all = torch.cat([b.reshape(-1) for _, b in hp])
                ev, ev_grads = torch.cuda.Event(), torch.cuda.Event()
                tau, (d_a, d_b) = BayesianLinear._tau_draw(a_all, b_all, value_ready=ev)
                ev_grads.record(self._tau_stream)
                for u in (tau, d_a, d_b):
                    u.record_stream(cur)
                    for st in self._layer_streams:
                        u.record_stream(st)
                parts, off = [], 0
                for a, _ in hp:
                    n = a.numel()
                    parts.append((tau[off:off + n].view_as(a), (d_a[off:off + n].view_as(a), d_b[off:off + n].view_as(a))))
                    off += n
                L = len(self.layers)
                for i, l in enumerate(self.layers):
                    l._tau_pre = (parts[i], parts[L + i], ev, ev_grads)
        if fork is not None and os.environ.get("LBBNN_MF_STREAMS", "1") == "1":
            # Mask, weights, bias and log-probabilities of a layer depend on parameters and noise only: each layer's on ITS
            # stream, all three at once from the start of the step; the caller's stream carries just the linear layers and
            # waits for one event per layer.  Autograd replays every node on its forward stream, so the log-probability
            # backward of layer l (sampler + scalar tail: 14-23 us) runs beside the linear backward of layer l - 1 as well.
            drawn = []
            for i, l in enumerate(ls):
                with torch.cuda.stream(self._layer_streams[i]):
                    w, bias = l._draw_weights(gs[i], True, False, False, None)
                    ev = torch.cuda.Event()
                    ev.record(self._layer_streams[i])
                for t in (w, bias, l.log_prior, l.log_variational_posterior):
                    t.record_stream(cur)
                drawn.append((w, bias, ev))
            x = input.view(-1, self.sizes[0])
            for i, (w, bias, ev) in enumerate(drawn):
                cur.wait_event(ev)
                x = _Linear.apply(x, w, bias, i < len(ls) - 1, i > 0)
            logits = x
        else:
            if fork is not None:
                for i, st in enumerate(self._layer_streams):
                    cur.wait_stream(st)
            logits = self._logits(input, *gs, sample=True, medimean=False)
        for l in self.layers:
            l.__dict__.pop("_tau_pre", None)
            l.__dict__.pop("_alpha_fresh", None)
        lq = [l.log_variational_posterior for l in self.layers]
        lp = [l.log_prior for l in self.layers]
        return logits, lq + lp, [1.0] * len(lq) + [-1.0] * len(lp)

    def log_prior(self):
        return sum(l.log_prior for l in self.layers)

    def log_variational_posterior(self):
        return sum(l.log_variational_posterior for l in self.layers)

    def sample_elbo(self, input, target, samples=1, noises=None, us=None):
        """MF:285-319.  noises / us: per-sample lists of per-layer injected noise (tests)."""
        outs, lps, lqs, nlls = [], [], [], []
        for i in range(samples):
            gs = []
            for li, l in enumerate(self.layers):
                l.alpha = torch.sigmoid(l.lambdal)            # 1 / (1 + exp(-lambda)) (MF:290) as one kernel each way
                l.gamma.alpha = l.alpha
                gs.append(l.gamma.rsample(None if us is None else us[i][li]))
            out = self.forward(input, *gs, sample=True, medimean=False, noises=None if noises is None else noises[i])
            outs.append(out)
            lps.append(self.log_prior())
            lqs.append(self.log_variational_posterior())
            nlls.append(F.nll_loss(out, target, reduction="sum"))
        log_prior, log_q, nll = torch.stack(lps).mean(), torch.stack(lqs).mean(), torch.stack(nlls).mean()
        loss = nll + (log_q - log_prior) / self.num_batches
        return loss, log_prior, log_q, nll


class SimStudyNetwork(nn.Module):
    """The simulation-study model: one MF layer 20 -> 1 as a logistic regression, drop-in for
    LBBNN-GP-MFsim_study.py:250-300 (`BayesianNetwork` there).  Differences from the MNIST script that the layer
    reproduces: init ranges mu~U(-.01,.01), lambda~U(-.5,.5) (MFsim:182,191), the log-probs are evaluated at the
    UNMASKED weights ws (MFsim:233,237), the output is sigmoid + BCELoss(sum) (MFsim:258,287)."""

    def __init__(self, in_features=20, num_batches=5.0, **layer_kwargs):
        super().__init__()
        kw = dict(mu_init=0.01, lambda_init=(-0.5, 0.5), logprob_on_ws=True)
        kw.update(layer_kwargs)
        self.l1 = BayesianLinear(in_features, 1, 1, **kw)
        self.num_batches = num_batches

    @property
    def layers(self):
        return [self.l1]

    def forward(self, x, g1, sample=False, medimean=False, noise=None):
        return torch.sigmoid(self.l1(x, g1, sample, medimean, noise=noise))

    def log_prior(self):
        return self.l1.log_prior

    def log_variational_posterior(self):
        return self.l1.log_variational_posterior

    def sample_elbo(self, input, target, samples=1, noises=None, us=None):
        """MFsim:272-300.  Returns (loss, log_prior, log_variational_posterior, negative_log_likelihood, out)."""
        outs, lps, lqs, nlls = [], [], [], []
        tgt = target.unsqueeze(1).float()
        for i in range(samples):
            self.l1.alpha = torch.sigmoid(self.l1.lambdal)
            self.l1.gamma.alpha = self.l1.alpha
            g1 = self.l1.gamma.rsample(None if us is None else us[i])
            out = self.forward(input, g1, sample=True, medimean=False, noise=None if noises is None else noises[i])
            outs.append(out)
            lps.append(self.log_prior())
            lqs.append(self.log_variational_posterior())
            nlls.append(F.binary_cross_entropy(out, tgt, reduction="sum"))
        log_prior, log_q, nll = torch.stack(lps).mean(), torch.stack(lqs).mean(), torch.stack(nlls).mean()
        loss = nll + (log_q - log_prior) / self.num_batches
        return loss, log_prior, log_q, nll, torch.stack(outs).mean(0)


# the 11 tensors of a sim-study layer in the packed order of lbbnn_mfsim (include/lbbnn.h) and the study's SGD learning
# rates (MFsim:359-374)
SIM_PARAM_NAMES = ("weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho", "weight_a", "weight_b", "bias_a", "bias_b",
                   "pa", "pb")
SIM_STUDY_LRS = {"weight_mu": 1e-4, "weight_rho": 1e-4, "lambdal": 1e-3, "bias_mu": 1e-4, "bias_rho": 1e-4, "weight_a": 1e-3,
                 "weight_b": 1e-3, "bias_a": 1e-3, "bias_b": 1e-3, "pa": 1e-3, "pb": 1e-3}
_SIM_NOISE = ("eps_w", "eps_b", "g0_w", "g0_b")


class SimStudyEnsemble:
    """Every repetition of the simulation study (MFsim:344-429) trained in ONE kernel launch (csrc/mf_sim.cu): R
    SimStudyNetwork replicas, each running sample_elbo + backward + per-tensor SGD for whole epochs over minibatches of
    `batch_size` consecutive rows of X.

    The replicas' parameters live in one packed (R, P) device buffer; every module's nn.Parameters are re-pointed at views of
    it (and, with materialize_grads, their .grad at the last step's gradients), so state_dict() and eager sample_elbo keep
    working on each replica.  X is (n, in) shared by every replica or (R, n, in); y the {0, 1} targets (n,) or (R, n).
    lrs: None = the study's rates (SIM_STUDY_LRS); a dict overrides per tensor name.  Native noise is Philox keyed by
    (seed, replica, the replica's step, kind of draw).  The `.exact` flags of gamma / weight_prior / gamma_prior are read from
    the modules at every run()."""

    def __init__(self, nets, X, y, batch_size=400, lrs=None, seed=0, materialize_grads=True):
        nets = list(nets)
        if not nets:
            raise K.LbbnnError("SimStudyEnsemble needs at least one network")
        layers = [n.l1 for n in nets]
        in_f = layers[0].in_features
        for n, l in zip(nets, layers):
            if (l.in_features, l.out_features) != (in_f, 1):
                raise K.LbbnnError(f"every replica must be an {in_f} -> 1 SimStudyNetwork, got {l.in_features} -> {l.out_features}")
            if not l.logprob_on_ws:
                raise K.LbbnnError("the replicas must evaluate their log-probabilities at the unmasked ws (SimStudyNetwork)")
            if float(n.num_batches) != float(nets[0].num_batches) or float(l.gamma.temperature) != float(layers[0].gamma.temperature):
                raise K.LbbnnError("the replicas' num_batches and gamma temperature must agree")
        if in_f > K.MFSIM_MAX_IN:
            raise K.LbbnnError(f"in_features = {in_f} is above the kernel's limit of {K.MFSIM_MAX_IN}")
        R = len(nets)
        if X.dim() == 2:
            n = X.shape[0]
        elif X.dim() == 3 and X.shape[0] == R:
            n = X.shape[1]
        else:
            raise K.LbbnnError(f"X must be (n, {in_f}) or ({R}, n, {in_f}), got {tuple(X.shape)}")
        if X.shape[-1] != in_f:
            raise K.LbbnnError(f"X has {X.shape[-1]} features, the networks {in_f}")
        if tuple(y.shape) not in ((n,), (R, n)):
            raise K.LbbnnError(f"y must be ({n},) or ({R}, {n}), got {tuple(y.shape)}")
        B = int(batch_size)
        if B < 1 or n % B:
            raise K.LbbnnError(f"the {n} rows are not a whole number of minibatches of {B}")
        rates = dict(SIM_STUDY_LRS)
        if lrs is not None:
            unknown = set(lrs) - set(SIM_PARAM_NAMES)
            if unknown:
                raise K.LbbnnError(f"unknown parameter names in lrs: {sorted(unknown)}")
            rates.update(lrs)
        self._flags_of(layers)
        params = [getattr(l, name) for l in layers for name in SIM_PARAM_NAMES]
        if any(not p.is_cuda for p in params) or not X.is_cuda or not y.is_cuda:
            raise K.LbbnnError("SimStudyEnsemble takes CUDA networks and data (no CPU fallback)")
        dev = params[0].device
        if any(p.device != dev for p in params) or X.device != dev or y.device != dev:
            raise K.LbbnnError("networks and data must live on one device")
        K.require_device()
        self.nets, self.layers, self.R, self.in_features, self.rows, self.batch = nets, layers, R, in_f, n, B
        self.num_batches, self.temperature = float(nets[0].num_batches), float(layers[0].gamma.temperature)
        self.lrs = [float(rates[name]) for name in SIM_PARAM_NAMES]
        self.seed = int(seed)
        self.X = X.detach().to(torch.float32).contiguous()
        self.y = y.detach().to(torch.float32).contiguous()
        self.P = (3 * in_f + 8 + 3) // 4 * 4
        f32 = dict(dtype=torch.float32, device=dev)
        self.flat = torch.zeros(R, self.P, **f32)
        self.grads = torch.zeros(R, self.P, **f32) if materialize_grads else None
        self.step = torch.zeros(R, dtype=torch.int64, device=dev)
        self._offsets = {}
        off = 0
        for name in SIM_PARAM_NAMES:
            self._offsets[name] = off
            off += getattr(layers[0], name).numel()
        with torch.no_grad():
            for r, l in enumerate(layers):
                for name in SIM_PARAM_NAMES:
                    p = getattr(l, name)
                    o, k = self._offsets[name], p.numel()
                    view = self.flat[r, o:o + k].view(p.shape)
                    view.copy_(p.data)
                    p.data = view
                    if self.grads is not None:
                        p.grad = self.grads[r, o:o + k].view(p.shape)

    @staticmethod
    def _flags_of(layers):
        def one(l):
            return (K.MF_FLAG_EXACT_GAMMA if l.gamma.exact else 0) | (K.MF_FLAG_EXACT_WPRIOR if l.weight_prior.exact else 0) \
                | (K.MF_FLAG_EXACT_GPRIOR if l.gamma_prior.exact else 0)
        flags = {one(l) for l in layers}
        if len(flags) != 1:
            raise K.LbbnnError("the replicas' .exact flags (gamma, weight_prior, gamma_prior) differ")
        return flags.pop()

    def steps_per_epoch(self):
        return self.rows // self.batch

    def run(self, epochs, noise=None):
        """Train every replica for `epochs` epochs in one launch on the current stream; returns the (R, steps, 4) device tensor
        of [loss, nll, log_prior, log_q] per step.  noise: injected draws instead of Philox (tests) -- a dict of eps_w
        (R, steps, in), eps_b, g0_w, g0_b (R, steps) and exactly one of u (R, steps, in) or gamma (R, steps, in): constant masks,
        no gradient through gamma."""
        epochs = int(epochs)
        if epochs < 1:
            raise K.LbbnnError(f"epochs must be >= 1, got {epochs}")
        flags = self._flags_of(self.layers)
        R, in_f, steps = self.R, self.in_features, epochs * self.steps_per_epoch()
        stats = torch.empty(R, steps, 4, dtype=torch.float32, device=self.flat.device)
        d = K.MfSim()
        d.replicas, d.in_features, d.rows, d.batch = R, in_f, self.rows, self.batch
        d.params, d.param_stride = K.ptr(self.flat), self.P
        d.x, d.x_stride = K.ptr(self.X), (self.rows * in_f if self.X.dim() == 3 else 0)
        d.y, d.y_stride = K.ptr(self.y), (self.rows if self.y.dim() == 2 else 0)
        d.lr = (C.c_float * 11)(*self.lrs)
        d.num_batches, d.temperature, d.flags = self.num_batches, self.temperature, flags
        d.seed = self.seed & (2 ** 64 - 1)
        d.step = K.ptr(self.step, torch.int64)
        d.stats, d.grads = K.ptr(stats), K.ptr(self.grads, allow_none=True)
        keep = []
        if noise is not None:
            if set(noise) - set(_SIM_NOISE) - {"u", "gamma"} or not set(_SIM_NOISE) <= set(noise) \
                    or ("u" in noise) == ("gamma" in noise):
                raise K.LbbnnError("injected noise: eps_w, eps_b, g0_w, g0_b and exactly one of u / gamma")
            for name, t in noise.items():
                want = (R, steps, in_f) if name in ("eps_w", "u", "gamma") else (R, steps)
                t = t.to(torch.float32).contiguous()
                if tuple(t.shape) != want:
                    raise K.LbbnnError(f"injected {name} must be {want}, got {tuple(t.shape)}")
                keep.append(t)
                setattr(d, name, K.ptr(t))
        K.check(K.lib.lbbnn_mfsim_train_f32(C.byref(d), epochs, K.current_stream()))
        return stats

    def inclusion_probabilities(self):
        """alpha = 1 / (1 + exp(-lambda)) of every replica, (R, in): what the study reports per repetition (MFsim:347-350)."""
        o = self._offsets["lambdal"]
        return 1.0 / (1.0 + torch.exp(-self.flat[:, o:o + self.in_features]))


class _McLane:
    """Buffers, device sample counter, fp64 accumulators, stream and captured graph of one concurrent slice of the loop."""

    def __init__(self, mc, dev):
        f32 = dict(dtype=torch.float32, device=dev)
        SB, B, sizes = mc.SB, mc.B, mc.sizes
        self.w = [torch.zeros(SB, o, i, **f32) for i, o in sizes]
        self.b = [torch.zeros(SB, o, **f32) for _, o in sizes]
        self.h = [torch.zeros(SB, B, o, **f32) for _, o in sizes]
        self.w_lo = [torch.zeros_like(self.w[i]) for i in range(mc.n_tc)]
        self.h_hi = [torch.zeros(B, SB * sizes[i][1], **f32) for i in range(mc.n_tc - 1)]
        self.h_lo = [torch.zeros_like(t) for t in self.h_hi]
        C_ = sizes[-1][1]
        self.sum_logp = torch.zeros(B, C_, dtype=torch.float64, device=dev)
        self.sum_prob = torch.zeros(B, C_, dtype=torch.float64, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.stream = None
        self.graph = None

    def reset(self, first_sample):
        self.sum_logp.zero_()
        self.sum_prob.zero_()
        self.counter.fill_(int(first_sample))


class MCPredictor:
    """Posterior-predictive model averaging over Monte-Carlo weight samples (test_ensemble, MF:345-436):
    for each sample, fresh hard masks gamma ~ Bernoulli(alpha) and weights per layer, a forward over the whole
    input batch, and the two accumulators of the reference (mean log-softmax -> ensemble argmax, MF:416-417;
    mean row-normalised expit -> predictive probabilities / OOD entropy, MF:397-408, 478-494).

    samples_per_launch samples = one CUDA-graph replay (2 kernels per layer + 1).  Sample s draws from Philox streams keyed
    by s itself (a device counter), so any split of [0, S) across ranks, lanes or launches reproduces the same draws;
    partial sums are fp64 and are combined in a fixed order (lanes, then ONE all-reduce over the process_group) -- argmax
    is independent of the split.
    """

    NSTREAMS = 4   # Philox streams per (sample, layer): gamma u, eps_w, eps_b, spare

    def __init__(self, net, batch, seed=None, use_graph=True, process_group=None, samples_per_launch=8, gemm="auto",
                 lanes=None, fused_head=True):
        """samples_per_launch: weight samples pushed through every kernel of the loop together (csrc/mc_predict.cu);
        1 = the one-sample kernels.  Results do not depend on it: every sample draws from streams keyed by its index.
        gemm: "simt" = fp32 CUDA-core GEMMs; "tc" = every eligible leading layer on the tensor cores at fp32 accuracy
        (3xTF32 on tcgen05, csrc/tc_gemm_tf32.cu); "auto" = tensor cores for the leading layers at least 64 wide.
        lanes: the samples of a run() are dealt to this many independent launch sequences on their own streams (own
        buffers and accumulators), so one lane's ALU-bound weight sampling overlaps another's tensor-core GEMMs;
        default 2 with tensor-core GEMMs, else 1.
        fused_head: a last layer of <= 16 classes runs fused with the accumulation (lbbnn_mc_head_accumulate)."""
        K.require_device()
        if gemm not in ("auto", "simt", "tc"):
            raise ValueError(f"gemm must be 'auto', 'simt' or 'tc', got {gemm!r}")
        self.net, self.layers, self.B = net, list(net.layers), int(batch)
        dev = self.layers[0].weight_mu.device
        self.device = dev
        self.seed = current_seed() if seed is None else int(seed)
        self.pg = process_group
        self.SB = SB = max(1, int(samples_per_launch))
        f32 = dict(dtype=torch.float32, device=dev)
        self.sizes = sizes = [(l.in_features, l.out_features) for l in self.layers]
        self.x = torch.zeros(self.B, sizes[0][0], **f32)
        # leading layers that run as 3xTF32 tensor-core GEMMs: operands travel as (hi, lo) pairs; a layer feeding another
        # tensor-core layer writes its activations as (batch, SB * out) so the next one reads them as a strided batch
        self.n_tc = 0
        if SB > 1 and gemm != "simt":
            for i, (k, o) in enumerate(sizes):
                ok = k % 4 == 0 and (i == 0 or sizes[i - 1][1] % 4 == 0) and (gemm == "tc" or o >= 64)
                if not ok:
                    break
                self.n_tc = i + 1
        self.prepared = SB > 1          # batched sampler reads sigma / alpha computed once per run()
        kl, cl = sizes[-1]
        self.fused_head = (SB > 1 and fused_head and self.n_tc < len(sizes) and len(sizes) > 1 and cl <= 16 and kl % 4 == 0
                           and 16 * (cl + 8) * kl <= 220 * 1024)
        if self.n_tc:
            self.x_hi, self.x_lo = torch.zeros_like(self.x), torch.zeros_like(self.x)
        if self.prepared:
            self.sigma = [torch.zeros(o, i, **f32) for i, o in sizes]
            self.alpha = [torch.zeros(o, i, **f32) for i, o in sizes]
            self.bias_sigma = [torch.zeros(o, **f32) for _, o in sizes]
        n_lanes = (2 if self.n_tc else 1) if lanes is None else max(1, int(lanes))
        if SB == 1:
            n_lanes = 1     # the one-sample kernels share self.ws (split-K scratch of lbbnn_linear_f32_fwd): no concurrent lanes
        self.lanes = [_McLane(self, dev) for _ in range(n_lanes)]
        self.ws = torch.empty(max(K.lrt_workspace_bytes(self.B, i, o) for i, o in sizes), dtype=torch.uint8, device=dev)
        self.kernels_per_launch = 0
        for lane in self.lanes:
            lane.stream = torch.cuda.Stream(device=dev) if (use_graph or n_lanes > 1) else None
        if use_graph:
            self._prepare()
            for lane in self.lanes:
                s = lane.stream
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    self._enqueue(lane, SB)
                torch.cuda.current_stream().wait_stream(s)
                torch.cuda.synchronize()
                lane.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(lane.graph):
                    self._enqueue(lane, SB)
            self.reset()

    # single-lane views of the buffers (tests, profiling scripts)
    w = property(lambda self: self.lanes[0].w)
    b = property(lambda self: self.lanes[0].b)
    h = property(lambda self: self.lanes[0].h)
    w_lo = property(lambda self: self.lanes[0].w_lo)
    counter = property(lambda self: self.lanes[0].counter)

    @property
    def graph(self):
        return self.lanes[0].graph

    @graph.setter
    def graph(self, value):
        if value is not None:
            raise ValueError("graphs are captured by the constructor; only None (drop them) can be assigned")
        for lane in self.lanes:
            lane.graph = None

    @property
    def sum_logp(self):
        """This rank's partial sum over the samples of the last run(): lanes added in lane order."""
        return self._lane_sum("sum_logp")

    @property
    def sum_prob(self):
        return self._lane_sum("sum_prob")

    def _lane_sum(self, name):
        tot = getattr(self.lanes[0], name)
        for lane in self.lanes[1:]:
            tot = tot + getattr(lane, name)
        return tot

    @property
    def kernels_per_sample(self):
        return self.kernels_per_launch / self.SB

    def _noise(self, lane, layer, which):
        stride = self.NSTREAMS * len(self.layers)
        return K.make_noise(None, self.seed, layer * self.NSTREAMS + which, lane.counter, stride)

    def _desc(self, i):
        l = self.layers[i]
        if self.prepared:
            return K.make_layer(l.weight_mu.data, self.sigma[i], self.alpha[i], l.bias_mu.data, self.bias_sigma[i])
        return K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)

    def _prepare(self):
        """Per-run() work on the current stream: sigma / alpha of the (possibly updated) parameters, hi / lo of the input."""
        st = K.current_stream()
        if self.prepared:
            for i, l in enumerate(self.layers):
                raw = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
                K.check(K.lib.lbbnn_mc_prepare(raw, K.ptr(self.sigma[i]), K.ptr(self.alpha[i]), K.ptr(self.bias_sigma[i]), st))
        if self.n_tc:
            K.check(K.lib.lbbnn_tf32_split(K.ptr(self.x), self.x.numel(), K.ptr(self.x_hi), K.ptr(self.x_lo), st))

    def _enqueue(self, lane, n):
        """One launch sequence for the next n <= samples_per_launch samples of a lane, on the current stream."""
        st = K.current_stream()
        L = len(self.layers)
        if self.SB == 1:
            return self._enqueue_one(lane)
        stride = self.NSTREAMS * L
        h, hs = self.x, 0
        for i, l in enumerate(self.layers):
            desc = self._desc(i)
            if i < self.n_tc:
                self._enqueue_tc_layer(lane, i, l, desc, n, stride, st)
                h, hs = lane.h[i], self.B * l.out_features
                continue
            K.check(K.lib.lbbnn_mc_sample_split(desc, n, K.ptr(lane.counter, torch.int64), self.seed & (2 ** 64 - 1),
                                                i * self.NSTREAMS, stride, 1, K.ptr(lane.w[i]), None, K.ptr(lane.b[i]), st))
            if i == L - 1 and self.fused_head:      # classifier head and the accumulators in one kernel, no logits
                K.check(K.lib.lbbnn_mc_head_accumulate(K.ptr(h), hs, K.ptr(lane.w[i]), K.ptr(lane.b[i]), n, self.B,
                                                       l.in_features, l.out_features, lane.sum_logp.data_ptr(),
                                                       lane.sum_prob.data_ptr(), K.ptr(lane.counter, torch.int64), st))
                self.kernels_per_launch = 2 * L + (n - 1 if self.n_tc == 1 else 0)
                return
            K.check(K.lib.lbbnn_linear_f32_batched(K.ptr(h), hs, K.ptr(lane.w[i]), K.ptr(lane.b[i]), n, self.B,
                                                   l.in_features, l.out_features, K.FLAG_RELU if i < L - 1 else 0,
                                                   K.ptr(lane.h[i]), st))
            h, hs = lane.h[i], self.B * l.out_features
        K.check(K.lib.lbbnn_mc_accumulate_batched(K.ptr(h), n, self.B, self.layers[-1].out_features,
                                                  lane.sum_logp.data_ptr(), lane.sum_prob.data_ptr(),
                                                  K.ptr(lane.counter, torch.int64), st))
        self.kernels_per_launch = 2 * L + 1 + (n - 1 if self.n_tc == 1 else 0)

    def _enqueue_tc_layer(self, lane, i, l, desc, n, stride, st):
        L, SB, B = len(self.layers), self.SB, self.B
        k, o = l.in_features, l.out_features
        K.check(K.lib.lbbnn_mc_sample_split(desc, n, K.ptr(lane.counter, torch.int64), self.seed & (2 ** 64 - 1),
                                            i * self.NSTREAMS, stride, 1, K.ptr(lane.w[i]), K.ptr(lane.w_lo[i]),
                                            K.ptr(lane.b[i]), st))
        flags = K.FLAG_RELU if i < L - 1 else 0
        feeds_tc = i + 1 < self.n_tc
        if feeds_tc:      # (batch, SB * out) hi / lo for the next tensor-core layer
            out, out_hi, out_lo, pitch, bstride = None, K.ptr(lane.h_hi[i]), K.ptr(lane.h_lo[i]), SB * o, o
        else:             # (SB, batch, out) fp32 for the CUDA-core layer / the accumulation kernel
            out, out_hi, out_lo, pitch, bstride = K.ptr(lane.h[i]), None, None, o, B * o
        if i == 0:        # all samples read the same input
            if feeds_tc:  # ONE problem, N = n * out
                K.check(K.lib.lbbnn_tc_linear_tf32x3(K.ptr(self.x_hi), K.ptr(self.x_lo), k, 0, K.ptr(lane.w[i]),
                                                     K.ptr(lane.w_lo[i]), K.ptr(lane.b[i]), 1, B, n * o, k, flags,
                                                     out, out_hi, out_lo, pitch, bstride, st))
            else:         # (SB, batch, out) wanted: one problem per sample
                for z in range(n):
                    K.check(K.lib.lbbnn_tc_linear_tf32x3(K.ptr(self.x_hi), K.ptr(self.x_lo), k, 0, K.ptr(lane.w[i][z]),
                                                         K.ptr(lane.w_lo[i][z]), K.ptr(lane.b[i][z]), 1, B, o, k, flags,
                                                         K.ptr(lane.h[i][z]), None, None, o, 0, st))
        else:
            pk = SB * k   # previous layer's row pitch; its sample z sits at column offset z * k
            K.check(K.lib.lbbnn_tc_linear_tf32x3(K.ptr(lane.h_hi[i - 1]), K.ptr(lane.h_lo[i - 1]), pk, k,
                                                 K.ptr(lane.w[i]), K.ptr(lane.w_lo[i]), K.ptr(lane.b[i]), n, B, o, k,
                                                 flags, out, out_hi, out_lo, pitch, bstride, st))

    def _enqueue_one(self, lane):
        st = K.current_stream()
        L = len(self.layers)
        h = self.x
        n = 0
        for i, l in enumerate(self.layers):
            desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
            K.check(K.lib.lbbnn_mf_sample_predict(desc, self._noise(lane, i, 0), self._noise(lane, i, 1),
                                                  self._noise(lane, i, 2), K.ptr(lane.w[i]), K.ptr(lane.b[i]), st))
            K.check(K.lib.lbbnn_linear_f32_fwd(K.ptr(h), K.ptr(lane.w[i]), K.ptr(lane.b[i]), self.B, l.in_features,
                                               l.out_features, K.FLAG_RELU if i < L - 1 else 0, K.ptr(lane.h[i]),
                                               self.ws.data_ptr(), self.ws.numel(), st))
            n += 3
            h = lane.h[i]
        K.check(K.lib.lbbnn_mc_accumulate(K.ptr(h), self.B, self.layers[-1].out_features, lane.sum_logp.data_ptr(),
                                          lane.sum_prob.data_ptr(), K.ptr(lane.counter, torch.int64), st))
        self.kernels_per_launch = n + 1

    def reset(self, first_sample=0):
        for lane in self.lanes:
            lane.reset(first_sample)

    def run(self, x, samples, first_sample=0, masks=None):
        """Accumulate `samples` weight samples with global indices first_sample.. on this rank.
        masks: per-layer {0, 1} tensors that REPLACE the Bernoulli(alpha) draw of the inclusion masks -- the
        median-probability model [alpha > 0.5] of `outofsample(medimod=True)` (MF:462-465); weights and biases are still
        sampled.  (A mask value of 1 / 0 is drawn with certainty: the sampler compares a uniform in (0, 1) with it.)"""
        self.x.copy_(x.reshape(self.x.shape), non_blocking=True)
        self._prepare()
        if masks is not None:
            if not self.prepared:
                raise K.LbbnnError("fixed masks need samples_per_launch > 1 (the batched sampler reads alpha from a buffer)")
            for a, m in zip(self.alpha, masks):
                a.copy_(m)
        # whole launches are dealt to the lanes as contiguous index ranges; the partial last launch goes to the last lane
        full, rest = divmod(int(samples), self.SB)
        nl = len(self.lanes)
        main = torch.cuda.current_stream()
        first = int(first_sample)
        for j, lane in enumerate(self.lanes):
            launches = full // nl + (1 if j < full % nl else 0)
            tail = rest if j == nl - 1 else 0
            side = lane.stream if nl > 1 else None
            if side is not None:
                side.wait_stream(main)
            with torch.cuda.stream(side) if side is not None else _null_ctx():
                lane.reset(first)
                for _ in range(launches):
                    if lane.graph is not None:
                        lane.graph.replay()
                    else:
                        self._enqueue(lane, self.SB)
                if tail:
                    self._enqueue(lane, tail)      # a partial last launch runs outside the captured graph
            first += launches * self.SB + tail
        for lane in self.lanes:
            if nl > 1:
                main.wait_stream(lane.stream)

    def result(self, total_samples):
        """Combine lanes and ranks (one all-reduce of the two fp64 accumulators) and form the reference's statistics.

        `pred` is the argmax of the mean log-softmax over ALL `total_samples` samples.  The reference's ensemble
        prediction is `outputs[0:10].mean(0)` (MF:416): the first TEN samples whatever TEST_SAMPLES is -- identical to
        `pred` at the reference's TEST_SAMPLES = 10; `predict(x, samples, ensemble_first=10)` returns both."""
        sum_logp, sum_prob = self.sum_logp, self.sum_prob
        if self.pg is not None:
            both = torch.stack([sum_logp, sum_prob])
            torch.distributed.all_reduce(both, group=self.pg)
            sum_logp, sum_prob = both[0], both[1]
        mean_logp = sum_logp / total_samples
        probs = sum_prob / total_samples
        return {"mean_logp": mean_logp, "pred": mean_logp.argmax(1), "probs": probs,
                "entropy": -(probs * torch.log(probs)).sum(1)}


    def predict(self, x, samples, ensemble_first=10):
        """test_ensemble's per-batch statistics (MF:366-418) for `samples` MC weight samples on this rank's group:
        result(samples) plus `pred_first` = argmax of the mean of the FIRST `ensemble_first` samples' log-softmax outputs
        (`outputs[0:10].mean(0)`, MF:416-417).  Sample streams are keyed by the sample index, so the first-k statistics are
        those very samples: they are run first as their own (short) pass, then the whole range."""
        k = min(int(ensemble_first), int(samples))
        world = 1 if self.pg is None else torch.distributed.get_world_size(self.pg)
        rank = 0 if self.pg is None else torch.distributed.get_rank(self.pg)
        first, count = shard_samples(k, world, rank)
        self.run(x, count, first_sample=first)
        pred_first = self.result(k)["pred"]
        first, count = shard_samples(int(samples), world, rank)
        self.run(x, count, first_sample=first)
        out = self.result(int(samples))
        out["pred_first"] = pred_first
        return out


# ---- ensemble / sparsity statistics of the driver loops, on the parameters' device (SURVEY.md §8f rank 2) -------------------
# The reference computes these with a device -> host NumPy round trip per MC sample (MF:376-396, 427-433, 612-637).  They
# are plain reductions over the inclusion probabilities and Bernoulli masks, so they stay torch expressions here (no
# custom kernel: nothing on the hot path), run wherever the parameters live and touch the host once, at the end.
def reference_param_groups(net):
    """The 33 optimizer groups of the MF script (MF:520-553), in its order: lr 1e-4 for bias_mu, bias_rho, weight_mu,
    weight_rho; 1e-3 for pa, pb; 1e-5 for weight_a, weight_b, bias_a, bias_b; 0.1 for lambdal.  Feed to torch.optim.Adam,
    lbbnn.MultiTensorAdam or GraphedTrainer(param_groups=..., lr=1e-4)."""
    groups = []
    for names, lr in ((("bias_mu", "bias_rho", "weight_mu", "weight_rho"), 1e-4), (("pa", "pb"), 1e-3),
                      (("weight_a", "weight_b", "bias_a", "bias_b"), 1e-5), (("lambdal",), 0.1)):
        for name in names:
            for l in net.layers:
                groups.append({"params": getattr(l, name), "lr": lr})
    return groups


def refresh_inclusion(net):
    """alpha = 1 / (1 + exp(-lambdal)) for every layer and its `.gamma`, and `.gamma.exact = True` -- what the driver does
    before `test_ensemble` (MF:612-625)."""
    with torch.no_grad():
        for l in net.layers:
            l.alpha = 1 / (1 + torch.exp(-l.lambdal.detach()))
            l.gamma.alpha = l.alpha
            l.gamma.exact = True
    return net


def median_probability_masks(net):
    """The median-probability model: one {0, 1} float mask [alpha > 0.5] per layer (the g1..g3 of `outofsample(medimod=True)`,
    MF:462-465)."""
    return [(l.alpha.detach() > 0.5).to(l.alpha.dtype) for l in net.layers]


def median_probability_density(net):
    """Fraction of weights whose inclusion probability exceeds 0.5 (`os`, MF:634-637), as a 0-dim tensor on the device."""
    tot = sum(l.alpha.numel() for l in net.layers)
    return sum((l.alpha.detach() > 0.5).sum() for l in net.layers).to(torch.float64) / tot


def mask_statistics(net, samples, draws=None):
    """`spars / ctr`, `ps` and `np.mean(density)` of `test_ensemble` (MF:376-396, 427-433) for one test batch: per MC sample
    the reference draws one set of masks for the sparsity / ever-active counters and ANOTHER set for `density` (the
    forward uses a third).  draws[i] = (masks_a, masks_b) injects them (lists of per-layer tensors); None = Bernoulli(alpha)
    on the device.  Returns 0-dim float64 device tensors {"sparsity", "ever_active", "density"}; `ever_active` is the
    reference's `ps` without its hard-coded division by the 10 test batches."""
    layers = list(net.layers)
    tot = sum(l.alpha.numel() for l in layers)
    dev = layers[0].alpha.device
    spars = torch.zeros((), dtype=torch.float64, device=dev)
    dens = torch.zeros((), dtype=torch.float64, device=dev)
    ever = [torch.zeros_like(l.alpha, dtype=torch.bool) for l in layers]
    with torch.no_grad():
        for i in range(samples):
            ga = draws[i][0] if draws is not None else [torch.bernoulli(l.alpha) for l in layers]
            gb = draws[i][1] if draws is not None else [torch.bernoulli(l.alpha) for l in layers]
            on = [g > 0.5 for g in ga]
            spars += sum(o.sum() for o in on).to(torch.float64) / tot
            ever = [e | o for e, o in zip(ever, on)]
            dens += torch.cat([g.flatten() for g in gb]).mean().to(torch.float64)
    return {"sparsity": spars / samples, "ever_active": sum(e.sum() for e in ever).to(torch.float64) / tot,
            "density": dens / samples}


class _null_ctx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def shard_samples(total, world, rank):
    """Contiguous split of the MC sample indices [0, total) across ranks: (first, count)."""
    base, rem = divmod(total, world)
    first = rank * base + min(rank, rem)
    return first, base + (1 if rank < rem else 0)
