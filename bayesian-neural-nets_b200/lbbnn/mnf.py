"""Drop-in MNF layer and network (reference LBBNN-GP-MF-MNF.py:133-260; sim-study parametrisation
LBBNN-GP-MF-MNFsim_study.py:145-251 through the prior / init keyword arguments).

What runs where: the z flows and the auxiliary r flow -> fused flow kernels (flows.py); the activation
path mm(x*z, M^T), mm(x^2, V^T), eps/sqrt -> the fused LRT kernels with z folded into the weight prologue
(MNF:197-198: mm(x*z, M^T) == mm(x, (M*z)^T) because z is a single (in,) vector); the KL over all weights
with (mu*z2 - mu_p)^2 (MNF:230-233) and the W_mean/W_var moments -> prologue/finalize kernels; log q0, the two
auxiliary GEMVs r0_c @ W^T (MNF:216-217), tanh, the outer-product means and log r_b -> one fused forward and one
fused backward kernel (csrc/mnf_aux.cu).  Only z0 = q0_mean + sqrt(exp(q0_log_var)) eps and the final scalar sum
stay in torch.

Reference quirks kept (SURVEY.md §0 #4): one z (the last batch row's) is broadcast over the batch, so only
that row is pushed through the flow; the KL branch draws its own z (self.z becomes (1,in)); z_b[-1] in
log r_b is the last ELEMENT of the flowed vector; log pi (not log 2 pi) in both Gaussians.
"""
import ctypes as C
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi as K
from .flows import PropagateFlow, _build_flow
from .lrt import BernoulliView, GaussianView, LayerConfig, _LRTFunction, current_seed, _layer_ids


class _MomentsKL(torch.autograd.Function):
    """(M0 = alpha mu, V = sigma^2 alpha^2, kl(weights with mu*z_kl, biases)) and their gradients."""

    @staticmethod
    def forward(ctx, wmu, wrho, lam, bmu, brho, z_kl, cfg):
        K.require_device()
        ps = [t.contiguous() for t in (wmu, wrho, lam, bmu, brho)]
        zc = z_kl.contiguous()
        layer = K.make_layer(*ps, None, zc)
        M, V = torch.empty_like(ps[0]), torch.empty_like(ps[0])
        kl = torch.zeros((), dtype=torch.float32, device=wmu.device)
        ws = K.workspace(1 << 20, wmu.device)
        K.check(K.lib.lbbnn_lrt_f32_prologue(layer, cfg.priors, cfg.var_mode, K.FLAG_SAMPLE, K.ptr(M), K.ptr(V), K.ptr(kl),
                                             ws.data_ptr(), ws.numel(), K.current_stream()))
        ctx.save_for_backward(*ps, zc)
        ctx.cfg = cfg
        return M, V, kl

    @staticmethod
    def backward(ctx, dM, dV, dkl):
        wmu, wrho, lam, bmu, brho, z = ctx.saved_tensors
        cfg = ctx.cfg
        layer = K.make_layer(wmu, wrho, lam, bmu, brho, None, z)
        dM = torch.zeros_like(wmu) if dM is None else dM.contiguous()
        dV = torch.zeros_like(wmu) if dV is None else dV.contiguous()
        colsum = torch.zeros(2 * wmu.shape[0], dtype=torch.float32, device=wmu.device)
        grads = [torch.empty_like(t) for t in (wmu, wrho, lam, bmu, brho)]
        dz = torch.zeros_like(z)
        use_kl = dkl is not None
        g = K.LayerGrads(*[K.ptr(t) for t in grads], None, K.ptr(dz))
        K.check(K.lib.lbbnn_lrt_f32_finalize(layer, K.ptr(dM), K.ptr(dV), K.ptr(colsum), cfg.priors, cfg.var_mode,
                                             K.FLAG_SAMPLE, K.ptr(dkl.contiguous().float()) if use_kl else None,
                                             1.0 if use_kl else 0.0, g, K.current_stream()))
        return (*grads, dz, None)


class _AuxKL(torch.autograd.Function):
    """log_q0 - log_rb of the KL branch (MNF:212-227 minus the flows) in one forward and one backward kernel
    (csrc/mnf_aux.cu).  Inputs: q0_mean, q0_log_var, z0 (the KL row's pre-flow draw), r0_c, r0_b1, r0_b2, z2 (its flow
    image), M0 = alpha mu, V, eps_r, z_b = r_flow(z2)."""

    @staticmethod
    def forward(ctx, q0_mean, q0_log_var, z0, r0_c, r0_b1, r0_b2, z2, M0, V, eps_r, z_b, ticket):
        K.require_device()
        ts = [t.contiguous() for t in (q0_mean, q0_log_var, z0, r0_c, r0_b1, r0_b2, z2, M0, V, eps_r, z_b)]
        O, D = ts[7].shape
        dev = ts[7].device
        out = torch.empty(3, dtype=torch.float32, device=dev)
        save = torch.empty(int(K.lib.lbbnn_mnf_aux_save_floats(O)), dtype=torch.float32, device=dev)
        aux = K.MnfAux(D, O, *[K.ptr(t) for t in ts])
        K.check(K.lib.lbbnn_mnf_aux_kl_fwd(aux, K.ptr(out), K.ptr(save), ticket.data_ptr(), K.current_stream()))
        ctx.save_for_backward(*ts, save)
        ctx.shapes = [t.shape for t in (q0_mean, q0_log_var, z0, r0_c, r0_b1, r0_b2, z2, z_b)]
        return out[0]

    @staticmethod
    def backward(ctx, g):
        *ts, save = ctx.saved_tensors
        O, D = ts[7].shape
        dev = ts[7].device
        vec = torch.empty(8, D, dtype=torch.float32, device=dev)
        dM0, dV = torch.empty_like(ts[7]), torch.empty_like(ts[8])
        aux = K.MnfAux(D, O, *[K.ptr(t) for t in ts])
        grads = K.MnfAuxGrads(*[vec[i].data_ptr() for i in range(8)], K.ptr(dM0), K.ptr(dV))
        K.check(K.lib.lbbnn_mnf_aux_kl_bwd(aux, K.ptr(save), K.ptr(g.contiguous().float()), grads, K.current_stream()))
        v = [vec[i].view(ctx.shapes[i]) for i in range(8)]
        #      q0_mean q0_lv z0    r0_c  b1    b2    z2    M0   V   eps_r z_b  ticket
        return v[0], v[1], v[2], v[3], v[4], v[5], v[6], dM0, dV, None, v[7], None


_N_LAYER_PARAMS = 10      # weight_mu, weight_rho, lambdal, bias_mu, bias_rho, q0_mean, q0_log_var, r0_c, r0_b1, r0_b2
_zero_colsums = {}


def _zeros_const(n, dev):
    """A never-written zero buffer (the weight-KL finalize's `colsum` input: the KL branch has no activation gradient)."""
    key = (dev.index, n)
    t = _zero_colsums.get(key)
    if t is None:
        if torch.cuda.is_current_stream_capturing():
            raise K.LbbnnError("constant buffer would be created during CUDA-graph capture; run one eager step first")
        t = torch.zeros(n, dtype=torch.float32, device=dev)
        _zero_colsums[key] = t
    return t


def _flow_grad_table(flow, params, gbuf):
    """lbbnn_flow_grads over a (rows, P) buffer laid out like `params` (PropagateFlow._params() order); returns it with
    the per-parameter offsets."""
    sizes = [p.numel() for p in params]
    offs = [0]
    for n in sizes:
        offs.append(offs[-1] + n)
    grads = K.FlowGrads()
    grads.row_stride = gbuf.shape[1]
    base = gbuf.data_ptr()
    i = 0
    for t in range(flow.n_transforms):
        for l in range(flow.n_hidden):
            grads.t[t].hidden[l].dW, grads.t[t].hidden[l].db = base + 4 * offs[i], base + 4 * offs[i + 1]
            i += 2
        grads.t[t].shift.dW, grads.t[t].shift.db = base + 4 * offs[i], base + 4 * offs[i + 1]
        grads.t[t].scale.dW, grads.t[t].scale.db = base + 4 * offs[i + 2], base + 4 * offs[i + 3]
        i += 4
    return grads, offs


class _ZDraw(torch.autograd.Function):
    """The z0 draw (MNF:183-185) and the z flow (MNF:186-189) of one layer call, both rows in ONE launch each: row 0 is the
    activation's z (the last batch row's draw, SURVEY quirk #4), row 1 -- training / calculate_log_probs -- the KL branch's
    own sample_z() (MNF:210).  Returns (z_k, z2, log_det_q of row 1, z0 row 1 = what the reference leaves in self.z,
    aliases of q0_mean and q0_log_var for the KL branch) or, without the KL row, (z_k, z0 row 0)."""

    @staticmethod
    def forward(ctx, meta, q0m, q0lv, *zp):
        K.require_device()
        layer, want_kl, nz = meta
        q0m, q0lv = q0m.contiguous(), q0lv.contiguous()
        zp = [p.contiguous() for p in zp]
        dev, D = q0m.device, layer.in_features
        f32 = dict(dtype=torch.float32, device=dev)
        st = K.current_stream()
        R = 2 if want_kl else 1
        inj = "eps_z" in nz
        layer._prep_calls += 1
        skey = (layer._uid << 40) | (1 << 39) | (layer._prep_calls << 2)
        if inj:
            eps_rows = torch.cat([nz["eps_z"][-1:], nz["eps_z2"]], 0) if want_kl else nz["eps_z"][-1:]
            noise_z = K.make_noise(eps_rows.contiguous())
        else:
            noise_z = K.make_noise(None, current_seed(), skey)
        eps, z0 = torch.empty(R, D, **f32), torch.empty(R, D, **f32)
        K.check(K.lib.lbbnn_mnf_draw(K.ptr(q0m), K.ptr(q0lv), noise_z, R, D, K.ptr(eps), K.ptr(z0), None, 0, None, st))
        zf = layer.z_flow
        masks = None
        if inj:
            rows = [[m[-1:] for m in nz["z_masks"]]] + ([list(nz["z_masks2"])] if want_kl else [])
            masks = torch.stack([torch.cat([r[t].reshape(1, D) for r in rows], 0) for t in range(len(rows[0]))]).contiguous()
        key = zf._next_key()
        flow = _build_flow(zf.kind, D, len(zf.transforms), zf.n_hidden, zp)
        zs, ld = torch.empty(R, D, **f32), torch.empty(R, **f32)
        save = torch.empty(int(K.lib.lbbnn_flow_save_floats(flow, R)), **f32)
        K.check(K.lib.lbbnn_flow_fwd(flow, K.ptr(z0), R, K.ptr(masks, allow_none=True), K.make_noise(None, *key), K.ptr(zs),
                                     K.ptr(ld), K.ptr(save), st))
        ctx.meta = (layer, want_kl, key)
        ctx.save_for_backward(q0lv, eps, masks, save, *zp)
        if not want_kl:
            z_row = z0[:1]
            ctx.mark_non_differentiable(z_row)
            return zs[0], z_row
        # q0_mean / q0_log_var for the KL branch pass through this node: their gradients from there arrive HERE and are
        # added inside mnf_draw_bwd (aux_d_q0_*), instead of as two accumulation kernels at the very end of the backward
        return zs[0], zs[1], ld[1:], z0[1:2], q0m.view_as(q0m), q0lv.view_as(q0lv)

    @staticmethod
    def backward(ctx, d_zk, *rest):
        layer, want_kl, key = ctx.meta
        q0lv, eps, masks, save, *zp = ctx.saved_tensors
        zf = layer.z_flow
        dev, D = q0lv.device, layer.in_features
        f32 = dict(dtype=torch.float32, device=dev)
        st = K.current_stream()
        R = 2 if want_kl else 1
        flow = _build_flow(zf.kind, D, len(zf.transforms), zf.n_hidden, zp)
        gz = torch.empty(R, sum(p.numel() for p in zp), **f32)
        gt, offs = _flow_grad_table(flow, zp, gz)
        dz0 = torch.empty(R, D, **f32)
        d_mean, d_lv = torch.empty(D, **f32), torch.empty(D, **f32)
        cz = lambda t: None if t is None else t.contiguous()
        d_zk = cz(d_zk)
        if not want_kl:
            rows = d_zk.reshape(1, D) if d_zk is not None else torch.zeros(1, D, **f32)
            dld, d_z0row, d_q0m_kl, d_q0lv_kl = None, None, None, None
        else:
            d_z2, d_ld, d_z0row, d_q0m_kl, d_q0lv_kl = (cz(t) for t in rest)
            rows, dld = torch.empty(2, D, **f32), torch.empty(2, **f32)
            if d_ld is None:
                dld.zero_()
            K.check(K.lib.lbbnn_mnf_bwd_rows(K.ptr(d_ld, allow_none=True), 1.0, K.ptr(dld) if d_ld is not None else None,
                                             K.ptr(d_zk, allow_none=True), K.ptr(d_z2, allow_none=True), None, D, K.ptr(rows), st))
        K.check(K.lib.lbbnn_flow_bwd(flow, gt, R, K.ptr(masks, allow_none=True), K.make_noise(None, *key), K.ptr(rows),
                                     K.ptr(dld, allow_none=True), K.ptr(save), K.ptr(dz0), st))
        K.check(K.lib.lbbnn_mnf_draw_bwd(K.ptr(q0lv), K.ptr(eps), K.ptr(dz0), R, D, 1 if want_kl else -1,
                                         K.ptr(d_q0m_kl, allow_none=True), K.ptr(d_q0lv_kl, allow_none=True),
                                         K.ptr(d_z0row, allow_none=True), K.ptr(d_mean), K.ptr(d_lv), st))
        gzs = gz[0] + gz[1] if R == 2 else gz[0]
        return (None, d_mean, d_lv, *[gzs[offs[j]:offs[j + 1]].view_as(zp[j]) for j in range(len(zp))])


class _KLBranch(torch.autograd.Function):
    """The KL branch of one layer call after its z draw (MNF:211-235) as ONE autograd node: weight moments + weight / bias KL
    with the KL row's z2, the auxiliary r flow on z2, log q0 - log r_b, and the combination into the layer's kl.  Nothing
    here depends on the input batch, so network forward and backward run it on a side stream under the activation path.
    Forward = 5 launches, backward = 5 (one autograd node per piece: ~40 per layer, mostly elementwise glue)."""

    @staticmethod
    def forward(ctx, meta, wmu, wrho, lam, bmu, brho, q0m, q0lv, r0c, rb1, rb2, z2, ld_q, z0row, *rp):
        K.require_device()
        layer, nz = meta
        ts = [t.contiguous() for t in (wmu, wrho, lam, bmu, brho, q0m, q0lv, r0c, rb1, rb2, z2, ld_q, z0row)]
        wmu, wrho, lam, bmu, brho, q0m, q0lv, r0c, rb1, rb2, z2, ld_q, z0row = ts
        rp = [p.contiguous() for p in rp]
        dev, D, O = wmu.device, layer.in_features, layer.out_features
        f32 = dict(dtype=torch.float32, device=dev)
        st = K.current_stream()
        # ---- weight moments + weight / bias KL with the KL row's z (MNF:211, 228-234)
        M0, V = torch.empty_like(wmu), torch.empty_like(wmu)
        kls, out3 = torch.empty(2, **f32), torch.empty(3, **f32)     # kls = [kl_wb, kl]
        ws = K.workspace(1 << 20, dev)
        lay = K.make_layer(wmu, wrho, lam, bmu, brho, None, z2)
        K.check(K.lib.lbbnn_lrt_f32_prologue(lay, layer.cfg.priors, layer.cfg.var_mode, K.FLAG_SAMPLE, K.ptr(M0), K.ptr(V),
                                             kls.data_ptr(), ws.data_ptr(), ws.numel(), st))
        # ---- auxiliary r flow on z2 (MNF:222-223); eps_r (MNF:218) rides in the flow-independent draw kernel's second half
        rf = layer.r_flow
        masks_r = torch.stack([m.reshape(1, D) for m in nz["r_masks"]]).contiguous() if "r_masks" in nz else None
        key_r = rf._next_key()
        flow_r = _build_flow(rf.kind, D, len(rf.transforms), rf.n_hidden, rp)
        z_b, ld_r = torch.empty(1, D, **f32), torch.empty(1, **f32)
        save_r = torch.empty(int(K.lib.lbbnn_flow_save_floats(flow_r, 1)), **f32)
        K.check(K.lib.lbbnn_flow_fwd(flow_r, K.ptr(z2), 1, K.ptr(masks_r, allow_none=True), K.make_noise(None, *key_r),
                                     K.ptr(z_b), K.ptr(ld_r), K.ptr(save_r), st))
        if "eps_r" in nz:
            eps_r = nz["eps_r"].contiguous()
        else:
            eps_r = torch.empty(O, **f32)
            skey = (layer._uid << 40) | (1 << 39) | (layer._prep_calls << 2) | 1
            K.check(K.lib.lbbnn_philox_normal_ex(K.ptr(eps_r), O, K.make_noise(None, current_seed(), skey), st))
        # ---- log q0 - log r_b (MNF:212-227) and the layer's kl (MNF:235)
        if layer._aux_ticket is None or layer._aux_ticket.device != dev:
            layer._aux_ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        save_a = torch.empty(int(K.lib.lbbnn_mnf_aux_save_floats(O)), **f32)
        aux = K.MnfAux(D, O, K.ptr(q0m), K.ptr(q0lv), K.ptr(z0row), K.ptr(r0c), K.ptr(rb1), K.ptr(rb2), K.ptr(z2), K.ptr(M0), K.ptr(V),
                       K.ptr(eps_r), K.ptr(z_b))
        K.check(K.lib.lbbnn_mnf_aux_kl_fwd(aux, K.ptr(out3), K.ptr(save_a), layer._aux_ticket.data_ptr(), st))
        K.check(K.lib.lbbnn_mnf_kl_combine(kls.data_ptr(), out3.data_ptr(), K.ptr(ld_q), K.ptr(ld_r), kls[1:].data_ptr(), st))
        ctx.meta = (layer, key_r)
        ctx.save_for_backward(*ts, *rp, M0, V, eps_r, z_b, masks_r, save_r, save_a)
        return kls[1]

    @staticmethod
    def backward(ctx, d_kl):
        layer, key_r = ctx.meta
        saved = ctx.saved_tensors
        wmu, wrho, lam, bmu, brho, q0m, q0lv, r0c, rb1, rb2, z2, ld_q, z0row = saved[:13]
        M0, V, eps_r, z_b, masks_r, save_r, save_a = saved[-7:]
        rp = saved[13:-7]
        rf = layer.r_flow
        dev, D, O = wmu.device, layer.in_features, layer.out_features
        f32 = dict(dtype=torch.float32, device=dev)
        st = K.current_stream()
        g = d_kl.reshape(1).contiguous().float()
        neg = torch.empty(2, **f32)                                  # [0, -g]: d kl / d log_det_q = d kl / d log_det_r = -1
        K.check(K.lib.lbbnn_mnf_bwd_rows(K.ptr(g), -1.0, K.ptr(neg), None, None, None, D, None, st))
        # auxiliary term: every direct gradient + the rank-one dM0, dV
        vec = torch.empty(8, D, **f32)
        dM0, dV = torch.empty_like(M0), torch.empty_like(V)
        aux = K.MnfAux(D, O, K.ptr(q0m), K.ptr(q0lv), K.ptr(z0row), K.ptr(r0c), K.ptr(rb1), K.ptr(rb2), K.ptr(z2), K.ptr(M0), K.ptr(V),
                       K.ptr(eps_r), K.ptr(z_b))
        ag = K.MnfAuxGrads(*[vec[i].data_ptr() for i in range(8)], K.ptr(dM0), K.ptr(dV))
        K.check(K.lib.lbbnn_mnf_aux_kl_bwd(aux, K.ptr(save_a), K.ptr(g), ag, st))
        # r flow: d z_b from the auxiliary term, d log_det_r = -g
        flow_r = _build_flow(rf.kind, D, len(rf.transforms), rf.n_hidden, rp)
        gr = torch.empty(1, sum(p.numel() for p in rp), **f32)
        grt, roffs = _flow_grad_table(flow_r, rp, gr)
        dzr = torch.empty(1, D, **f32)
        K.check(K.lib.lbbnn_flow_bwd(flow_r, grt, 1, K.ptr(masks_r, allow_none=True), K.make_noise(None, *key_r),
                                     vec[7].data_ptr(), neg[1:].data_ptr(), K.ptr(save_r), K.ptr(dzr), st))
        # d z2 = auxiliary + r flow, then the weight KL's share accumulated on top by the finalize pass
        rows = torch.empty(2, D, **f32)
        K.check(K.lib.lbbnn_mnf_bwd_rows(None, 0.0, None, None, vec[6].data_ptr(), K.ptr(dzr), D, K.ptr(rows), st))
        grads = [torch.empty_like(t) for t in (wmu, wrho, lam, bmu, brho)]
        lay = K.make_layer(wmu, wrho, lam, bmu, brho, None, z2)
        lg = K.LayerGrads(*[K.ptr(t) for t in grads], None, rows[1].data_ptr())
        K.check(K.lib.lbbnn_lrt_f32_finalize(lay, K.ptr(dM0), K.ptr(dV), K.ptr(_zeros_const(2 * O, dev)), layer.cfg.priors,
                                             layer.cfg.var_mode, K.FLAG_SAMPLE, K.ptr(g), 1.0, lg, st))
        grp = [gr[0, roffs[j]:roffs[j + 1]].view_as(rp[j]) for j in range(len(rp))]
        #       meta  5 LRT params  q0_mean  q0_log_var  r0_c  r0_b1  r0_b2   z2      ld_q     z0 row
        return (None, *grads, vec[0], vec[1], vec[3], vec[4], vec[5], rows[1], neg[1:], vec[2].view(1, D), *grp)


class BayesianLinear(nn.Module):
    """MNF layer, drop-in for LBBNN-GP-MF-MNF.py:133-239: ctor `(in_features, out_features, num_transforms)`.
    `noise=` on forward injects the draws of SURVEY.md §3.2 (see tests/cases.py:mnf_noise)."""

    def __init__(self, in_features, out_features, num_transforms=2, *, device=None, mu_prior=0.0, sigma_prior=1.0,
                 alpha_prior=0.05, bias_mu_prior=0.0, bias_sigma_prior=1.0, mu_init=0.01, lambda_init=(0.0, 1.0),
                 z_flow_type="RNVP", r_flow_type="RNVP", h_sizes=(75, 75, 75, 75)):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        E = torch.empty
        self.weight_mu = nn.Parameter(E(out_features, in_features).uniform_(-mu_init, mu_init))
        self.weight_rho = nn.Parameter(E(out_features, in_features).uniform_(-5, -4))
        self.lambdal = nn.Parameter(E(out_features, in_features).uniform_(*lambda_init))
        E(out_features, in_features).uniform_(0.999, 0.9999)            # the reference's alpha_q draw (MNF:149)
        self.bias_mu = nn.Parameter(E(out_features).uniform_(-0.2, 0.2))
        self.bias_rho = nn.Parameter(E(out_features).uniform_(-5, -4))
        self.q0_mean = nn.Parameter(0.1 * torch.randn(in_features))
        self.q0_log_var = nn.Parameter(-9 + 0.1 * torch.randn(in_features))
        self.r0_c = nn.Parameter(0.1 * torch.randn(in_features))
        self.r0_b1 = nn.Parameter(0.1 * torch.randn(in_features))
        self.r0_b2 = nn.Parameter(0.1 * torch.randn(in_features))
        self.z_flow = PropagateFlow(z_flow_type, in_features, num_transforms, h_sizes)
        self.r_flow = PropagateFlow(r_flow_type, in_features, num_transforms, h_sizes)
        self.cfg = LayerConfig(mu_prior, sigma_prior, alpha_prior, bias_mu_prior, bias_sigma_prior)
        self.weight = GaussianView(self.weight_mu, self.weight_rho)
        self.bias = GaussianView(self.bias_mu, self.bias_rho)
        self.gamma = BernoulliView(self)
        self.kl = 0
        self.z = 0
        self._uid = next(_layer_ids)
        self._calls = 0
        self._prep_calls = 0
        self.last_noise_key = None
        self._aux_ticket = None
        if device is not None:
            self.to(device)

    @property
    def alpha_q(self):
        return 1 / (1 + torch.exp(-self.lambdal.detach()))

    def _z0(self, eps):
        return self.q0_mean + self.q0_log_var.exp().sqrt() * eps       # MNF:183-185

    def _draw(self, want_kl, nz):
        """z0 draw + z flow of this call (one autograd node); returns the handle _kl_branch() continues from."""
        out = _ZDraw.apply((self, bool(want_kl), nz), self.q0_mean, self.q0_log_var, *self.z_flow._params())
        self.z = out[3] if want_kl else out[-1]                         # sample_z() leaves its last draw in self.z
        return out

    def _kl_branch(self, drawn, nz):
        """The layer's kl from the KL row of _draw() (one autograd node)."""
        _, z2, ld_q, z0row, q0_mean, q0_log_var = drawn
        return _KLBranch.apply((self, nz), *self._lrt_params(), q0_mean, q0_log_var, self.r0_c, self.r0_b1, self.r0_b2,
                               z2, ld_q, z0row, *self.r_flow._params())

    def _lrt_params(self):
        """weight_mu, weight_rho, lambdal, bias_mu, bias_rho as the KL branch and the activation kernels take them: the
        parameters themselves, or the aliases BayesianNetwork._logits made on the layer's accumulation stream -- the two
        gradient contributions of each (KL branch, activation path) are then summed THERE, not on the streams that carry the
        flows' backward."""
        shared = getattr(self, "_shared", None)
        return shared if shared is not None else (self.weight_mu, self.weight_rho, self.lambdal, self.bias_mu, self.bias_rho)

    def _prepare(self, want_kl, nz):
        """Everything of forward() that does not depend on the input batch: the z flow on the live rows, and (training /
        calculate_log_probs) the whole KL branch with the auxiliary r flow.  Returns (z_k, kl or 0)."""
        drawn = self._draw(want_kl, nz)
        return drawn[0], (self._kl_branch(drawn, nz) if want_kl else 0)

    def _activation(self, input, z_k, sample_branch, nz, relu=False, mask_dx=False):
        self._calls += 1
        self.last_noise_key = (current_seed(), (self._uid << 40) | self._calls)
        act, _ = _LRTFunction.apply(input, *self._lrt_params(), z_k,
                                    nz.get("eps"), self.cfg, sample_branch, False, self.last_noise_key, relu, mask_dx)
        return act

    def forward(self, input, sample=False, calculate_log_probs=False, noise=None):
        nz = noise or {}
        z_k, self.kl = self._prepare(self.training or calculate_log_probs, nz)
        return self._activation(input, z_k, self.training or sample, nz)


class BayesianNetwork(nn.Module):
    """784-400-600-10 MNF network, drop-in for LBBNN-GP-MF-MNF.py:244-260."""

    def __init__(self, sizes=(28 * 28, 400, 600, 10), num_transforms=2, **layer_kwargs):
        super().__init__()
        self.sizes = tuple(sizes)
        for n, (i, o) in enumerate(zip(sizes[:-1], sizes[1:]), 1):
            setattr(self, f"l{n}", BayesianLinear(i, o, num_transforms=num_transforms, **layer_kwargs))
        self._names = [f"l{n}" for n in range(1, len(sizes))]
        self._streams = None
        self._acc_streams = None

    @property
    def layers(self):
        return [getattr(self, n) for n in self._names]

    def forward(self, x, sample=False, noises=None, calculate_log_probs=False):
        return F.log_softmax(self._logits(x, sample, noises, calculate_log_probs), dim=1)

    def _logits(self, x, sample=False, noises=None, calculate_log_probs=False):
        """forward() without the closing log_softmax (the trainers fuse it with the loss).
        The flows and the KL branch of a layer depend on parameters and noise only, never on the activations.  Every
        layer gets its own CUDA stream: the z draw + z flow first (the activation path only waits for THAT), then the KL
        branch (weight KL, auxiliary r flow, log q0 - log r_b), which runs under the LRT layers of the caller's stream --
        and, because autograd replays a node on its forward stream, so does its backward.  Inside a captured graph these
        are parallel branches."""
        x = x.view(-1, self.sizes[0])
        ls = self.layers
        nzs = [(None if noises is None else noises[i]) or {} for i in range(len(ls))]
        cur = torch.cuda.current_stream()
        if self._streams is None or self._streams[0].device != x.device:
            self._streams = [torch.cuda.Stream(device=x.device) for _ in ls]
            self._acc_streams = [torch.cuda.Stream(device=x.device) for _ in ls]
        for s in self._streams:
            s.wait_stream(cur)
        # One alias per shared parameter and layer, made on that layer's ACCUMULATION stream: autograd sums the KL branch's
        # and the activation path's gradients at the alias node, i.e. on that stream.  Summed at the leaf they ran on the
        # layer's flow stream between the activation path's finalize and the z flow's backward -- five dependent ~3 us
        # launches on the step's critical tail (profiles/r02_timeline_mnf.txt).  LBBNN_MNF_SHARE=0 keeps the leaf accumulation.
        share = torch.is_grad_enabled() and os.environ.get("LBBNN_MNF_SHARE", "1") == "1"
        for l, sa in zip(ls, self._acc_streams):
            l._shared = None
            if share and (l.training or calculate_log_probs):
                sa.wait_stream(cur)
                with torch.cuda.stream(sa):
                    l._shared = tuple(p.view_as(p) for p in (l.weight_mu, l.weight_rho, l.lambdal, l.bias_mu, l.bias_rho))
        # issue order (same dependency graph either way; same-box A/B of the captured step, ms: 0.32-0.335 against 0.366-0.368
        # when each layer's KL branch is issued after that layer's activation kernels): every layer's draw + KL branch first
        interleave = os.environ.get("LBBNN_MNF_ORDER") == "layer"
        drawn = []
        for l, s, nz in zip(ls, self._streams, nzs):
            want_kl = l.training or calculate_log_probs
            with torch.cuda.stream(s):
                d = l._draw(want_kl, nz)
                ev = torch.cuda.Event()
                ev.record(s)
                if not interleave:
                    l.kl = l._kl_branch(d, nz) if want_kl else 0
            drawn.append((d, ev))
        for i, (l, s, nz) in enumerate(zip(ls, self._streams, nzs)):
            cur.wait_event(drawn[i][1])
            z_k = drawn[i][0][0]
            z_k.record_stream(cur)
            # F.relu (MNF:252-253) rides in the layer kernels: forward flag here, its backward as the next layer's dx mask
            x = l._activation(x, z_k, l.training or sample, nz, relu=i < len(ls) - 1, mask_dx=i > 0)
            if interleave:
                with torch.cuda.stream(s):
                    l.kl = l._kl_branch(drawn[i][0], nz) if (l.training or calculate_log_probs) else 0
        for l, s, sa in zip(ls, self._streams, self._acc_streams):
            cur.wait_stream(s)
            if l._shared is not None:
                cur.wait_stream(sa)
            l._shared = None
            if torch.is_tensor(l.kl):
                l.kl.record_stream(cur)
        return x

    def kl(self):
        return sum(l.kl for l in self.layers)

    def late_grad_params(self):
        """The parameters whose gradients are produced by the LAST node of a backward pass -- the first layer's z draw + z
        flow (it waits for that layer's dz from the activation path, which finishes last): MultiTensorAdam.set_late_params
        updates everything else while that node runs."""
        l = self.layers[0]
        return [l.q0_mean, l.q0_log_var, *l.z_flow.parameters()]


# the sim study's layer (MNFsim:145-251 through BayesianLinear's keyword arguments; flows_simstudy hidden sizes [50] * 5)
SIM_LAYER_DEFAULTS = dict(mu_prior=0.1, sigma_prior=1.3, alpha_prior=0.3, bias_sigma_prior=1.3, lambda_init=(1.5, 2.5),
                          h_sizes=(50,) * 5)


class SimStudyNetwork(nn.Module):
    """The MNF simulation-study model (LBBNN-GP-MF-MNFsim_study.py): one MNF layer in_features -> 1 with two RNVP
    transforms per flow, as a logistic regression.  `layer_kwargs` override SIM_LAYER_DEFAULTS (and num_transforms).

    Stated assumption: the reference script is not part of this project, and what is recorded of it is the model ("MNF
    layer as 20 -> 1 logistic regression"), its `train` (MNFsim:272-298) and an LR-staged Adam (MNFsim:321-384).  The
    objective below is therefore the mean-field study's (sigmoid output and BCELoss(sum), MFsim:258, 287) with the MNF
    layer's kl in place of log q - log p, in the MNF script's train form (MNF:263-275):
    loss = BCE(sigmoid(l1(x)), y, sum) + kl / num_batches."""

    def __init__(self, in_features=20, num_batches=5.0, **layer_kwargs):
        super().__init__()
        kw = dict(SIM_LAYER_DEFAULTS)
        kw.update(layer_kwargs)
        num_transforms = kw.pop("num_transforms", 2)
        self.l1 = BayesianLinear(in_features, 1, num_transforms, **kw)
        self.num_batches = num_batches

    def forward(self, x, sample=False, noise=None):
        return torch.sigmoid(self.l1(x, sample, noise=noise))

    def kl(self):
        return self.l1.kl

    def loss(self, x, y, noise=None):
        """One training objective on a minibatch (sampled forward, kl computed).  Returns (loss, nll, kl)."""
        out = torch.sigmoid(self.l1(x, True, calculate_log_probs=True, noise=noise))
        nll = F.binary_cross_entropy(out, y.reshape(out.shape).to(out.dtype), reduction="sum")
        kl = self.kl()
        return nll + kl / self.num_batches, nll, kl


# the ten layer tensors in the packed order of lbbnn_mnfsim (include/lbbnn.h), then the two flows: the 12 Adam groups
SIM_LAYER_NAMES = ("weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho", "q0_mean", "q0_log_var", "r0_c", "r0_b1", "r0_b2")
SIM_GROUPS = SIM_LAYER_NAMES + ("z_flow", "r_flow")
_SIM_NOISE = ("eps_z", "eps_z2", "z_masks", "z_masks2", "r_masks", "eps", "eps_r")


def _flow_arch(flow):
    """(kind, number of transforms, hidden widths) of a PropagateFlow."""
    hidden, _, _ = flow.transforms[0].linears()
    return flow.kind, len(flow.transforms), tuple(m.out_features for m in hidden)


class SimStudyEnsemble:
    """Every repetition of the MNF simulation study trained in ONE kernel launch (csrc/mnf_sim.cu): R SimStudyNetwork
    replicas, each running the sampled forward, kl, loss = nll + kl / num_batches, its backward and torch.optim.Adam (betas
    (0.9, 0.999), eps 1e-8, one learning rate per group) for whole epochs over minibatches of `batch_size` consecutive rows.

    The replicas' parameters live in one packed (R, P) device buffer `flat` (ten layer tensors, then the z flow's and the r
    flow's parameters); every nn.Parameter is re-pointed at a view of it (and, with materialize_grads, its .grad at the
    last step's gradients), so state_dict() and the eager SimStudyNetwork.loss keep working on each replica.  The Adam state
    is public: exp_avg, exp_avg_sq (laid out like `flat`) and the (R,) int64 step counts; it carries over between run()
    calls, so a staged learning-rate schedule is a sequence of run(epochs, lrs=...) calls.
    X is (n, in) shared by every replica or (R, n, in); y the {0, 1} targets (n,) or (R, n).  lrs: one float for every
    group, or a dict over all 12 SIM_GROUPS.  Native noise is Philox keyed by (seed, replica, the replica's step, kind of
    draw); see include/lbbnn.h for the streams."""

    BETAS, EPS = (0.9, 0.999), 1e-8

    def __init__(self, nets, X, y, batch_size=400, lrs=1e-3, seed=0, materialize_grads=True):
        nets = list(nets)
        if not nets:
            raise K.LbbnnError("SimStudyEnsemble needs at least one network")
        layers = [n.l1 for n in nets]

        def signature(n):
            l = n.l1
            pr = l.cfg.priors
            return (l.in_features, l.out_features, _flow_arch(l.z_flow), _flow_arch(l.r_flow),
                    (pr.mu, pr.sigma, pr.alpha, pr.bias_mu, pr.bias_sigma), l.cfg.var_mode, float(n.num_batches))
        sig = signature(nets[0])
        if any(signature(n) != sig for n in nets[1:]):
            raise K.LbbnnError("the replicas differ in shape, priors, flows (kind, transforms, hidden sizes) or num_batches")
        in_f, out_f, zarch, rarch, _, var_mode, num_batches = sig
        if out_f != 1 or not 1 <= in_f <= K.MNFSIM_MAX_IN:
            raise K.LbbnnError(f"the kernel trains in_features <= {K.MNFSIM_MAX_IN} -> 1 layers, got {in_f} -> {out_f}")
        if zarch != rarch or zarch[0] != K.FLOW_RNVP:
            raise K.LbbnnError("the z and r flows must be RNVP flows of one architecture (IAF flows are not supported)")
        _, T, hidden = zarch
        if T > K.MNFSIM_MAX_T or max(hidden) > K.MNFSIM_MAX_H or len(hidden) > K.FLOW_MAX_HIDDEN:
            raise K.LbbnnError(f"flows limited to {K.MNFSIM_MAX_T} transforms and {K.FLOW_MAX_HIDDEN} hidden layers of width <= "
                               f"{K.MNFSIM_MAX_H}, got {T} transforms of {hidden}")
        if var_mode != K.VAR_REFERENCE:
            raise K.LbbnnError("the kernel implements the reference weight variance (var_mode='reference') only")
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
        self.lrs = self._rates(lrs)
        per_net = [[getattr(l, k) for k in SIM_LAYER_NAMES] + l.z_flow._params() + l.r_flow._params() for l in layers]
        if any(not p.is_cuda for ps in per_net for p in ps) or not X.is_cuda or not y.is_cuda:
            raise K.LbbnnError("SimStudyEnsemble takes CUDA networks and data (no CPU fallback)")
        dev = per_net[0][0].device
        if any(p.device != dev for ps in per_net for p in ps) or X.device != dev or y.device != dev:
            raise K.LbbnnError("networks and data must live on one device")
        K.require_device()
        self.nets, self.layers, self.R, self.in_features, self.rows, self.batch = nets, layers, R, in_f, n, B
        self.num_batches, self.n_transforms, self.hidden = num_batches, T, hidden
        self.priors = sig[4]
        self.seed = int(seed)
        self.X = X.detach().to(torch.float32).contiguous()
        self.y = y.detach().to(torch.float32).contiguous()
        count = sum(p.numel() for p in per_net[0])
        hid = (C.c_int * len(hidden))(*hidden)
        assert count == K.lib.lbbnn_mnfsim_param_count(in_f, T, len(hidden), hid)
        self.P = (count + 3) // 4 * 4
        f32 = dict(dtype=torch.float32, device=dev)
        self.flat = torch.zeros(R, self.P, **f32)
        self.exp_avg = torch.zeros(R, self.P, **f32)
        self.exp_avg_sq = torch.zeros(R, self.P, **f32)
        self.grads = torch.zeros(R, self.P, **f32) if materialize_grads else None
        self.step = torch.zeros(R, dtype=torch.int64, device=dev)
        self._lam = sum(getattr(layers[0], k).numel() for k in SIM_LAYER_NAMES[:2])
        with torch.no_grad():
            for r, ps in enumerate(per_net):
                o = 0
                for p in ps:
                    k = p.numel()
                    view = self.flat[r, o:o + k].view(p.shape)
                    view.copy_(p.data)
                    p.data = view
                    if self.grads is not None:
                        p.grad = self.grads[r, o:o + k].view(p.shape)
                    o += k

    @staticmethod
    def _rates(lrs):
        if isinstance(lrs, dict):
            if set(lrs) != set(SIM_GROUPS):
                raise K.LbbnnError(f"lrs must name exactly the groups {SIM_GROUPS}; unknown {sorted(set(lrs) - set(SIM_GROUPS))}, "
                                   f"missing {sorted(set(SIM_GROUPS) - set(lrs))}")
            return [float(lrs[g]) for g in SIM_GROUPS]
        if isinstance(lrs, (int, float)) and not isinstance(lrs, bool):
            return [float(lrs)] * len(SIM_GROUPS)
        raise K.LbbnnError(f"lrs must be a float or a dict over {SIM_GROUPS}, got {type(lrs).__name__}")

    def steps_per_epoch(self):
        return self.rows // self.batch

    def run(self, epochs, lrs=None, noise=None):
        """Train every replica for `epochs` epochs in one launch on the current stream; returns the (R, steps, 3) device tensor
        of [loss, nll, kl] per step.  lrs: new learning rates from this run on (kept for later runs).  noise: injected
        draws instead of Philox (tests), a dict of eps_z, eps_z2 (R, steps, in), z_masks, z_masks2, r_masks
        (R, steps, T, in), eps (R, steps, batch), eps_r (R, steps)."""
        if isinstance(epochs, bool) or int(epochs) != epochs or epochs < 1:
            raise K.LbbnnError(f"epochs must be an integer >= 1, got {epochs}")
        epochs = int(epochs)
        rates = self.lrs if lrs is None else self._rates(lrs)
        R, D, T, steps = self.R, self.in_features, self.n_transforms, epochs * self.steps_per_epoch()
        keep = {}
        if noise is not None:
            if set(noise) != set(_SIM_NOISE):
                raise K.LbbnnError(f"injected noise takes exactly {_SIM_NOISE}, got {sorted(noise)}")
            want = {"eps_z": (R, steps, D), "eps_z2": (R, steps, D), "z_masks": (R, steps, T, D), "z_masks2": (R, steps, T, D),
                    "r_masks": (R, steps, T, D), "eps": (R, steps, self.batch), "eps_r": (R, steps)}
            for name, t in noise.items():
                if not torch.is_tensor(t) or tuple(t.shape) != want[name]:
                    raise K.LbbnnError(f"injected {name} must be a tensor of shape {want[name]}, got "
                                       f"{tuple(t.shape) if torch.is_tensor(t) else type(t).__name__}")
            for name, t in noise.items():
                if not t.is_cuda or t.device != self.flat.device:
                    raise K.LbbnnError(f"injected {name} must live on {self.flat.device}")
                keep[name] = t.detach().to(torch.float32).contiguous()
        self.lrs = rates
        stats = torch.empty(R, steps, 3, dtype=torch.float32, device=self.flat.device)
        d = K.MnfSim()
        d.replicas, d.in_features, d.rows, d.batch = R, D, self.rows, self.batch
        d.n_transforms, d.n_hidden = T, len(self.hidden)
        for i, h in enumerate(self.hidden):
            d.hidden[i] = h
        d.params, d.exp_avg, d.exp_avg_sq, d.param_stride = K.ptr(self.flat), K.ptr(self.exp_avg), K.ptr(self.exp_avg_sq), self.P
        d.x, d.x_stride = K.ptr(self.X), (self.rows * D if self.X.dim() == 3 else 0)
        d.y, d.y_stride = K.ptr(self.y), (self.rows if self.y.dim() == 2 else 0)
        d.lr = (C.c_float * 12)(*rates)
        d.beta1, d.beta2, d.adam_eps = self.BETAS[0], self.BETAS[1], self.EPS
        d.num_batches = self.num_batches
        d.priors = K.Priors(*self.priors)
        d.seed = self.seed & (2 ** 64 - 1)
        d.step = K.ptr(self.step, torch.int64)
        d.stats, d.grads = K.ptr(stats), K.ptr(self.grads, allow_none=True)
        for name, t in keep.items():
            setattr(d, name, K.ptr(t))
        K.check(K.lib.lbbnn_mnfsim_train_f32(C.byref(d), epochs, K.current_stream()))
        return stats

    def inclusion_probabilities(self):
        """alpha = 1 / (1 + exp(-lambdal)) of every replica, (R, in)."""
        o = self._lam
        return 1.0 / (1.0 + torch.exp(-self.flat[:, o:o + self.in_features]))
