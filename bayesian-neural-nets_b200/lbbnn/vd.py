"""Drop-in variational-dropout layer, network and training step (reference: variational_dropout.py:55-110;
SURVEY.md §8f rank 4).

`BayesianLayer(n, m)` keeps the reference's constructor, its `theta` (n, m) parameter (= the only state_dict key:
the reference's `alpha = nn.Parameter(zeros) + 0.2` is a NON-leaf tensor, so it is neither registered nor trained,
VD:61) and `forward(x)`.  What the reference reads from its module-level `config` / `device` are keyword arguments.
`alpha_trainable=True` turns alpha into the trainable per-neuron dropout rate the docstring of the script describes.
The compute is lbbnn_vd_{fwd,bwd,kl} of liblbbnn (csrc/vd.cu) -- CUDA tensors only, no fallback.
"""
import itertools

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi as K
from . import lrt as _lrt
from .engine import LRTTrainer, MultiTensorAdam, check_replicas
from .predict import ShardedPredictor

_layer_ids = itertools.count(1)


def workspace_bytes(batch, n, m):
    return int(K.lib.lbbnn_vd_workspace_bytes(batch, n, m))


class _VDFunction(torch.autograd.Function):
    """act = x theta + sqrt((x^2 theta^2) alpha) zeta (VD:63-68); backward: the formulas at the top of csrc/vd.cu."""

    @staticmethod
    def forward(ctx, x, theta, alpha, zeta, noise_key):
        K.require_device()
        x = x.contiguous()
        theta_c, alpha_c = theta.contiguous(), alpha.contiguous()
        B, n = x.shape
        if theta_c.shape[0] != n:
            raise K.LbbnnError(f"input has {n} features, layer expects {theta_c.shape[0]}")
        m = theta_c.shape[1]
        if zeta is not None:
            zeta = zeta.contiguous()
            if tuple(zeta.shape) != (B, m):
                raise K.LbbnnError(f"zeta must be {(B, m)}, got {tuple(zeta.shape)}")
        noise = K.make_noise(zeta, noise_key[0], noise_key[1])
        need_bwd = any(ctx.needs_input_grad[:3])
        act = torch.empty(B, m, dtype=torch.float32, device=x.device)
        dsf = torch.empty_like(act) if need_bwd else None
        q = torch.empty_like(act) if need_bwd else None
        ws = K.workspace(workspace_bytes(B, n, m), x.device)
        K.check(K.lib.lbbnn_vd_fwd(K.ptr(theta_c), K.ptr(alpha_c), K.ptr(x), B, n, m, noise, 0, K.ptr(act),
                                   K.ptr(dsf, True), K.ptr(q, True), ws.data_ptr(), ws.numel(), K.current_stream()))
        ctx.save_for_backward(x, theta_c, alpha_c, dsf, q)
        return act

    @staticmethod
    def backward(ctx, g):
        x, theta, alpha, dsf, q = ctx.saved_tensors
        B, n = x.shape
        m = theta.shape[1]
        g = g.contiguous()
        d_theta = torch.empty_like(theta) if ctx.needs_input_grad[1] else None
        d_alpha = torch.empty_like(alpha) if ctx.needs_input_grad[2] else None
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        ws = K.workspace(workspace_bytes(B, n, m), x.device)
        K.check(K.lib.lbbnn_vd_bwd(K.ptr(theta), K.ptr(alpha), K.ptr(x), None, K.ptr(dsf), K.ptr(q), K.ptr(g), B, n, m, 0,
                                   K.ptr(d_theta, True), K.ptr(d_alpha, True), K.ptr(dx, True), ws.data_ptr(), ws.numel(),
                                   K.current_stream()))
        return dx, d_theta, d_alpha, None, None


class _VDKL(torch.autograd.Function):
    """sum 0.5 log a + c1 a + c2 a^2 + c3 a^3 (VD:98-102)."""

    @staticmethod
    def forward(ctx, alpha):
        K.require_device()
        alpha = alpha.contiguous()
        kl = torch.empty((), dtype=torch.float32, device=alpha.device)
        K.check(K.lib.lbbnn_vd_kl(K.ptr(alpha), alpha.numel(), K.ptr(kl), 0, None, 0.0, K.current_stream()))
        ctx.save_for_backward(alpha)
        return kl

    @staticmethod
    def backward(ctx, g):
        (alpha,) = ctx.saved_tensors
        d = torch.zeros_like(alpha)
        K.check(K.lib.lbbnn_vd_kl(K.ptr(alpha), alpha.numel(), None, 0, K.ptr(d), 1.0, K.current_stream()))
        return d * g


def vd_linear(x, theta, alpha, *, zeta=None, noise_key=(0, 0)):
    """Functional form of BayesianLayer.forward."""
    return _VDFunction.apply(x, theta, alpha, zeta, noise_key)


def vd_kl(alpha):
    return _VDKL.apply(alpha)


class BayesianLayer(nn.Module):
    """Drop-in for variational_dropout.py:55-68.  `zeta=` on forward injects the N(0,1) draw of VD:66 (parity tests);
    otherwise it is drawn natively (Philox) inside the kernel, reproducible through `last_noise_key`."""

    def __init__(self, n, m, *, device=None, low=-0.1, high=0.1, alpha_init=0.2, alpha_trainable=False):
        super().__init__()
        self.n, self.m = n, m
        self.theta = nn.Parameter((low - high) * torch.rand(size=(n, m)) + high)        # VD:59-60, same RNG use
        if alpha_trainable:
            self.alpha = nn.Parameter(torch.full((m,), float(alpha_init)))
        else:
            # the reference's alpha is a plain tensor attribute (see module docstring); a buffer so that .to() moves it
            self.register_buffer("alpha", torch.full((m,), float(alpha_init)), persistent=False)
        self._uid = next(_layer_ids)
        self._calls = 0
        self.last_noise_key = None
        if device is not None:
            self.to(device)

    def _next_noise_key(self):
        self._calls += 1
        self.last_noise_key = (_lrt.current_seed(), (0x5D << 56) | (self._uid << 40) | self._calls)
        return self.last_noise_key

    def forward(self, x, zeta=None):
        key = self._next_noise_key() if zeta is None else (0, 0)
        return _VDFunction.apply(x, self.theta, self.alpha, zeta, key)

    def kl(self):
        return _VDKL.apply(self.alpha)


class BNN(nn.Module):
    """784-1200-1200-1200-10 variational-dropout MLP, drop-in for variational_dropout.py:71-85 (sizes configurable)."""

    def __init__(self, sizes=(28 * 28, 1200, 1200, 1200, 10), **layer_kwargs):
        super().__init__()
        self.sizes = tuple(sizes)
        for i, (n, m) in enumerate(zip(sizes[:-1], sizes[1:]), 1):
            setattr(self, f"l{i}", BayesianLayer(n, m, **layer_kwargs))
        self._names = [f"l{i}" for i in range(1, len(sizes))]

    @property
    def layers(self):
        return [getattr(self, n) for n in self._names]

    def forward(self, x, zetas=None):
        x = x.view(-1, self.sizes[0])
        ls = self.layers
        for i, l in enumerate(ls):
            x = l(x, None if zetas is None else zetas[i])
            x = F.relu(x) if i < len(ls) - 1 else F.log_softmax(x, dim=1)
        return x


def loss_fn(prediction, target, model, num_batches=600.0):
    """loss_fn of variational_dropout.py:88-106: KL / num_batches + nll_loss(sum); num_batches = N / batch_size, which the
    reference derives from its module-level loaders (and, `model.train()` being truthy, always from the TRAIN set)."""
    kl = 0
    for layer in model.children():
        if isinstance(layer, BayesianLayer):
            kl = kl + layer.kl()
    return kl / num_batches + F.nll_loss(prediction, target, reduction="sum")


def predict_ensemble(model, images, samples=10):
    """The evaluation branch of run_epoch (VD:148-157): mean over `samples` stochastic forwards of the log-probabilities.
    EnsemblePredictor computes the same statistic with the samples batched on the device (and sharded over GPUs)."""
    with torch.no_grad():
        acc = None
        for _ in range(samples):
            out = model(images)
            acc = out if acc is None else acc + out
        return acc / samples


class EnsemblePredictor(ShardedPredictor):
    """predict_ensemble (the evaluation branch of run_epoch, VD:148-157) with the Monte-Carlo samples batched on the device:
    the samples of a launch are stacked along the batch dimension and every layer runs ONCE per launch.

      * layer 1 sees the same input in every sample: E1 = x theta and S1 = x^2 theta^2 are computed once per run()
        (lbbnn_vd_fwd_ex with FLAG_MOMENTS, or two 3xTF32 GEMMs on the tensor cores) and every sample only adds its
        sqrt(S1 alpha) zeta (lbbnn_vd_mc_epilogue with shared E and S);
      * layers 2.. are ONE problem of samples_per_launch * batch rows: lbbnn_vd_fwd_ex with per-sample noise streams on the
        CUDA cores, or E = A theta and S = A^2 theta^2 as two lbbnn_tc_linear_tf32x3 calls and lbbnn_vd_mc_epilogue on the
        tensor cores (theta^T and (theta^2)^T split into hi / lo once per run() by lbbnn_vd_tc_prepare);
      * log-softmax and the running sum stay on the device in fp64 (lbbnn_mc_accumulate_batched).

    Sample g (global index) of layer l draws zeta from Philox stream (0x5E << 56) | (l + g * n_layers) of the predictor's
    seed, so results do not depend on samples_per_launch, on sharding or on the GEMM path.  theta and alpha are read on
    every run(); alpha may be the reference's buffer or a parameter (alpha_trainable=True).

    gemm: "simt" = every layer on the CUDA cores; "tc" = every layer with in_features % 4 == 0 on the tensor cores at fp32
    accuracy except a <= 16-class head; "auto" = the tensor cores for layers with in and out features both >= 1024 (the
    784-1200-1200-1200-10 network: tc == [False, True, True, False]).
    process_group: predict_ensemble shards its samples over the ranks and every rank gets the same result."""

    STREAM_TAG = 0x5E << 56

    def __init__(self, model, batch, samples_per_launch=10, seed=None, gemm="auto", process_group=None):
        K.require_device()
        if gemm not in ("auto", "simt", "tc"):
            raise ValueError(f"gemm must be 'auto', 'simt' or 'tc', got {gemm!r}")
        self.net, self.layers, self.B = model, list(model.layers), int(batch)
        self.SB = max(1, int(samples_per_launch))
        self.seed = _lrt.current_seed() if seed is None else int(seed)
        dev = self.layers[0].theta.device
        if dev.type != "cuda":
            raise K.LbbnnError("vd.EnsemblePredictor needs the network on a CUDA device (no CPU fallback)")
        self.device = dev
        self._join_group(process_group, [getattr(l, n) for l in self.layers for n in ("theta", "alpha")],
                         "vd.EnsemblePredictor")
        self.sizes = sizes = [(l.n, l.m) for l in self.layers]
        L, B, SB, C = len(sizes), self.B, self.SB, sizes[-1][1]
        self.tc = [k % 4 == 0 and not (i == L - 1 and o <= 16) and (gemm == "tc" or (gemm == "auto" and k >= 1024 and o >= 1024))
                   for i, (k, o) in enumerate(sizes)]
        # layer 1 and the tensor-core layers end in lbbnn_vd_mc_epilogue, which writes the next tensor-core layer's operands
        # directly; an fp32 output is kept where a CUDA-core layer or the head reads it, or a CUDA-core layer must split it
        self._feeds_tc = [i + 1 < L and self.tc[i + 1] for i in range(L)]
        f32 = dict(dtype=torch.float32, device=dev)
        self.x = torch.zeros(B, sizes[0][0], **f32)
        self.E1, self.S1 = torch.zeros(B, sizes[0][1], **f32), torch.zeros(B, sizes[0][1], **f32)
        self.h = [torch.zeros(SB * B, o, **f32) if not self._feeds_tc[i] or (i > 0 and not self.tc[i]) else None
                  for i, (_, o) in enumerate(sizes)]
        self.ws = torch.empty(max([workspace_bytes(B, *sizes[0])] + [workspace_bytes(SB * B, k, o) for k, o in sizes[1:]]),
                              dtype=torch.uint8, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        self.sum_logp, self.sum_prob = torch.zeros(B, C, **f64), torch.zeros(B, C, **f64)
        self.kernels_per_launch = 0
        self.samples, self.global_samples = 0, None
        self.w, self.wsq, self.a, self.asq = {}, {}, {}, {}
        if any(self.tc):
            pair = lambda *shape: (torch.zeros(*shape, **f32), torch.zeros(*shape, **f32))      # noqa: E731
            for i, (k, o) in enumerate(sizes):
                if self.tc[i]:          # theta^T, (theta^2)^T (once per run()) and the inputs A, A^2 (the test batch for
                    rows = B if i == 0 else SB * B      # layer 1, the stacked rows after it), all as hi / lo
                    self.w[i], self.wsq[i] = pair(o, k), pair(o, k)
                    self.a[i], self.asq[i] = pair(rows, k), pair(rows, k)
            mo = max(o for (_, o), t in zip(sizes, self.tc) if t)
            self.E, self.S = torch.zeros(SB * B * mo, **f32), torch.zeros(SB * B * mo, **f32)
            self.zero_bias = torch.zeros(mo, **f32)

    def _stream(self, layer, sample):
        return self.STREAM_TAG | (layer + sample * len(self.layers))

    def _noise_for(self, li, s0, off, n, zetas):
        """(lbbnn_noise, group stride, keepalive) for the n samples with global indices s0 .. of layer li (injected zeta is
        indexed by `off`: the position inside this run() call, or the global index under global_samples)."""
        if zetas is not None:
            z = zetas[li][off:off + n].reshape(n * self.B, self.sizes[li][1]).contiguous()
            return K.make_noise(z), 0, z
        return K.make_noise(None, self.seed, self._stream(li, s0)), len(self.layers), None

    def _prepare(self, st):
        """Per run(): theta^T, (theta^2)^T of the tensor-core layers as hi / lo, and layer 1's E1 = x theta, S1 = x^2 theta^2
        for the test batch."""
        for i in self.w:
            k, o = self.sizes[i]
            K.check(K.lib.lbbnn_vd_tc_prepare(K.ptr(self.layers[i].theta.data), k, o, K.ptr(self.w[i][0]), K.ptr(self.w[i][1]),
                                              K.ptr(self.wsq[i][0]), K.ptr(self.wsq[i][1]), st))
        l = self.layers[0]
        k, o = self.sizes[0]
        if self.tc[0]:
            K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(self.x), 0, self.B, k, 1, None, K.ptr(self.a[0][0]), K.ptr(self.a[0][1]),
                                                K.ptr(self.asq[0][0]), K.ptr(self.asq[0][1]), st))
            self._gemm(self.a[0], self.w[0], self.B, k, o, self.E1.view(-1), st)
            self._gemm(self.asq[0], self.wsq[0], self.B, k, o, self.S1.view(-1), st)
        else:
            K.check(K.lib.lbbnn_vd_fwd_ex(K.ptr(l.theta.data), K.ptr(l.alpha.data), K.ptr(self.x), self.B, k, o, None,
                                          K.FLAG_MOMENTS, K.ptr(self.E1), None, K.ptr(self.S1), self.B, 0, self.ws.data_ptr(),
                                          self.ws.numel(), st))

    def _layer(self, li, s0, off, n, zetas, h, st):
        """Layer li for the n samples s0 .. of a launch (h: the stacked activations of layer li - 1); returns (its stacked
        fp32 activations or None, the number of kernels it launched)."""
        L, B = len(self.layers), self.B
        l = self.layers[li]
        k, o = self.sizes[li]
        flags = 0 if li == L - 1 else K.FLAG_RELU
        nz, gstride, keep = self._noise_for(li, s0, off, n, zetas)
        out = None if self.h[li] is None else self.h[li][:n * B]
        nxt = (self.a[li + 1], self.asq[li + 1]) if self._feeds_tc[li] else ((None, None), (None, None))
        if li == 0 or self.tc[li]:
            if li == 0:
                E, es, S, ss, nk = self.E1, 0, self.S1, 0, 0
            else:
                self._gemm(self.a[li], self.w[li], n * B, k, o, self.E, st)
                self._gemm(self.asq[li], self.wsq[li], n * B, k, o, self.S, st)
                E, es, S, ss, nk = self.E, B * o, self.S, B * o, 2
            K.check(K.lib.lbbnn_vd_mc_epilogue(K.ptr(E), es, K.ptr(S), ss, K.ptr(l.alpha.data), B, o, n, nz, gstride, flags,
                                               K.ptr(None if self._feeds_tc[li] else out, True), K.ptr(nxt[0][0], True),
                                               K.ptr(nxt[0][1], True), K.ptr(nxt[1][0], True), K.ptr(nxt[1][1], True), st))
            return (None if self._feeds_tc[li] else out), nk + 1
        K.check(K.lib.lbbnn_vd_fwd_ex(K.ptr(l.theta.data), K.ptr(l.alpha.data), K.ptr(h), n * B, k, o, nz, flags, K.ptr(out),
                                      None, None, B, gstride, self.ws.data_ptr(), self.ws.numel(), st))
        nk = K.lib.lbbnn_vd_gemm_launches(n * B, o, k)
        if self._feeds_tc[li]:        # a CUDA-core layer feeding a tensor-core one
            K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(out), 0, n * B, o, 1, None, K.ptr(nxt[0][0]), K.ptr(nxt[0][1]),
                                                K.ptr(nxt[1][0]), K.ptr(nxt[1][1]), st))
            nk += 1
        return out, nk

    def _launch(self, s0, off, n, zetas):
        st = K.current_stream()
        nk, h = 0, None
        for li in range(len(self.layers)):
            h, k = self._layer(li, s0, off, n, zetas, h, st)
            nk += k
        K.check(K.lib.lbbnn_mc_accumulate_batched(K.ptr(h), n, self.B, self.sizes[-1][1], self.sum_logp.data_ptr(),
                                                  self.sum_prob.data_ptr(), None, st))
        self.kernels_per_launch = nk + 1

    def _check_inputs(self, x, zetas, end):
        B, n0 = self.B, self.sizes[0][0]
        if not torch.is_tensor(x) or not x.is_cuda:
            raise K.LbbnnError("vd.EnsemblePredictor takes CUDA inputs only (no CPU fallback)")
        if x.numel() != B * n0 or x.shape[0] != B:
            raise K.LbbnnError(f"input must be ({B}, {n0}) (or reshape to it), got {tuple(x.shape)}")
        if zetas is not None:
            if len(zetas) != len(self.layers):
                raise K.LbbnnError(f"zetas: one tensor per layer ({len(self.layers)}), got {len(zetas)}")
            for z, (_, o) in zip(zetas, self.sizes):
                if z.dim() != 3 or tuple(z.shape[1:]) != (B, o) or z.shape[0] < end:
                    raise K.LbbnnError(f"zetas: expected (>= {end}, {B}, {o}) per layer, got {tuple(z.shape)}")

    @torch.no_grad()
    def run(self, x, samples, first_sample=0, zetas=None, global_samples=None):
        """Accumulate `samples` stochastic forwards (global sample indices first_sample ..) of the input batch x into the
        fp64 sum_logp.  zetas: optional injected N(0,1) noise, one (S, batch, out) tensor per layer.  global_samples: this
        call runs part of a run over samples 0 .. global_samples (one rank's shard), and zetas are indexed by global sample;
        without it they are indexed from first_sample."""
        st = K.current_stream()
        first, count = int(first_sample), int(samples)
        base = first if global_samples is None else 0
        if global_samples is not None and first + count > int(global_samples):
            raise ValueError(f"samples {first} .. {first + count} lie outside the global run of {global_samples}")
        self._check_inputs(x, zetas, first + count - base)
        self.x.copy_(x.reshape(self.x.shape))
        self.sum_logp.zero_()
        self.sum_prob.zero_()
        self._prepare(st)
        s, end = first, first + count
        while s < end:
            n = min(self.SB, end - s)
            self._launch(s, s - base, n, zetas)
            s += n
        self.samples = count
        self.global_samples = None if global_samples is None else int(global_samples)

    def result(self, total_samples=None):
        """mean_logp (fp64, (batch, classes)) and its argmax over the samples of the last run(); under a process group the
        sums are first added over the ranks and the default sample count is the global one."""
        S = self._total_samples(total_samples)
        (sum_logp,) = self._reduce((self.sum_logp,))
        mean = sum_logp / S
        return {"mean_logp": mean, "pred": mean.argmax(1)}

    @torch.no_grad()
    def predict_ensemble(self, images, samples, zetas=None):
        """What predict_ensemble(model, images, samples) returns: the fp32 mean over `samples` stochastic forwards of the
        log-probabilities.  Under a process group each rank runs its share of the samples and every rank returns the same
        value; injected zetas are indexed by global sample."""
        first, count = self._shard(samples)
        self.run(images, count, first_sample=first, zetas=zetas, global_samples=None if self.pg is None else samples)
        return self.result(samples)["mean_logp"].float()


class VDTrainer:
    """One training step of variational_dropout.py:160-166 (forward, loss_fn, backward, AdamW) on preallocated buffers,
    captured once in a CUDA graph: per layer lbbnn_vd_fwd with the relu fused in, the log-softmax / nll head,
    lbbnn_vd_bwd per layer (relu mask folded into the gradient staging), ONE AdamW launch over the flat theta buffer.
    alpha is constant unless the model was built with alpha_trainable=True (then its KL gradient is added and it is
    updated by the same AdamW rule).  stats = [nll, kl].

    Data parallel (process_group): each rank runs the captured step on its own `batch_size` rows of the minibatch and the
    update applies the SUM over ranks of the gradients (the nll is a sum over rows, VD:104-106), so the step is the
    single-GPU step on the concatenated minibatch.  Each rank draws its zeta from seed + 0x9E3779B97F4A7C15 * rank (the
    rows' noise is disjoint); the KL term is replicated, so its alpha gradient enters each rank at 1 / (num_batches * world).
    The ranks must be built alike (same seeds and shapes: checked), rank 0's parameters are broadcast, and every rank must
    replay the same number of steps: the update is MultiTensorAdam(weight_decay=).data_parallel -- the sharded multicast
    exchange, or the NCCL all-reduce under LBBNN_DP_UPDATE=nccl or without multicast (`dp_update` says which)."""

    def __init__(self, model, batch_size, num_batches=600.0, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2,
                 seed=None, use_graph=True, inject_noise=False, process_group=None):
        """process_group: data-parallel training over the ranks of this torch.distributed group (see the class docstring);
        batch_size is the rows of ONE rank."""
        K.require_device()
        self.net = model
        self.layers = list(model.layers)
        self.B = int(batch_size)
        self.num_batches = float(num_batches)
        self.lr, self.betas, self.eps, self.wd = float(lr), betas, float(eps), float(weight_decay)
        self.seed = _lrt.current_seed() if seed is None else int(seed)
        self.pg = process_group
        self.world = 1 if process_group is None else torch.distributed.get_world_size(process_group)
        self.rank = 0 if process_group is None else torch.distributed.get_rank(process_group)
        dev = self.layers[0].theta.device
        self.device = dev
        f32 = dict(dtype=torch.float32, device=dev)
        self.train_alpha = isinstance(self.layers[0].alpha, nn.Parameter)
        names = ("theta", "alpha") if self.train_alpha else ("theta",)
        if process_group is not None:
            check_replicas(process_group, [getattr(l, n) for l in self.layers for n in names], "data-parallel VDTrainer")
        offs, total = [], 0
        for l in self.layers:
            for name in names:
                p = getattr(l, name)
                offs.append((l, name, total, p.numel(), p.shape))
                total += (p.numel() + 3) // 4 * 4
        self.n_flat = total
        self.gflat = torch.zeros(total, **f32)
        self.opt, self.dp_update = None, None
        if process_group is None:
            self.flat = torch.zeros(total, **f32)
            self.exp_avg, self.exp_avg_sq = torch.zeros(total, **f32), torch.zeros(total, **f32)
        with torch.no_grad():
            for l, name, off, n, shape in offs:
                p = getattr(l, name)
                if process_group is None:
                    view = self.flat[off:off + n].view(shape)
                    view.copy_(p.data)
                    p.data = view
                p.grad = self.gflat[off:off + n].view(shape)
        if process_group is not None:
            # parameters move into the exchange's arena; the gradients stay in gflat, where lbbnn_vd_bwd writes them
            self.opt = MultiTensorAdam([getattr(l, n) for l in self.layers for n in names], lr=self.lr, betas=betas,
                                       eps=self.eps, weight_decay=self.wd)
            self.opt.data_parallel(process_group)
            self.dp_update = self.opt.dp["mode"]
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.adam_coef = torch.zeros(2, **f32)
        B = self.B
        self.sizes = [(l.n, l.m) for l in self.layers]
        self.x = torch.zeros(B, self.sizes[0][0], **f32)
        self.y = torch.zeros(B, dtype=torch.int64, device=dev)
        self.buf = [dict(act=torch.zeros(B, m, **f32), dsf=torch.zeros(B, m, **f32), q=torch.zeros(B, m, **f32),
                         g=torch.zeros(B, m, **f32), zeta=torch.zeros(B, m, **f32) if inject_noise else None,
                         d_alpha=torch.zeros(m, **f32))
                    for _, m in self.sizes]
        self.inject = inject_noise
        self.stats = torch.zeros(2, **f32)
        self.ws = torch.empty(max([1 << 20] + [workspace_bytes(B, n, m) for n, m in self.sizes]), dtype=torch.uint8,
                              device=dev)
        self.x_host = torch.zeros(B, self.sizes[0][0], dtype=torch.float32).pin_memory()
        self.y_host = torch.zeros(B, dtype=torch.int64).pin_memory()
        self.stats_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        self.kernels_per_step = 0
        self.graph = None
        if use_graph:
            self._capture()
            if self.opt is not None:
                self.opt.finish_capture()

    def _noise(self, i):
        if self.inject:
            return K.make_noise(self.buf[i]["zeta"])
        return K.make_noise(None, self.seed + 0x9E3779B97F4A7C15 * self.rank, (0x5D << 56) | i, self.step_dev,
                            len(self.layers))

    def _train_state(self):
        """What a step changes besides activations: restored after _capture's warm-up step, which must not count."""
        if self.opt is None:
            return self.flat, self.exp_avg, self.exp_avg_sq, self.step_dev
        o = self.opt
        return o.dp["arena"][:o.n_flat], o.exp_avg, o.exp_avg_sq, o.t_dev, self.step_dev

    def owned_range(self, layer_index, name):
        """Element range [lo, hi) of parameter `name` of layer `layer_index` whose AdamW moments THIS rank maintains: all of
        it, except under the sharded data-parallel update (MultiTensorAdam.owned_range)."""
        p = getattr(self.layers[layer_index], name)
        return (0, p.numel()) if self.opt is None else self.opt.owned_range(p)

    def _enqueue(self):
        st = K.current_stream()
        lib, P = K.lib, K.ptr
        L, B = len(self.layers), self.B
        ws, wsn = self.ws.data_ptr(), self.ws.numel()
        n = 0
        h = self.x
        for i, (l, b) in enumerate(zip(self.layers, self.buf)):
            fi, fo = self.sizes[i]
            K.check(lib.lbbnn_vd_fwd(P(l.theta.data), P(l.alpha.data), P(h), B, fi, fo, self._noise(i),
                                     0 if i == L - 1 else K.FLAG_RELU, P(b["act"]), P(b["dsf"]), P(b["q"]), ws, wsn, st))
            n += lib.lbbnn_vd_gemm_launches(B, fo, fi)
            K.check(lib.lbbnn_vd_kl(P(l.alpha.data), fo, self.stats[1:].data_ptr(), 1 if i else 0, None, 0.0, st))
            n += 1
            h = b["act"]
        last = self.buf[-1]
        K.check(lib.lbbnn_logsoftmax_nll_f32(P(last["act"]), P(self.y, torch.int64), B, self.sizes[-1][1], None,
                                             self.stats.data_ptr(), P(last["g"]), 1.0, P(self.step_dev, torch.int64),
                                             ws, wsn, st))
        n += 2 if B > 512 else 1
        for i in reversed(range(L)):
            l, b = self.layers[i], self.buf[i]
            fi, fo = self.sizes[i]
            xin = self.x if i == 0 else self.buf[i - 1]["act"]
            dx = None if i == 0 else self.buf[i - 1]["g"]
            d_alpha = l.alpha.grad if self.train_alpha else None
            K.check(lib.lbbnn_vd_bwd(P(l.theta.data), P(l.alpha.data), P(xin), P(b["act"]), P(b["dsf"]), P(b["q"]), P(b["g"]),
                                     B, fi, fo, 0 if i == L - 1 else K.FLAG_RELU, P(l.theta.grad), P(d_alpha, True),
                                     P(dx, True), ws, wsn, st))
            n += 1 + lib.lbbnn_vd_gemm_launches(fi, fo, B) + (lib.lbbnn_vd_gemm_launches(B, fi, fo) if dx is not None else 0)
            if self.train_alpha:      # the KL is replicated on every rank: its gradient is added once over the ranks
                K.check(lib.lbbnn_vd_kl(P(l.alpha.data), fo, None, 0, P(l.alpha.grad), 1.0 / (self.num_batches * self.world),
                                        st))
                n += 1
        if self.opt is not None:
            self.opt.step()       # pack, exchange, AdamW
            n += 5 if self.dp_update == "sharded" else 4
        else:
            K.check(lib.lbbnn_adamw_f32(P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq), self.n_flat,
                                        self.lr, self.betas[0], self.betas[1], self.eps, self.wd,
                                        P(self.step_dev, torch.int64), P(self.adam_coef), st))
            n += 2
        self.kernels_per_step = n

    _capture = LRTTrainer._capture
    step_device = LRTTrainer.step_device
    step = LRTTrainer.step
    step_async = LRTTrainer.step_async
    flush = LRTTrainer.flush
    h2d_bytes_per_step = LRTTrainer.h2d_bytes_per_step
    d2h_bytes_per_step = LRTTrainer.d2h_bytes_per_step

    def _stats_dict(self, st):
        """Data parallel: `nll` and `loss` are THIS RANK's contribution (its rows, the replicated kl at 1 / world); their
        sums over ranks are the single-GPU values of the concatenated minibatch.  `kl` is the replicated term."""
        nll, kl = float(st[0]), float(st[1])
        return {"nll": nll, "kl": kl, "loss": nll + kl / (self.num_batches * self.world)}
