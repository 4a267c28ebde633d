"""Posterior-predictive model averaging for the LRT and MNF networks, batched over Monte-Carlo samples.

Reference: the per-batch bodies of `test_ensemble` (LBBNN-GP-MF-LRT.py:239-265, LBBNN-GP-MF-MNF.py:287-318) and `outofsample`
(LBBNN-GP-MF-LRT.py:305-341): TEST_SAMPLES times `net(data, sample=True)`, a device -> host NumPy round trip per sample for
the row-normalised expit average, `outputs[0:10].mean(0)` for the ensemble prediction, `net(data, sample=False)` for the
posterior-mean prediction.

Here the samples of a launch are stacked along the batch dimension and go through the fused LRT forward kernels
(csrc/lrt_f32.cu, fp32: the 1e-5 / bit-exact-argmax parity mode) ONCE per layer:

  * the LRT weights' moments M = alpha mu, V = alpha^2 sigma^2 do not depend on the sample, so layers 2.. are ONE dual GEMM
    over (samples x batch) rows, with per-sample native noise streams (`lbbnn_lrt_f32_fwd_ex`);
  * layer 1 sees the same input for every sample: e_b = x M^T + b_mu and var_b = x^2 V^T + sigma_b^2 are computed once per
    test batch (LRT:247 "only eps changes") and every sample only adds its sqrt(var_b) eps (`lbbnn_lrt_sample_expand`);
  * MNF: every sample draws its own multiplicative z per layer (the flows run once per launch on one row per sample); z
    scales the input rows of the mean product only (MNF:197-198), which the kernel applies per row group;
  * log-softmax, the row-normalised expit and both running sums stay on the device in fp64 (`lbbnn_mc_accumulate_batched`).

Sample s of layer l draws from Philox stream  l * 2 + s * 2 n_layers  of the predictor's seed, whatever the launch width.

Wide layers (gemm="tc", or "auto" at >= 1024 in and out features) run on the tensor cores at fp32 accuracy instead: E = A_E M^T
and S = A_S V^T are each ONE 3xTF32 tcgen05 GEMM over the stacked rows (lbbnn_tc_linear_tf32x3, M and V split into hi / lo
once per run()), and lbbnn_lrt_mc_epilogue adds b_mu + sqrt(S + sigma_b^2) eps with the same expressions and the same eps
streams as the fp32 kernels, writing the hi / lo operands of the next tensor-core layer (act .* z for its mean product, act^2
for its variance product).  Layer 1 of an LRT network computes E1, S1 once per test batch; MNF layer 1 shares S1.  A
<= 16-class head stays on the fp32 forward.

With a process_group, test_ensemble / outofsample run this rank's contiguous share of the samples (lbbnn.mf.shard_samples) and
ONE all-reduce of the four fp64 accumulators gives every rank the same statistics.  MNF's z rows are drawn for the whole run on
every rank, in the single-process order, so a sample gets the same z wherever it runs.
"""
import torch
import torch.nn.functional as F

from . import _capi as K
from .engine import check_replicas
from .lrt import current_seed
from .mf import shard_samples


class ShardedPredictor:
    """What the batched posterior-predictive loops (EnsemblePredictor here, lbbnn.vd.EnsemblePredictor) share: the process
    group (replica and seed checks at construction, contiguous sample shards, ONE all-reduce of the fp64 accumulators), the
    sample count of result() and the 3xTF32 tensor-core GEMM of a layer.  Subclasses set device, seed, samples,
    global_samples and zero_bias."""

    def _join_group(self, process_group, params, what):
        self.pg = process_group
        if process_group is None:
            return
        import torch.distributed as dist
        check_replicas(process_group, params, what)
        seeds = [None] * dist.get_world_size(process_group)
        dist.all_gather_object(seeds, self.seed, group=process_group)
        if len(set(seeds)) != 1:
            raise K.LbbnnError(f"{what}: ranks differ in the predictor seed: {seeds}")

    def _reduce(self, sums):
        """The fp64 accumulators `sums` over every rank: ONE all-reduce under a process group, this rank's own otherwise."""
        if self.pg is None:
            return tuple(sums)
        both = torch.stack(tuple(sums))
        torch.distributed.all_reduce(both, group=self.pg)
        return tuple(both.unbind(0))

    def _shard(self, samples):
        """(first, count) of this rank's samples of a global run of `samples` (all of them without a process group)."""
        if self.pg is None:
            return 0, int(samples)
        import torch.distributed as dist
        return shard_samples(int(samples), dist.get_world_size(self.pg), dist.get_rank(self.pg))

    def _total_samples(self, total_samples=None):
        """The sample count result() divides by: `total_samples`, else the global count of the last run, else (under a
        process group) the sum of the ranks' run() calls, else this process's."""
        if total_samples is not None:
            return int(total_samples)
        if self.global_samples is not None:
            return self.global_samples
        if self.pg is not None:
            n = torch.tensor([self.samples], dtype=torch.int64, device=self.device)
            torch.distributed.all_reduce(n, group=self.pg)
            return int(n.item())
        return self.samples

    def _gemm(self, a, w, rows, k, o, out, st):
        """out (rows, o) = a w^T in 3xTF32, a and w as (hi, lo) pairs: ONE problem, the weights are shared by all samples."""
        K.check(K.lib.lbbnn_tc_linear_tf32x3(K.ptr(a[0][:rows]), K.ptr(a[1][:rows]), k, 0, K.ptr(w[0]), K.ptr(w[1]),
                                             K.ptr(self.zero_bias), 1, rows, o, k, 0, K.ptr(out[:rows * o]), None, None, o,
                                             0, st))


class EnsemblePredictor(ShardedPredictor):
    def __init__(self, net, batch, samples_per_launch=10, seed=None, gemm="auto", process_group=None):
        """gemm: "simt" = every layer on the fused fp32 CUDA-core kernels; "tc" = every layer with in_features % 4 == 0 on the
        tensor cores at fp32 accuracy (3xTF32, see the module docstring) except a <= 16-class head; "auto" = the tensor cores
        only for layers with in and out features both >= 1024.  That threshold is not the measured crossover, which lies
        between 64 and 400 features (profiles/bench_ensemble.py): it keeps MNIST-shape networks on their CUDA-core results.
        process_group: test_ensemble / outofsample shard their samples over its ranks."""
        K.require_device()
        if gemm not in ("auto", "simt", "tc"):
            raise ValueError(f"gemm must be 'auto', 'simt' or 'tc', got {gemm!r}")
        self.net, self.layers, self.B = net, list(net.layers), int(batch)
        self.SB = max(1, int(samples_per_launch))
        self.seed = current_seed() if seed is None else int(seed)
        self.mnf = hasattr(self.layers[0], "z_flow")
        dev = self.layers[0].weight_mu.device
        if dev.type != "cuda":
            raise K.LbbnnError("EnsemblePredictor needs the network on a CUDA device (no CPU fallback)")
        self.device = dev
        self._join_group(process_group, list(net.parameters()), "EnsemblePredictor")
        f32 = dict(dtype=torch.float32, device=dev)
        self.sizes = sizes = [(l.in_features, l.out_features) for l in self.layers]
        L, B, SB, C = len(sizes), self.B, self.SB, sizes[-1][1]
        self.tc = [k % 4 == 0 and not (i == L - 1 and o <= 16) and (gemm == "tc" or (gemm == "auto" and k >= 1024 and o >= 1024))
                   for i, (k, o) in enumerate(sizes)]
        self.x = torch.zeros(B, sizes[0][0], **f32)
        self.x_rep = torch.zeros(SB * B, sizes[0][0], **f32) if self.mnf and not self.tc[0] else None
        self.e1 = torch.zeros(B, sizes[0][1], **f32)
        self.var1 = torch.zeros(B, sizes[0][1], **f32)
        self.h = [torch.zeros(SB * B, o, **f32) for _, o in sizes]          # stacked activations; the last one = logits
        self.ws = torch.empty(max(K.lrt_workspace_bytes(SB * B, i, o) for i, o in sizes), dtype=torch.uint8, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        self.sum_logp, self.sum_prob = torch.zeros(B, C, **f64), torch.zeros(B, C, **f64)
        self.first_logp, self.first_prob = torch.zeros(B, C, **f64), torch.zeros(B, C, **f64)
        self.kernels_per_launch = 0
        self.samples, self.global_samples = 0, None
        self._z = None
        if any(self.tc):
            self._init_tc(f32)

    def _init_tc(self, f32):
        """Buffers of the tensor-core layers: M, V as hi / lo pairs (once per run()), each layer's two GEMM inputs as hi / lo
        pairs (written by the epilogue of the layer below), one E / S scratch pair shared by the layers, a zero bias."""
        B, SB = self.B, self.SB
        tcs = [(i, k, o) for i, ((k, o), on) in enumerate(zip(self.sizes, self.tc)) if on]
        pair = lambda *shape: (torch.zeros(*shape, **f32), torch.zeros(*shape, **f32))
        self.w_m, self.w_v, self.a_m, self.a_v, self.a_mean = {}, {}, {}, {}, {}
        for i, k, o in tcs:
            self.w_m[i], self.w_v[i] = pair(o, k), pair(o, k)
            shared = i == 0                      # layer 1 reads the test input: x^2 (and, for LRT, x) once per batch
            self.a_m[i] = pair(B if shared and not self.mnf else SB * B, k)
            self.a_v[i] = pair(B if shared else SB * B, k)
            self.a_mean[i] = pair(B, k)          # the posterior-mean forward (one row set)
        self.mv32 = torch.zeros(2, max(o * k for _, k, o in tcs), **f32)
        mo = max(o for _, _, o in tcs)
        self.E, self.S = torch.zeros(SB * B * mo, **f32), torch.zeros(SB * B * mo, **f32)
        self.zero_bias = torch.zeros(mo, **f32)
        if self.tc[0]:
            self.E1, self.S1 = torch.zeros(B, self.sizes[0][1], **f32), torch.zeros(B, self.sizes[0][1], **f32)

    # ---- noise -------------------------------------------------------------------------------------------------------
    def _stream(self, layer, sample):
        return layer * 2 + sample * 2 * len(self.layers)

    def _group_noise_ok(self, out_features):
        return (self.B * out_features) % 4 == 0

    def _noise_for(self, li, s0, off, n, eps):
        """(lbbnn_noise, group stride, keepalive) for the n samples with global indices s0 .. of layer li (injected noise is
        indexed by `off`: the position inside this run() call, or the global index under a process group)."""
        o = self.sizes[li][1]
        if eps is not None:
            e = eps[li][off:off + n].reshape(n * self.B, o).contiguous()
            return K.make_noise(e), 0, e
        stride = 2 * len(self.layers)
        if self._group_noise_ok(o):
            return K.make_noise(None, self.seed, self._stream(li, s0)), stride, None
        # odd shapes: materialise each sample's stream (what a batch-B call on that stream draws) and inject
        e = torch.cat([K.philox_normal((self.B, o), self.seed, self._stream(li, s0 + j), self.device) for j in range(n)])
        return K.make_noise(e), 0, e

    def _z_rows(self, li, off, n, z_noise):
        """MNF: the n samples' z of layer li = the flow image of one draw z0 per sample (MNF:182-187 with batch rows that are
        never used dropped).  z_noise[li] = {"eps_z": (S, in), "z_masks": [T x (S, in)]} injects the draws."""
        l = self.layers[li]
        if z_noise is not None:
            eps_z = z_noise[li]["eps_z"][off:off + n]
            masks = [m[off:off + n] for m in z_noise[li]["z_masks"]]
        else:
            eps_z, masks = torch.randn(n, l.in_features, device=self.device), None
        z0 = l.q0_mean + l.q0_log_var.exp().sqrt() * eps_z
        zs, _ = l.z_flow(z0, masks, per_row=True)
        return zs.contiguous()

    def _draw_z(self, start, count, z_noise):
        """MNF: the z rows of samples start .. start + count of every layer, drawn launch by launch (samples_per_launch
        samples at a time from `start`) and layer by layer within a launch: the order of torch.randn and flow-key draws
        of one launch loop over that range, whichever of its samples this process then runs."""
        zs = [[] for _ in self.layers]
        s = start
        while s < start + count:
            n = min(self.SB, start + count - s)
            for li in range(len(self.layers)):
                zs[li].append(self._z_rows(li, s - start, n, z_noise))
            s += n
        self._z = [torch.cat(z) if z else None for z in zs]
        self._z_start = start

    def _z_of(self, li, s0, n):
        return self._z[li][s0 - self._z_start:s0 - self._z_start + n]

    # ---- tensor-core layers ------------------------------------------------------------------------------------------------
    def _prepare_weights(self, st, sample=True):
        """M (and, for the sampled forward, V) of every tensor-core layer as hi / lo, from the current parameters."""
        flag = K.FLAG_SAMPLE if sample else 0
        for i in self.w_m:
            l = self.layers[i]
            k, o = self.sizes[i]
            desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
            m32, v32 = self.mv32[0, :o * k], self.mv32[1, :o * k]
            K.check(K.lib.lbbnn_lrt_f32_prologue(desc, l.cfg.priors, l.cfg.var_mode, flag, K.ptr(m32),
                                                 K.ptr(v32 if sample else None, True), None, None, 0, st))
            for src, (hi, lo) in ((m32, self.w_m[i]), (v32, self.w_v[i])) if sample else ((m32, self.w_m[i]),):
                K.check(K.lib.lbbnn_tf32_split(K.ptr(src), o * k, K.ptr(hi), K.ptr(lo), st))

    def _prepare_batch(self, st):
        """Per run(), before the first launch: layer 1's e_b / var_b (CUDA-core LRT layer 1); M, V of the tensor-core layers
        and, on a tensor-core layer 1, its input products for the test batch (E1 and S1 for LRT, S1 for MNF)."""
        if not self.mnf and not self.tc[0]:
            l = self.layers[0]
            desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
            K.check(K.lib.lbbnn_lrt_f32_fwd_ex(desc, K.ptr(self.x), self.B, K.make_noise(None, 0, 0), l.cfg.priors, l.cfg.var_mode,
                                               K.FLAG_SAMPLE | K.FLAG_MOMENTS, K.ptr(self.e1), K.ptr(self.var1), None, None, None, 0,
                                               0, self.ws.data_ptr(), self.ws.numel(), st))
        if not any(self.tc):
            return
        self._prepare_weights(st)
        if self.tc[0]:
            k, o = self.sizes[0]
            m = (None, None) if self.mnf else self.a_m[0]
            K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(self.x), 0, self.B, k, 1, None, K.ptr(m[0], True), K.ptr(m[1], True),
                                                K.ptr(self.a_v[0][0]), K.ptr(self.a_v[0][1]), st))
            if not self.mnf:
                self._gemm(self.a_m[0], self.w_m[0], self.B, k, o, self.E1.view(-1), st)
            self._gemm(self.a_v[0], self.w_v[0], self.B, k, o, self.S1.view(-1), st)

    def _tc_layer(self, li, n, nz, gstride, flags, out, s0, st):
        """One tensor-core layer for the n samples of a launch; returns the number of kernels it launched."""
        L, B = len(self.layers), self.B
        k, o = self.sizes[li]
        l = self.layers[li]
        rows, nk = n * B, 0
        if li == 0 and not self.mnf:            # E1, S1 of this test batch (run())
            E, es, S, ss = self.E1, 0, self.S1, 0
        else:
            if li == 0:                         # MNF: z scales the mean product's input only (MNF:197-198); S1 is shared
                K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(self.x), 0, B, k, n, K.ptr(self._z_of(0, s0, n)),
                                                    K.ptr(self.a_m[0][0]), K.ptr(self.a_m[0][1]), None, None, st))
                S, ss = self.S1, 0
                nk += 1
            else:
                self._gemm(self.a_v[li], self.w_v[li], rows, k, o, self.S, st)
                S, ss = self.S, B * o
                nk += 1
            self._gemm(self.a_m[li], self.w_m[li], rows, k, o, self.E, st)
            E, es = self.E, B * o
            nk += 1
        feeds_tc = li + 1 < L and self.tc[li + 1]
        z = self._z_of(li + 1, s0, n) if (feeds_tc and self.mnf) else None
        m, v = (self.a_m[li + 1], self.a_v[li + 1]) if feeds_tc else ((None, None), (None, None))
        K.check(K.lib.lbbnn_lrt_mc_epilogue(K.ptr(E), es, K.ptr(S), ss, K.ptr(l.bias_mu.data), K.ptr(l.bias_rho.data), B, o, n,
                                            nz, gstride, flags, None if feeds_tc else K.ptr(out), K.ptr(z, True),
                                            K.ptr(m[0], True), K.ptr(m[1], True), K.ptr(v[0], True), K.ptr(v[1], True), st))
        return nk + 1

    # ---- one launch: samples s0 .. s0 + n ----------------------------------------------------------------------------------
    def _layer(self, li, s0, off, n, eps, h, st):
        """Layer li for the n samples s0 .. of a launch (h: the stacked activations of layer li - 1); returns (its stacked
        activations, the number of kernels it launched)."""
        L, B = len(self.layers), self.B
        l = self.layers[li]
        fi, fo = self.sizes[li]
        last = li == L - 1
        flags = K.FLAG_SAMPLE | (0 if last else K.FLAG_RELU)
        nz, gstride, keep = self._noise_for(li, s0, off, n, eps)
        out = self.h[li][:n * B]
        if self.tc[li]:
            nk = self._tc_layer(li, n, nz, gstride, flags, out, s0, st)
        elif li == 0 and not self.mnf:
            # e_b, var_b were computed once for this test batch (run()); every sample adds its own sqrt(var_b) eps
            K.check(K.lib.lbbnn_lrt_sample_expand(K.ptr(self.e1), K.ptr(self.var1), B, fo, n, nz, gstride, flags, K.ptr(out), st))
            nk = 1
        else:
            desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
            xin = self.x_rep[:n * B] if li == 0 else h
            z = self._z_of(li, s0, n) if self.mnf else None
            K.check(K.lib.lbbnn_lrt_f32_fwd_ex(desc, K.ptr(xin), n * B, nz, l.cfg.priors, l.cfg.var_mode, flags, K.ptr(out), None,
                                               None, None, K.ptr(z, allow_none=True), B, gstride, self.ws.data_ptr(),
                                               self.ws.numel(), st))
            nk = 3
        if not self.tc[li] and not last and self.tc[li + 1]:      # a CUDA-core layer feeding a tensor-core one
            z = self._z_of(li + 1, s0, n) if self.mnf else None
            m, v = self.a_m[li + 1], self.a_v[li + 1]
            K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(out), B * fo, B, fo, n, K.ptr(z, True), K.ptr(m[0]), K.ptr(m[1]),
                                                K.ptr(v[0]), K.ptr(v[1]), st))
            nk += 1
        return out, nk

    def _launch(self, s0, off, n, eps, first_k):
        st = K.current_stream()
        B = self.B
        nk = 0
        h = None
        for li in range(len(self.layers)):
            h, k = self._layer(li, s0, off, n, eps, h, st)
            nk += k
        C = self.sizes[-1][1]
        K.check(K.lib.lbbnn_mc_accumulate_batched(K.ptr(h), n, B, C, self.sum_logp.data_ptr(), self.sum_prob.data_ptr(), None, st))
        nk += 1
        nf = min(n, first_k - s0)
        if nf > 0:     # the statistic over the FIRST first_k samples (outputs[0:10].mean(0), LRT:262)
            K.check(K.lib.lbbnn_mc_accumulate_batched(K.ptr(h), nf, B, C, self.first_logp.data_ptr(), self.first_prob.data_ptr(),
                                                      None, st))
            nk += 1
        self.kernels_per_launch = nk

    @torch.no_grad()
    def run(self, x, samples, first_sample=0, eps=None, z_noise=None, first_k=10, global_samples=None):
        """Accumulate `samples` stochastic forwards (global sample indices first_sample ..) over the input batch x.
        eps: optional injected N(0,1) noise, one (S, batch, out) tensor per layer; z_noise: MNF draws (see _z_rows).
        global_samples: this call runs part of a run over samples 0 .. global_samples (one rank's shard): MNF's z rows are
        drawn for that whole run and injected eps / z_noise are indexed by global sample.  Without it they are indexed from
        first_sample, and z is drawn for this call's samples only."""
        st = K.current_stream()
        first, count = int(first_sample), int(samples)
        base = first if global_samples is None else 0
        if global_samples is not None and first + count > int(global_samples):
            raise ValueError(f"samples {first} .. {first + count} lie outside the global run of {global_samples}")
        self.x.copy_(x.reshape(self.x.shape), non_blocking=True)
        for t in (self.sum_logp, self.sum_prob, self.first_logp, self.first_prob):
            t.zero_()
        if self.mnf:
            self._draw_z(base, count if global_samples is None else int(global_samples), z_noise)
            if self.x_rep is not None:
                self.x_rep.view(self.SB, *self.x.shape).copy_(self.x.unsqueeze(0).expand(self.SB, *self.x.shape))
        self._prepare_batch(st)
        s, end = first, first + count
        while s < end:
            n = min(self.SB, end - s)
            self._launch(s, s - base, n, eps, first_k)
            s += n
        self.samples = count
        self.global_samples = None if global_samples is None else int(global_samples)

    # ---- the LRT posterior-mean forward --------------------------------------------------------------------------------------
    @torch.no_grad()
    def mean_logits(self, x):
        """Logits of the LRT mean branch, x (alpha mu)^T + b_mu per layer with relu between (LRT:177-180, net(x, sample=False)
        before its log_softmax), on the same per-layer path as the sampled forward: the E product and the epilogue without
        noise on the tensor-core layers, the fused fp32 forward on the others.  Every layer reads the current parameters."""
        if self.mnf:
            raise K.LbbnnError("the MNF mean branch draws z (MNF:202-206): use net(x, sample=False)")
        st = K.current_stream()
        if any(self.tc):
            self._prepare_weights(st, sample=False)
        L, B = len(self.layers), self.B
        self.x.copy_(x.reshape(self.x.shape), non_blocking=True)
        h = self.x
        for li, l in enumerate(self.layers):
            k, o = self.sizes[li]
            flags = 0 if li == L - 1 else K.FLAG_RELU
            out = self.h[li][:B]
            if self.tc[li]:
                if li == 0 or not self.tc[li - 1]:
                    K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(h), 0, B, k, 1, None, K.ptr(self.a_mean[li][0]),
                                                        K.ptr(self.a_mean[li][1]), None, None, st))
                self._gemm(self.a_mean[li], self.w_m[li], B, k, o, self.E, st)
                feeds_tc = li + 1 < L and self.tc[li + 1]
                m = self.a_mean[li + 1] if feeds_tc else (None, None)
                K.check(K.lib.lbbnn_lrt_mc_epilogue(K.ptr(self.E), 0, None, 0, K.ptr(l.bias_mu.data), None, B, o, 1, None, 0,
                                                    flags, None if feeds_tc else K.ptr(out), None, K.ptr(m[0], True),
                                                    K.ptr(m[1], True), None, None, st))
            else:
                desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
                K.check(K.lib.lbbnn_lrt_f32_fwd_ex(desc, K.ptr(h), B, K.make_noise(None, 0, 0), l.cfg.priors, l.cfg.var_mode,
                                                   flags, K.ptr(out), None, None, None, None, 0, 0, self.ws.data_ptr(),
                                                   self.ws.numel(), st))
            h = out
        return h.clone()

    # ---- the reference's statistics ------------------------------------------------------------------------------------------
    def _sums(self):
        """(sum_logp, sum_prob, first_logp, first_prob) over every rank: ONE all-reduce of the four fp64 accumulators under a
        process group, this rank's own otherwise."""
        return self._reduce((self.sum_logp, self.sum_prob, self.first_logp, self.first_prob))

    def result(self, total_samples=None, first_k=10):
        """Statistics of the last run(); under a process group the accumulators are first summed over the ranks, and the
        default sample count is the global one (that of test_ensemble / outofsample, or the sum of the ranks' run() calls)."""
        S = self._total_samples(total_samples)
        k = min(S, first_k)
        sum_logp, sum_prob, first_logp, _ = self._sums()
        probs = sum_prob / S
        return {"mean_logp": sum_logp / S, "mean_prob": probs,                                          # `mydata_means`, LRT:249-258
                "ensemble": (first_logp / k).argmax(1),                                                  # LRT:262-263
                "entropy": -(probs * torch.log(probs)).sum(1)}                                           # LRT:325-330

    @torch.no_grad()
    def test_ensemble(self, x, samples, ensemble_first=10, eps=None, z_noise=None, mean_forward=None):
        """The per-batch statistics of `test_ensemble` (LRT:239-265 / MNF:287-318): mean_prob, ensemble (argmax of the mean
        of the first `ensemble_first` log-softmax outputs), posterior_mean (argmax of net(x, sample=False)), entropy.
        Under a process group `samples` is the global count; every rank gets the same statistics."""
        first, count = self._shard(samples)
        self.run(x, count, first_sample=first, eps=eps, z_noise=z_noise, first_k=ensemble_first,
                 global_samples=None if self.pg is None else samples)
        out = self.result(samples, ensemble_first)
        was_training = self.net.training
        self.net.eval()
        if mean_forward is not None:
            mean_out = mean_forward(x)
        elif any(self.tc) and not self.mnf:
            mean_out = self.mean_logits(x)
        else:
            mean_out = self.net(x, sample=False)                                                        # LRT:264
        if was_training:
            self.net.train()
        out["posterior_mean"] = mean_out.argmax(1)
        return out

    @torch.no_grad()
    def outofsample(self, x, samples, eps=None, z_noise=None):
        """`outofsample` for one batch (LRT:305-341): predictive entropy of the averaged row-normalised expit over all
        samples, and the prediction from `outputs[1:TEST_SAMPLES].mean(0)` -- the reference skips sample 0 there.
        Under a process group `samples` is the global count."""
        first, count = self._shard(samples)
        self.run(x, count, first_sample=first, eps=eps, z_noise=z_noise, first_k=1,
                 global_samples=None if self.pg is None else samples)
        sum_logp, sum_prob, first_logp, _ = self._sums()
        probs = sum_prob / samples
        rest = (sum_logp - first_logp) / max(samples - 1, 1)
        return {"entropy": -(probs * torch.log(probs)).sum(1), "pred": rest.argmax(1), "mean_prob": probs}


@torch.no_grad()
def mf_outofsample(net, x, samples, medimod=False, seed=None, samples_per_launch=32, predictor=None):
    """`outofsample` of the MF script for one batch (LBBNN-GP-MF.py:450-502) on the batched MC kernels (lbbnn.mf.MCPredictor):
    `samples` stochastic forwards with fresh weights; medimod=True fixes the inclusion masks to the median-probability model
    [alpha > 0.5] (MF:462-465) instead of drawing gamma ~ Bernoulli(alpha).  Returns the predictive entropy of the averaged
    row-normalised expit (MF:478-494), the prediction from outputs[1:TEST_SAMPLES].mean(0) (MF:496-498) and the predictor."""
    from . import mf
    mc = predictor or mf.MCPredictor(net, batch=x.shape[0], seed=seed, samples_per_launch=min(samples_per_launch, max(samples, 1)))
    masks = mf.median_probability_masks(net) if medimod else None
    mc.run(x, 1, first_sample=0, masks=masks)                    # sample 0 alone: the reference leaves it out of `output`
    l0, p0 = mc.sum_logp.clone(), mc.sum_prob.clone()
    if samples > 1:
        mc.run(x, samples - 1, first_sample=1, masks=masks)
        lr, pr = mc.sum_logp, mc.sum_prob
    else:
        lr, pr = torch.zeros_like(l0), torch.zeros_like(p0)
    probs = (p0 + pr) / samples
    return {"entropy": -(probs * torch.log(probs)).sum(1), "pred": (lr / max(samples - 1, 1)).argmax(1), "mean_prob": probs,
            "predictor": mc}
