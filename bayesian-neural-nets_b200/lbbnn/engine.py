"""Whole-step runner for the LRT network: forward, loss, backward and Adam as one CUDA-graph replay.

Reference: the body of `train` (LBBNN-GP-MF-LRT.py:217-229) for one minibatch --
net(data, sample=True), nll_loss(sum) + kl/NUM_BATCHES, backward, optimizer.step().
The eager drop-in modules (lrt.py) launch the same kernels one Python call at a time; at MNIST shape
the step is a few tens of microseconds of GPU work, so the Python/launch overhead dominates unless the
sequence is captured once and replayed.  Parameters, gradients and Adam state live in flat buffers
(one Adam launch); the nn.Parameters of the network are re-pointed at views of the flat buffer, so the
module keeps working (state_dict, eager forward) while the trainer owns the storage.
"""
from ctypes import create_string_buffer as C_create_string_buffer
from ctypes import c_void_p as C_void_p
from ctypes import c_float as C_float

import os

import torch

from . import _capi as K
from . import lrt as _lrt

_PARAM_NAMES = ("weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho")


def _pad4(n):
    return (n + 3) // 4 * 4


def shard_blocks(total_blocks, world, rank):
    """[lo, hi) of the 1024-element blocks of an Adam table that `rank` of `world` updates under the sharded data-parallel
    update: contiguous runs of ceil(total / world) blocks, the last ranks' runs shorter or empty."""
    per = -(-int(total_blocks) // int(world))
    return min(total_blocks, rank * per), min(total_blocks, (rank + 1) * per)


def check_replicas(process_group, params, what):
    """Start of data-parallel training: every rank must make the same parameter-side draws -- same lbbnn and torch CUDA
    seeds (checked), same modules in the same order (the parameter shapes are checked); then rank 0's parameters are
    broadcast.  Raises LbbnnError naming `what` on a mismatch."""
    import torch.distributed as dist
    mine = (_lrt.current_seed(), torch.cuda.initial_seed(), [tuple(p.shape) for p in params])
    allv = [None] * dist.get_world_size(process_group)
    dist.all_gather_object(allv, mine, group=process_group)
    if any(v != allv[0] for v in allv):
        raise K.LbbnnError("%s: ranks differ in lbbnn.manual_seed / torch.manual_seed or in the network (seed, torch seed, "
                           "parameter shapes per rank: %r)" % (what, [v[:2] for v in allv]))
    src = dist.get_global_rank(process_group, 0)
    with torch.no_grad():
        for p in params:
            dist.broadcast(p.data, src=src, group=process_group)


class LRTTrainer:
    def __init__(self, net, batch_size, num_batches, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, seed=None,
                 use_graph=True, inject_noise=False, process_group=None, fused=None, materialize_grads=True):
        """fused: run the step as the single persistent kernel of csrc/lrt_step.cu (None = whenever it applies:
        batch <= 128, <= 8 layers); False = one launch sequence per layer (csrc/lrt_f32.cu).
        materialize_grads: also write the parameter gradients to `.grad` (the fused kernel otherwise consumes
        them in registers inside the Adam update)."""
        K.require_device()
        self.net = net
        self.layers = list(net.layers)
        self.B = int(batch_size)
        self.num_batches = int(num_batches)
        self.lr, self.betas, self.eps = float(lr), betas, float(eps)
        self.seed = _lrt.current_seed() if seed is None else int(seed)
        self.pg = process_group
        self.world = 1 if process_group is None else torch.distributed.get_world_size(process_group)
        self.rank = 0 if process_group is None else torch.distributed.get_rank(process_group)
        dev = self.layers[0].weight_mu.device
        if dev.type != "cuda":
            raise K.LbbnnError("LRTTrainer needs the network on a CUDA device (no CPU fallback)")
        self.device = dev
        can_fuse = self.B <= 128 and len(self.layers) <= K.STEP_MAX_LAYERS
        if fused and not can_fuse:
            raise K.LbbnnError("the fused step kernel needs batch <= 128 and <= 8 layers")
        self.fused = can_fuse if fused is None else bool(fused)
        self.materialize_grads = bool(materialize_grads)

        # ---- flat parameter / gradient / Adam-state storage ------------------------------------
        offs, total = [], 0
        for l in self.layers:
            for name in _PARAM_NAMES:
                p = getattr(l, name)
                offs.append((l, name, total, p.numel(), p.shape))
                total += _pad4(p.numel())
        self.n_flat = total
        # data parallel + fused step kernel: parameters and workspace in one NVSwitch-multicast arena, exchange inside the launch
        self._dp_arena = None
        if self.fused and self.pg is not None and not self.materialize_grads:
            self._try_dp_arena(total, [(l.in_features, l.out_features) for l in self.layers])
        self.flat = self._dp_arena["flat"] if self._dp_arena else torch.zeros(total, dtype=torch.float32, device=dev)
        self.gflat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.adam_coef = torch.zeros(2, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for l, name, off, n, shape in offs:
                p = getattr(l, name)
                view = self.flat[off:off + n].view(shape)
                view.copy_(p.data)
                p.data = view
                p.grad = self.gflat[off:off + n].view(shape)
        self._offsets = {(id(l), name): off for l, name, off, n, shape in offs}

        # ---- static activations / scratch --------------------------------------------------------
        sizes = [(l.in_features, l.out_features) for l in self.layers]
        f32 = dict(dtype=torch.float32, device=dev)
        self.x = torch.zeros(self.B, sizes[0][0], **f32)
        self.y = torch.zeros(self.B, dtype=torch.int64, device=dev)
        if self.fused:
            self._init_fused(sizes, inject_noise, use_graph)
            return
        self.acts = [torch.zeros(self.B, o, **f32) for _, o in sizes]
        self.dsf = [torch.zeros(self.B, o, **f32) for _, o in sizes]     # eps/(2 sqrt(var_b)) per layer
        self.mv = [None] + [torch.zeros(K.lrt_mv_bytes(i, o) // 4, **f32) for i, o in sizes[1:]]  # M,V kept for dX
        self.gbuf = [torch.zeros(self.B, o, **f32) for _, o in sizes]   # dL/d(pre-activation) per layer
        self.eps_in = [torch.zeros(self.B, o, **f32) for _, o in sizes] if inject_noise else None
        self.stats = torch.zeros(1 + len(sizes), **f32)                  # [nll, kl_1 .. kl_L]
        nbytes = max(K.lrt_workspace_bytes(self.B, i, o) for i, o in sizes)
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self.x_host = torch.zeros(self.B, sizes[0][0], dtype=torch.float32).pin_memory()
        self.y_host = torch.zeros(self.B, dtype=torch.int64).pin_memory()
        self.stats_host = torch.zeros(1 + len(sizes), dtype=torch.float32).pin_memory()
        self.kernels_per_step = 0
        self.graph = None
        if use_graph:
            self._capture()

    # ---- fused single-kernel step (csrc/lrt_step.cu) ------------------------------------------------
    def _try_dp_arena(self, n_flat, sizes):
        """LBBNN_DP_ALLREDUCE = auto | sharded: one symmetric-memory arena [parameters | step workspace | signal pad | KL
        exchange] bound to an NVSwitch multicast object, for the in-launch sharded update (lbbnn_step_dp).  Leaves
        self._dp_arena None (two launches around an all-reduce of the raw gradients) when the fabric has no multicast."""
        import os
        # measured at 2 GPUs (us / step, 109-112 on one): two launches around torch's two-shot all-reduce 137; the exchange
        # inside the launch 140 (multicast) / 135-150 (peer-to-peer) -- four dependent NVLink round trips of ~6 us each
        # (flags, pull, push + fence, flags) cost what the second launch and the all-reduce kernel cost, so "auto" keeps the
        # two-launch form and the in-launch forms are opt-in (profiles/r02_step_dp_phases.txt)
        mode = os.environ.get("LBBNN_DP_ALLREDUCE", "auto")
        if mode not in ("sharded", "sharded_p2p"):
            return
        try:
            import torch.distributed._symmetric_memory as symm_mem
            probe = K.Step()
            probe.n_layers, probe.batch = len(sizes), self.B
            for i, (fi, fo) in enumerate(sizes):
                probe.layer[i].in_features, probe.layer[i].out_features = fi, fo
            ws_bytes = int(K.lib.lbbnn_lrt_step_workspace_bytes(probe))
            if ws_bytes == 0 or any((fi * fo) % 4 for fi, fo in sizes):
                raise RuntimeError("shape not supported by the sharded update")
            a256 = lambda v: (v + 255) // 256 * 256  # noqa: E731
            off_ws = a256(4 * n_flat)
            off_sig = off_ws + a256(ws_bytes)
            off_klx = off_sig + 256
            nbytes = off_klx + a256(8 * self.world * K.STEP_MAX_LAYERS)
            arena = symm_mem.empty(nbytes, dtype=torch.uint8, device=self.device)
            arena.zero_()
            hdl = symm_mem.rendezvous(arena, self.pg.group_name)
            if int(hdl.multicast_ptr) == 0 and mode != "sharded_p2p":
                raise RuntimeError("no multicast support on this fabric")
            hdl.barrier(channel=0)
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            if mode != "auto":
                raise
            self._ar_error = repr(e)
            return
        self._dp_arena = dict(p2p=(mode == "sharded_p2p"), arena=arena, hdl=hdl, flat=arena[:4 * n_flat].view(torch.float32), off_ws=off_ws, ws_bytes=ws_bytes,
                              off_sig=off_sig, off_klx=off_klx, epoch=torch.zeros(1, dtype=torch.int64, device=self.device))

    def _init_fused(self, sizes, inject_noise, use_graph):
        dev, f32 = self.device, dict(dtype=torch.float32, device=self.device)
        self.eps_in = [torch.zeros(self.B, o, **f32) for _, o in sizes] if inject_noise else None
        self.stats = torch.zeros(1 + len(sizes), **f32)
        st = K.Step()
        st.n_layers, st.batch = len(self.layers), self.B
        for i, l in enumerate(self.layers):
            sl = st.layer[i]
            sl.in_features, sl.out_features = l.in_features, l.out_features
            sl.off_weight_mu, sl.off_weight_rho, sl.off_lambdal, sl.off_bias_mu, sl.off_bias_rho = (
                self._offsets[(id(l), n)] for n in _PARAM_NAMES)
            sl.eps = K.ptr(self.eps_in[i]) if inject_noise else None
            sl.priors, sl.var_mode = l.cfg.priors, l.cfg.var_mode
        st.flat, st.exp_avg, st.exp_avg_sq = K.ptr(self.flat), K.ptr(self.exp_avg), K.ptr(self.exp_avg_sq)
        st.grad = K.ptr(self.gflat) if self.materialize_grads else None
        st.x, st.y, st.step_dev = K.ptr(self.x), K.ptr(self.y, torch.int64), K.ptr(self.step_dev, torch.int64)
        st.seed = (self.seed + 0x9E3779B97F4A7C15 * self.rank) & (2 ** 64 - 1)
        st.lr, st.beta1, st.beta2, st.eps = self.lr, self.betas[0], self.betas[1], self.eps
        # the update phase adds the KL gradient AFTER the raw gradients were sum-reduced, once and identically on every rank
        # (SURVEY.md §8e), so it is NOT pre-divided by the world size -- unlike the per-layer path below, whose finalize
        # kernels add it on every rank BEFORE the all-reduce of .grad
        st.kl_scale = 1.0 / self.num_batches
        st.stats = K.ptr(self.stats)
        self._step_desc = st
        nbytes = int(K.lib.lbbnn_lrt_step_workspace_bytes(st))
        if nbytes == 0:
            raise K.LbbnnError("fused step: " + K.lib.lbbnn_last_error().decode())
        self.allreduce = "none"
        self.ws = None
        self._step_dp = None
        if self._dp_arena is not None:
            A = self._dp_arena
            assert nbytes <= A["ws_bytes"]
            self.ws = A["arena"][A["off_ws"]:A["off_ws"] + A["ws_bytes"]]
            mc, peers = int(A["hdl"].multicast_ptr), [int(p) for p in A["hdl"].buffer_ptrs]
            dp = K.StepDp()
            dp.world, dp.rank = self.world, self.rank
            dp.flat_mc, dp.ws_mc = mc, mc + A["off_ws"]
            for p in range(self.world):
                dp.signal[p], dp.klx[p] = peers[p] + A["off_sig"], peers[p] + A["off_klx"]
            dp.epoch = A["epoch"].data_ptr()
            dp.use_p2p = 1 if A["p2p"] else 0
            for p in range(self.world):
                dp.flat_peer[p], dp.ws_peer[p] = peers[p], peers[p] + A["off_ws"]
            self._step_dp = dp
            import ctypes
            st.dp = ctypes.pointer(dp)
            self.allreduce = ("p2p-sharded-update" if A["p2p"] else "nvls-sharded-update") + " (inside the step kernel)"
        elif self.pg is not None:
            self.ws = self._symmetric_workspace(nbytes)                   # NVLink/NVSwitch peer-mapped, for the all-reduce
        if self.ws is None:
            self.ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)  # zero-filled once (barrier ticket lives in it)
            self.allreduce = "nccl" if self.pg is not None else "none"
        self.raw = self.ws[:4 * int(K.lib.lbbnn_lrt_step_raw_floats(st))].view(torch.float32)
        buf = C_create_string_buffer(2048)
        K.check(K.lib.lbbnn_lrt_step_describe(st, buf, 2048))
        self.schedule = buf.value.decode()
        self.x_host = torch.zeros(self.B, sizes[0][0], dtype=torch.float32).pin_memory()
        self.y_host = torch.zeros(self.B, dtype=torch.int64).pin_memory()
        self.stats_host = torch.zeros(1 + len(sizes), dtype=torch.float32).pin_memory()
        self.kernels_per_step = 1 if (self.pg is None or self._step_dp is not None) else 2
        self.graph = None
        if use_graph:
            self._capture()

    def owned_range(self, layer_index, name):
        """Element range [lo, hi) of parameter `name` of layer `layer_index` whose Adam moments THIS rank maintains: all of it,
        except under the in-launch sharded data-parallel update, where a rank owns a contiguous 1 / world of the weight quads of
        ALL layers taken as one index space (layer 0 first) and rank 0 owns the biases."""
        n = getattr(self.layers[layer_index], name).numel()
        if getattr(self, "_step_dp", None) is None:
            return 0, n
        if name.startswith("bias"):
            return (0, n) if self.rank == 0 else (0, 0)
        nq = [l.weight_mu.numel() // 4 for l in self.layers]
        total = sum(nq)
        per = -(-total // self.world)
        g0, g1 = min(total, self.rank * per), min(total, (self.rank + 1) * per)
        base = sum(nq[:layer_index])
        lo, hi = max(g0, base) - base, min(g1, base + nq[layer_index]) - base
        return (4 * lo, 4 * hi) if hi > lo else (0, 0)

    def _symmetric_workspace(self, nbytes):
        """The step workspace in symmetric (peer-mapped) memory so that the all-reduce of its raw-gradient head can be
        the in-switch multimem reduction over NVLink/NVSwitch (one kernel, no ring steps) instead of NCCL's.
        LBBNN_DP_ALLREDUCE = auto (default) | multimem | two_shot | nccl.  Measured on 8xB200, 4.5 MB, us/step:
        2 ranks nccl 157 / multimem 155 / two_shot 137;  8 ranks nccl 175 / two_shot 142 / multimem 134 -> auto picks
        two_shot up to 2 ranks and multimem beyond.  Returns None when unavailable (NCCL is used)."""
        import os
        mode = os.environ.get("LBBNN_DP_ALLREDUCE", "auto")
        if mode == "auto":
            mode = "two_shot" if self.world <= 2 else "multimem"
        if mode == "nccl":
            return None
        try:
            import torch.distributed._symmetric_memory as symm_mem
            name = self.pg.group_name
            ws = symm_mem.empty(nbytes, dtype=torch.uint8, device=self.device)
            ws.zero_()
            symm_mem.rendezvous(ws, name)
            probe = ws[:256].view(torch.float32)
            op = torch.ops.symm_mem.multimem_all_reduce_ if mode == "multimem" else torch.ops.symm_mem.two_shot_all_reduce_
            op(probe, "sum", name)                    # fails here (not inside a capture) if the fabric lacks the feature
            torch.cuda.synchronize()
            ws.zero_()
            torch.cuda.synchronize()
            torch.distributed.barrier(group=self.pg)
            self.allreduce, self._ar_op, self._ar_group = mode, op, name
            return ws
        except Exception as e:  # noqa: BLE001
            self._ar_error = repr(e)
            return None

    def _enqueue_fused(self):
        st, ws = K.current_stream(), self.ws
        if self.pg is None or self._step_dp is not None:     # one launch; data parallel: the exchange happens inside it
            K.check(K.lib.lbbnn_lrt_step_f32(self._step_desc, 3, ws.data_ptr(), ws.numel(), st))
        else:   # data parallel: sum-reduce the raw (dM, dV, bias column sums), then chain rule + KL + Adam
            K.check(K.lib.lbbnn_lrt_step_f32(self._step_desc, 1, ws.data_ptr(), ws.numel(), st))
            if self.allreduce == "nccl":
                torch.distributed.all_reduce(self.raw, group=self.pg)
            else:
                self._ar_op(self.raw, "sum", self._ar_group)
            K.check(K.lib.lbbnn_lrt_step_f32(self._step_desc, 2, ws.data_ptr(), ws.numel(), st))

    # ---- the launch sequence ------------------------------------------------------------------------
    def _noise(self, i):
        if self.eps_in is not None:
            return K.make_noise(self.eps_in[i])
        # stream = layer index + step * n_layers (+ rank offset in the seed so ranks draw disjoint noise)
        return K.make_noise(None, self.seed + 0x9E3779B97F4A7C15 * self.rank, i, self.step_dev, len(self.layers))

    def _enqueue(self):
        if self.fused:
            return self._enqueue_fused()
        st = K.current_stream()
        L = len(self.layers)
        n_launch = 0
        descs = [K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
                 for l in self.layers]
        ws, wsn = self.ws.data_ptr(), self.ws.numel()
        h = self.x
        for i, l in enumerate(self.layers):
            flags = K.FLAG_SAMPLE | K.FLAG_KL | (K.FLAG_RELU if i < L - 1 else 0)
            K.check(K.lib.lbbnn_lrt_f32_fwd(descs[i], K.ptr(h), self.B, self._noise(i), l.cfg.priors, l.cfg.var_mode,
                                            flags, K.ptr(self.acts[i]), K.ptr(self.dsf[i]),
                                            self.stats[1 + i:].data_ptr(), K.ptr(self.mv[i], allow_none=True),
                                            ws, wsn, st))
            n_launch += 3
            h = self.acts[i]
        C = self.layers[-1].out_features
        # loss head; also bumps the step counter: noise above used step t-1, Adam below uses t
        K.check(K.lib.lbbnn_logsoftmax_nll_f32(K.ptr(self.acts[-1]), K.ptr(self.y, torch.int64), self.B, C, None,
                                               self.stats.data_ptr(), K.ptr(self.gbuf[-1]), 1.0,
                                               K.ptr(self.step_dev, torch.int64), ws, wsn, st))
        n_launch += 1
        klg = 1.0 / (self.num_batches * self.world)   # KL is replicated on every rank: its grad is added once
        for i in reversed(range(L)):
            l = self.layers[i]
            xin = self.x if i == 0 else self.acts[i - 1]
            g = l.weight_mu.grad, l.weight_rho.grad, l.lambdal.grad, l.bias_mu.grad, l.bias_rho.grad
            K.check(K.lib.lbbnn_lrt_f32_bwd_params(
                descs[i], K.ptr(xin), self.B, K.ptr(self.gbuf[i]), K.ptr(self.dsf[i]), l.cfg.priors,
                l.cfg.var_mode, K.FLAG_SAMPLE, None, klg, K.LayerGrads(*[t.data_ptr() for t in g], None), ws, wsn, st))
            n_launch += 2
            if i > 0:
                K.check(K.lib.lbbnn_lrt_f32_bwd_input(
                    descs[i], K.ptr(xin), self.B, K.ptr(self.gbuf[i]), K.ptr(self.dsf[i]), l.cfg.priors,
                    l.cfg.var_mode, K.FLAG_SAMPLE | K.FLAG_MASK_DX, K.ptr(self.mv[i]), K.ptr(self.gbuf[i - 1]),
                    ws, wsn, st))
                n_launch += 2
        if self.pg is not None:
            torch.distributed.all_reduce(self.gflat, group=self.pg)
        K.check(K.lib.lbbnn_adam_f32(K.ptr(self.flat), K.ptr(self.gflat), K.ptr(self.exp_avg), K.ptr(self.exp_avg_sq),
                                     self.n_flat, self.lr, self.betas[0], self.betas[1], self.eps,
                                     K.ptr(self.step_dev, torch.int64), K.ptr(self.adam_coef), st))
        n_launch += 2
        self.kernels_per_step = n_launch

    def _capture(self):
        # side stream warm-up (also sizes nothing: all buffers are preallocated), then capture
        tensors = self._train_state() if hasattr(self, "_train_state") else (self.flat, self.exp_avg, self.exp_avg_sq,
                                                                             self.step_dev)
        state = [t.clone() for t in tensors]
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._enqueue()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        for t, saved in zip(tensors, state):
            t.copy_(saved)   # the warm-up step must not count as training
        if getattr(self, "pg", None) is not None and hasattr(self, "_train_state"):
            # data-parallel update: a peer's replay writes this rank's parameters, so no rank may replay before all restored
            torch.cuda.synchronize()
            torch.distributed.barrier(group=self.pg)
        if hasattr(self, "_after_restore"):
            self._after_restore()   # state derived from the parameters (carried bf16 operands)
        self.graph = torch.cuda.CUDAGraph()
        # wide trainer: the main path is captured on a HIGH-priority stream (kernel nodes inherit it): whenever a GEMM and a
        # side-stream pass (next layer's prologue, an update) become ready together, the block scheduler places the GEMM's
        # persistent CTAs first and the side kernel fills what is left of each SM -- a 4096-CTA prologue that got there first
        # kept the next forward GEMM (one ~200 KB CTA per SM) off the SMs until it had drained
        cap = getattr(self, "capture_stream", None)
        with (torch.cuda.graph(self.graph, stream=cap) if cap is not None else torch.cuda.graph(self.graph)):
            self._enqueue()

    def _retarget_inputs(self, x, y):
        """Point the step at another (x, y) pair of device buffers (the next capture / enqueue reads them)."""
        self.x, self.y = x, y
        st = getattr(self, "_step_desc", None)
        if st is not None:
            st.x, st.y = K.ptr(x), K.ptr(y, torch.int64)

    def _slot_graph(self, slot_x, slot_y):
        """The captured step once more, reading its batch from (slot_x, slot_y) instead of self.x / self.y: step_async
        replays the graph of the upload slot it has just filled, so the batch is not copied device-to-device first (134 MB
        per step at the wide shape, two launches on the critical stream at the MNIST shape).  Same private pool as the main
        graph; nothing in _enqueue allocates."""
        x0, y0 = self.x, self.y
        self._retarget_inputs(slot_x, slot_y)
        try:
            g = torch.cuda.CUDAGraph()
            cap = getattr(self, "capture_stream", None)
            kw = dict(pool=self.graph.pool())
            with (torch.cuda.graph(g, stream=cap, **kw) if cap is not None else torch.cuda.graph(g, **kw)):
                self._enqueue()
        finally:
            self._retarget_inputs(x0, y0)
        return g

    # ---- public API -----------------------------------------------------------------------------------
    def step_device(self):
        """One training step on the data already in self.x / self.y (device resident)."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self._enqueue()

    def step(self, x_host, y_host, read_loss=True):
        """One training step from HOST tensors: (pinned staging ->) H2D -> step -> D2H of [nll, kl...].
        Pinned inputs are uploaded straight from the caller's buffer."""
        if x_host.is_pinned() and y_host.is_pinned() and x_host.is_contiguous():
            self.x.copy_(x_host.reshape(self.x.shape), non_blocking=True)
            self.y.copy_(y_host, non_blocking=True)
        else:
            self.x_host.copy_(x_host.reshape(self.x_host.shape))
            self.y_host.copy_(y_host)
            self.x.copy_(self.x_host, non_blocking=True)
            self.y.copy_(self.y_host, non_blocking=True)
        self.step_device()
        if not read_loss:
            return None
        self.stats_host.copy_(self.stats, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._stats_dict(self.stats_host)

    def _stats_dict(self, st):
        """[nll, kl_1..kl_L] of the step.  Data parallel: `nll` (and so `loss`) is THIS RANK's shard of the minibatch only
        (the sum over ranks is never formed on the device); the KL terms are replicated."""
        nll = float(st[0])
        kl = float(st[1:].sum())
        return {"nll": nll, "kl": kl, "loss": nll + kl / self.num_batches}

    def step_async(self, x_host, y_host):
        """Pipelined form of step(): uploads this batch on a copy stream while the previous step is still running,
        enqueues the step, and returns the statistics of the PREVIOUS step (None on the first call) -- every step's
        [nll, kl...] still crosses to the host, one call late.  flush() returns the last one."""
        if not hasattr(self, "_pipe"):
            dev = self.device
            self._pipe = dict(
                copy_stream=torch.cuda.Stream(device=dev), n=0,
                xs=[torch.empty_like(self.x) for _ in range(2)], ys=[torch.empty_like(self.y) for _ in range(2)],
                xh=[None, None], yh=[None, None],        # pinned staging, only allocated for pageable inputs
                sh=[torch.empty_like(self.stats_host).pin_memory() for _ in range(2)],
                up=[torch.cuda.Event() for _ in range(2)], used=[torch.cuda.Event() for _ in range(2)],
                done=[None, None],
                slot_graphs=([None, None] if (getattr(self, "graph", None) is not None and hasattr(self, "_slot_graph") and
                                              os.environ.get("LBBNN_SLOT_GRAPHS", "1") == "1") else None))
        P = self._pipe
        i = P["n"] & 1
        cur = torch.cuda.current_stream()
        pinned = x_host.is_pinned() and y_host.is_pinned() and x_host.is_contiguous()
        if not pinned:                                   # stage through this slot's pinned buffers
            if P["xh"][i] is None:
                P["xh"][i] = torch.empty_like(self.x_host).pin_memory()
                P["yh"][i] = torch.empty_like(self.y_host).pin_memory()
            if P["n"] >= 2:
                P["up"][i].synchronize()                 # the upload that last read them has finished
            P["xh"][i].copy_(x_host.reshape(P["xh"][i].shape))
            P["yh"][i].copy_(y_host)
        src_x, src_y = (x_host.reshape(self.x.shape), y_host) if pinned else (P["xh"][i], P["yh"][i])
        with torch.cuda.stream(P["copy_stream"]):
            if P["n"] >= 2:
                P["copy_stream"].wait_event(P["used"][i])    # the step that consumed this device slot is past its copy
            P["xs"][i].copy_(src_x, non_blocking=True)
            P["ys"][i].copy_(src_y, non_blocking=True)
            P["up"][i].record(P["copy_stream"])
        cur.wait_event(P["up"][i])
        if P["slot_graphs"] is not None:                 # the step captured against THIS slot's buffers: no device copy
            if P["slot_graphs"][i] is None:
                P["slot_graphs"][i] = self._slot_graph(P["xs"][i], P["ys"][i])
            P["slot_graphs"][i].replay()
            P["used"][i].record(cur)                     # the slot is free again once this step has run
        else:
            self.x.copy_(P["xs"][i], non_blocking=True)
            self.y.copy_(P["ys"][i], non_blocking=True)
            P["used"][i].record(cur)
            self.step_device()
        P["sh"][i].copy_(self.stats, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(cur)
        P["done"][i] = ev
        P["n"] += 1
        prev = P["done"][i ^ 1]
        if prev is None:
            return None
        prev.synchronize()
        return self._stats_dict(P["sh"][i ^ 1])

    def flush(self):
        """Statistics of the last step enqueued by step_async()."""
        P = getattr(self, "_pipe", None)
        if P is None or P["n"] == 0:
            return None
        i = (P["n"] - 1) & 1
        P["done"][i].synchronize()
        return self._stats_dict(P["sh"][i])

    @property
    def h2d_bytes_per_step(self):
        return self.x_host.numel() * 4 + self.y_host.numel() * 8

    @property
    def d2h_bytes_per_step(self):
        return self.stats_host.numel() * 4


class LRTTensorCoreTrainer:
    """Whole-step runner for WIDE LRT stacks in bf16 on the tensor cores (BASELINE.json configs[4]:
    4096-4096-4096-10, batch 8192).  Master parameters, KL, chain rule and Adam stay fp32; the GEMM
    operands (x, x^2, M, V and the backward's dE, dS) are bf16 with fp32 accumulation in TMEM.

    Forward and dW GEMM pairs of EVERY layer run on the tcgen05 dual-GEMM kernel (ragged shapes such as
    the 10-class output are zero-filled by TMA).  The input-gradient GEMM of a layer whose out_features
    is not a multiple of 8 (the classifier: its contraction dim would break the TMA pitch) runs on the
    fp32 SIMT kernel instead.  Same reference step as LRTTrainer (LBBNN-GP-MF-LRT.py:217-229).

    fused_update (default): every layer owns a raw-gradient buffer [dM | dV | bias column sums]; as soon as its dW GEMM
    is done, chain rule + KL gradient + Adam run as ONE pass over it (lbbnn_lrt_f32_finalize_adam: parameters and Adam
    state updated in place, the three parameter gradients never stored).  Data parallel: that buffer -- 2/3 of the
    bytes of the parameter gradients it determines -- is all-reduced on a communication stream, layer by layer, while
    the main stream goes on with the input-gradient GEMM and the earlier layers' backward.  fused_update=False keeps the
    separate finalize / all-reduce of .grad / Adam passes (and leaves gradients in `.grad`).
    """

    def __init__(self, net, batch_size, num_batches, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, seed=None,
                 use_graph=True, inject_noise=False, process_group=None, fused_update=True, fused_prologue=True,
                 fused_head_dx=True, overlap=True, small_head=False, in_place=None, carry_operands=False):
        """in_place (default: whenever the stack allows it -- every layer but a <= 12-output head has out_features % 8 == 0):
        the backward GEMMs read dE, dS, x, x^2, M, V where the forward left them (tcgen05 MN-major operands) instead of
        transposed copies, the dX epilogue emits the bias-gradient partial sums, and on one GPU with fused_update the dW
        GEMM's epilogue applies chain rule + KL gradient + Adam to its accumulators (lbbnn_tc_lrt_dw_adam): dM / dV never
        reach memory.  in_place=False keeps the r01 sequence (transposed K-major operands, separate update pass).
        carry_operands (off): with that fused update the epilogue can also write the NEXT step's bf16 M, V and KL partial sums
        from the parameters it has just updated (lbbnn_tc_lrt_dw_adam_next), so the layer needs no prologue pass per step (its
        operands become derived state: call refresh_operands() after changing parameters from outside).  Measured on one box:
        3.92-4.00 ms / step with it against 3.53 without -- the prologue's exp / log1p / log work is cheap at full occupancy
        (91 us per layer, 91 % issue-active) but not on the GEMM's 8 epilogue warps per SM, where it outlasts the MMAs of the
        next tile.  Kept as a tested option."""
        K.require_device()
        self.net = net
        self.layers = list(net.layers)
        self.fused_prologue = bool(fused_prologue)
        self.overlap = bool(overlap)
        # <= 12-output layers: forward (if last) and dW on the CUDA-core row-streaming kernels instead of 128-wide tensor-core
        # tiles.  Off by default: measured 138 / 136 us against 81 / 69 us at the wide shape (shared-memory fill and too few
        # bytes in flight per SM); kept as a tested alternative for heads whose in_features break the TMA pitch.
        self.small_head = bool(small_head)
        L = len(self.layers)
        for l in self.layers:
            if l.in_features % 8:
                raise K.LbbnnError("tensor-core layers need in_features divisible by 8 (TMA pitch)")
        self.B = int(batch_size)
        if self.B % 8:
            raise K.LbbnnError("batch must be divisible by 8 (the dW GEMM contracts over it)")
        self.num_batches = int(num_batches)
        self.lr, self.betas, self.eps = float(lr), betas, float(eps)
        self.seed = _lrt.current_seed() if seed is None else int(seed)
        self.pg = process_group
        self.world = 1 if process_group is None else torch.distributed.get_world_size(process_group)
        self.rank = 0 if process_group is None else torch.distributed.get_rank(process_group)
        dev = self.layers[0].weight_mu.device
        self.device = dev

        B = self.B
        sizes = [(l.in_features, l.out_features) for l in self.layers]
        self.sizes = sizes
        self.fused_update = bool(fused_update)
        # input-gradient GEMM off the tensor cores: a head with <= 12 outputs goes through the fused CUDA-core kernel that
        # also stages the layer below's dE / dS / column sums (lbbnn_tc_lrt_bwd_input_small); other widths that break the
        # TMA pitch fall back to the fp32 SIMT GEMM + separate staging passes
        self.small_dx = [o <= 12 and o % 8 != 0 and fused_head_dx for _, o in sizes]
        self.simt_dx = [o % 8 != 0 and not sm for (_, o), sm in zip(sizes, self.small_dx)]
        can_in_place = (self.fused_prologue and L >= 2 and all(o % 8 == 0 for _, o in sizes[:-1]) and
                        (sizes[-1][1] % 8 == 0 or self.small_dx[-1]) and not self.small_head)
        if in_place and not can_in_place:
            raise K.LbbnnError("in_place needs out_features % 8 == 0 for every layer but a <= 12-output head (fused_head_dx)")
        self.in_place = can_in_place if in_place is None else bool(in_place)

        offs, total = [], 0
        for l in self.layers:
            for name in _PARAM_NAMES:
                p = getattr(l, name)
                offs.append((l, name, total, p.numel(), p.shape))
                total += _pad4(p.numel())
        self.n_flat = total
        f32 = dict(dtype=torch.float32, device=dev)
        bf = dict(dtype=torch.bfloat16, device=dev)
        # data parallel, fused update, operands in place: parameters and raw gradients live in ONE symmetric-memory arena
        # bound to an NVSwitch multicast object, and every layer's update is the sharded NVLS kernel
        # (lbbnn_lrt_f32_finalize_adam_dp: in-switch reduce-scatter of (dM, dV) -> chain rule + KL + Adam on the owner ->
        # multicast store of the new parameters).  LBBNN_DP_UPDATE = auto (default) | sharded | nccl.
        self.dp_sharded = False
        self.allreduce = "nccl" if self.world > 1 else "none"
        self._raw_off = {}
        arena_floats = total
        for li, (i, o) in enumerate(sizes):
            self._raw_off[li] = arena_floats
            arena_floats += _pad4(2 * o * i + 2 * o)
        if self.world > 1 and self.fused_update and self.in_place:
            self._setup_dp_arena(arena_floats, dev)
        self.flat = self.arena[:total] if self.dp_sharded else torch.zeros(total, **f32)
        self.gflat = torch.zeros(total, **f32)
        self.exp_avg, self.exp_avg_sq = torch.zeros(total, **f32), torch.zeros(total, **f32)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.adam_coef = torch.zeros(2, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for l, name, off, n, shape in offs:
                p = getattr(l, name)
                view = self.flat[off:off + n].view(shape)
                view.copy_(p.data)
                p.data = view
                p.grad = self.gflat[off:off + n].view(shape)
        self.x = torch.zeros(B, sizes[0][0], **f32)
        self.y = torch.zeros(B, dtype=torch.int64, device=dev)
        self.x_bf, self.x2_bf = torch.zeros(B, sizes[0][0], **bf), torch.zeros(B, sizes[0][0], **bf)
        maxnk = max(i * o for i, o in sizes)
        if not self.in_place:
            self.xT_bf, self.x2T_bf = torch.zeros(sizes[0][0], B, **bf), torch.zeros(sizes[0][0], B, **bf)
            self.M32, self.V32 = torch.zeros(maxnk, **f32), torch.zeros(maxnk, **f32)     # prologue out, reused
        if not self.in_place or not bool(fused_update):
            self.dM, self.dV = torch.zeros(maxnk, **f32), torch.zeros(maxnk, **f32)       # dW GEMM out, reused
        self.param_off = {(id(l), name): off for l, name, off, n, shape in offs}
        # side stream: the per-layer update (all-reduce +) chain rule + Adam pass runs there while the main stream goes on
        # with the backward GEMMs, and the next step's prologues (parameters -> bf16 operands + KL) run there ahead of the
        # forward GEMMs that consume them.  Those kernels are bandwidth-bound, have small CTAs (<= 17 KB of shared memory) and
        # fit on an SM next to the resident tensor-core GEMM CTA.
        self.comm_stream = (torch.cuda.Stream(device=dev)
                            if (self.fused_update and (self.world > 1 or self.overlap)) else None)
        self.side_prologue = self.fused_prologue and self.overlap and self.comm_stream is not None
        self.capture_stream = (torch.cuda.Stream(device=dev, priority=-1)
                               if (self.comm_stream is not None and os.environ.get("LBBNN_WIDE_PRIORITY", "1") == "1") else None)
        self.tc = []
        for li, (i, o) in enumerate(sizes if not self.in_place else []):
            last = li == L - 1
            need_g32 = last or self.simt_dx[li + 1]        # dL/d(pre-activation) arrives in fp32
            need_act32 = last or self.simt_dx[li + 1]      # fp32 activations: logits / input of a SIMT dX
            tc_dx = li > 0 and not self.simt_dx[li] and not self.small_dx[li]
            d = dict(
                M=torch.zeros(o, i, **bf), V=torch.zeros(o, i, **bf),
                MT=torch.zeros(i, o, **bf) if tc_dx else None, VT=torch.zeros(i, o, **bf) if tc_dx else None,
                mv32=(torch.zeros(K.lrt_mv_bytes(i, o) // 4, **f32)
                      if (li > 0 and (self.simt_dx[li] or self.small_dx[li])) else None),
                act=None if last else torch.zeros(B, o, **bf), act2=None if last else torch.zeros(B, o, **bf),
                actT=None if last else torch.zeros(o, B, **bf), act2T=None if last else torch.zeros(o, B, **bf),
                dsf=torch.zeros(B, o, **f32), act32=torch.zeros(B, o, **f32) if need_act32 else None,
                g32=torch.zeros(B, o, **f32) if need_g32 else None,
                dE=torch.zeros(B, o, **bf), dS=torch.zeros(B, o, **bf),
                dET=torch.zeros(o, B, **bf), dST=torch.zeros(o, B, **bf),
                colsum=torch.zeros(2 * o, **f32),
                klws=torch.empty(max(256, int(K.lib.lbbnn_lrt_bf16_prologue_workspace_bytes(i, o))), dtype=torch.uint8, device=dev),
                eps=torch.zeros(B, o, **f32) if inject_noise else None)
            if self.fused_update:      # [dM | dV | colsum]: what a data-parallel step all-reduces for this layer
                d["raw"] = torch.zeros(2 * o * i + 2 * o, **f32)
                d["colsum"] = d["raw"][2 * o * i:]
            self.tc.append(d)
        for li, (i, o) in enumerate(sizes if self.in_place else []):
            last = li == L - 1
            head = last and self.small_dx[li]        # <= 12 outputs: CUDA-core dX, K-major dE^T / dS^T for its dW
            # the dW GEMM's epilogue does the update: one GPU, fused update, tensor-core-sized layer
            epi_update = self.fused_update and self.world == 1 and not head
            # LBBNN_WIDE_EPI_LAYERS="0,2": only these layers update in their dW GEMM's epilogue; the others run raw dW GEMM +
            # the update pass on the side stream under the following GEMMs (A/B knob; default: every wide layer)
            if epi_update and os.environ.get("LBBNN_WIDE_EPI_LAYERS") is not None:
                epi_update = str(li) in os.environ["LBBNN_WIDE_EPI_LAYERS"].split(",")
            carry = epi_update and bool(carry_operands)
            d = dict(
                head=head, epi_update=epi_update, carry=carry,
                klpart=torch.zeros(int(K.lib.lbbnn_tc_lrt_dw_adam_kl_parts()), dtype=torch.float64, device=dev) if carry else None,
                M=torch.zeros(o, i, **bf), V=torch.zeros(o, i, **bf), MT=None, VT=None,
                mv32=torch.zeros(K.lrt_mv_bytes(i, o) // 4, **f32) if head else None,
                act=None if last else torch.zeros(B, o, **bf), act2=None if last else torch.zeros(B, o, **bf),
                dsf=torch.zeros(B, o, **f32), act32=torch.zeros(B, o, **f32) if last else None,
                g32=torch.zeros(B, o, **f32) if last else None,
                dE=torch.zeros(B, o, **bf), dS=torch.zeros(B, o, **bf),
                dET=torch.zeros(o, B, **bf) if head else None, dST=torch.zeros(o, B, **bf) if head else None,
                colsum=torch.zeros(2 * o, **f32),
                colpart=(torch.zeros(int(K.lib.lbbnn_tc_colsum_part_floats(B, o)), **f32)
                         if (not last and not (li + 1 == L - 1 and self.small_dx[li + 1])) else None),
                klws=torch.empty(max(256, int(K.lib.lbbnn_lrt_bf16_prologue_workspace_bytes(i, o))), dtype=torch.uint8, device=dev),
                eps=torch.zeros(B, o, **f32) if inject_noise else None)
            if self.fused_update and not epi_update:   # [dM | dV | colsum]: what a data-parallel step reduces over the ranks
                if self.dp_sharded:
                    d["raw"] = self.arena[self._raw_off[li]:self._raw_off[li] + 2 * o * i + 2 * o]
                else:
                    d["raw"] = torch.zeros(2 * o * i + 2 * o, **f32)
                d["colsum"] = d["raw"][2 * o * i:]
            self.tc.append(d)
        if self.in_place:          # no transposed input staging, no fp32 M / V scratch; dM / dV only for the unfused update
            self.xT_bf = self.x2T_bf = self.M32 = self.V32 = None
            if self.fused_update:
                self.dM = self.dV = None
        self.kl_next = torch.zeros(L, **f32)     # KL of the layers whose operands are carried from the previous update
        # Layer 0's operands for the NEXT step from a prologue pass at the END of this one: the backward issues layer 1's
        # input gradient and layer 0's dW (+ update) BEFORE layer 1's dW, so that the prologue of the freshly updated layer 0
        # (and its KL term) runs on the side stream under layer 1's dW GEMM, and the next step's first forward GEMM no longer
        # waits ~130 us for it.  M, V of layer 0 become derived state like the carried operands: refresh_operands().
        # Opt-in (LBBNN_WIDE_CARRY0=1): on the power-capped B200s of this pool it measured 3.372 against 3.365 ms per step --
        # the first GEMM does start ~100 us earlier, but the step is bound by its energy under the cap (sw_power_cap, SM
        # clocks 1.69-1.72 of 1.965 GHz), not by that idle stretch (DESIGN.md section 7).
        self.side_carry0 = bool(self.in_place and self.side_prologue and self.fused_update and L >= 3 and
                                not self.tc[0]["carry"] and not self.tc[1]["head"] and
                                os.environ.get("LBBNN_WIDE_CARRY0", "0") == "1")
        for li, d in enumerate(self.tc):
            d["carry_side"] = self.side_carry0 and li == 0
        self.carry_any = self.in_place and any(d["carry"] or d["carry_side"] for d in self.tc)
        if self.carry_any:       # parameters loaded from outside after construction: re-derive the carried operands
            net.register_load_state_dict_post_hook(lambda module, incompatible: self.refresh_operands())
        self.inject = inject_noise
        self.stats = torch.zeros(1 + L, **f32)
        nbytes = max([1 << 20, B // 8 * 4 + 1024] +
                     [int(K.lib.lbbnn_colsum2_workspace_bytes(B, o)) for _, o in sizes] +
                     [int(K.lib.lbbnn_lrt_bf16_prologue_workspace_bytes(i, o)) for i, o in sizes] +
                     [int(K.lib.lbbnn_tc_lrt_bwd_input_small_workspace_bytes(B, i)) for (i, o), sm in zip(sizes, self.small_dx) if sm] +
                     [K.lrt_workspace_bytes(B, i, o) for (i, o), sd in zip(sizes, self.simt_dx) if sd])
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self.x_host = torch.zeros(B, sizes[0][0], dtype=torch.float32).pin_memory()
        self.y_host = torch.zeros(B, dtype=torch.int64).pin_memory()
        self.stats_host = torch.zeros(1 + L, dtype=torch.float32).pin_memory()
        self.kernels_per_step = 0
        self.graph = None
        self.refresh_operands()
        if use_graph:
            self._capture()

    def refresh_operands(self):
        """bf16 M, V and the KL term of every layer whose operands are carried from update to update (carry_operands),
        recomputed from the current parameters: at construction, after the capture's warm-up step was rolled back, and to be
        called by the user after changing parameters from outside the trainer."""
        if not getattr(self, "carry_any", False):
            return
        st, bf = K.current_stream(), torch.bfloat16
        for i, (l, d) in enumerate(zip(self.layers, self.tc)):
            if not (d["carry"] or d["carry_side"]):
                continue
            desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
            K.check(K.lib.lbbnn_lrt_bf16_prologue(desc, l.cfg.priors, l.cfg.var_mode, K.ptr(d["M"], bf), K.ptr(d["V"], bf), None, None,
                                                  None, None, self.kl_next[i:].data_ptr(), d["klws"].data_ptr(), d["klws"].numel(), st))

    _after_restore = refresh_operands

    def _noise(self, i):
        if self.inject:
            return K.make_noise(self.tc[i]["eps"])
        return K.make_noise(None, self.seed + 0x9E3779B97F4A7C15 * self.rank, i, self.step_dev, len(self.layers))

    def _setup_dp_arena(self, arena_floats, dev):
        """Symmetric (peer-mapped) memory with an NVSwitch multicast mapping for [parameters | raw gradients of every layer]
        (torch.distributed._symmetric_memory: cuMemCreate + cuMulticastBindMem under the hood).  Leaves dp_sharded False --
        the NCCL all-reduce + replicated update path -- when the fabric has no multicast support or LBBNN_DP_UPDATE=nccl."""
        import os
        mode = os.environ.get("LBBNN_DP_UPDATE", "auto")
        if mode == "nccl":
            return
        try:
            import torch.distributed._symmetric_memory as symm_mem
            arena = symm_mem.empty(arena_floats, dtype=torch.float32, device=dev)
            arena.zero_()
            hdl = symm_mem.rendezvous(arena, self.pg.group_name)
            mc = int(hdl.multicast_ptr)
            if mc == 0:
                raise RuntimeError("no multicast support on this fabric")
            hdl.barrier(channel=0)
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            if mode == "sharded":
                raise
            self._dp_error = repr(e)
            return
        self.arena, self._symm, self._mc_base = arena, hdl, mc
        self.dp_sharded = True
        self.allreduce = "nvls-sharded-update"

    def owned_range(self, layer_index, name):
        """Element range [lo, hi) of parameter `name` of layer `layer_index` whose Adam moments THIS rank maintains: all of it,
        except under the sharded NVLS update (a contiguous 1 / world of each weight tensor's quads; rank 0 owns the biases)."""
        n = getattr(self.layers[layer_index], name).numel()
        if not self.dp_sharded:
            return 0, n
        if name.startswith("bias"):
            return (0, n) if self.rank == 0 else (0, 0)
        per = -(-(n // 4) // self.world)
        return min(n, 4 * self.rank * per), min(n, 4 * (self.rank + 1) * per)

    def _dp_layer(self, i):
        """Multicast addresses of layer i's parameters and raw-gradient buffer inside the arena."""
        l = self.layers[i]
        mc = lambda name: self._mc_base + 4 * self.param_off[(id(l), name)]  # noqa: E731
        return K.DpLayer(self.world, self.rank, self._mc_base + 4 * self._raw_off[i], mc("weight_mu"), mc("weight_rho"),
                         mc("lambdal"), mc("bias_mu"), mc("bias_rho"))

    def _sharded_layer_update(self, i, desc, main):
        """Layer i's raw gradients are complete on `main` on THIS rank: on the communication stream, wait for the other
        ranks (cross-rank barrier), run the sharded NVLS update, and fence it with a second barrier."""
        l = self.layers[i]
        self.comm_stream.wait_stream(main)
        with torch.cuda.stream(self.comm_stream):
            self._symm.barrier(channel=0)
            K.check(K.lib.lbbnn_lrt_f32_finalize_adam_dp(desc, self._dp_layer(i), l.cfg.priors, l.cfg.var_mode, K.FLAG_SAMPLE,
                                                         1.0 / self.num_batches, self._adam_state(l), K.current_stream()))
            self._symm.barrier(channel=0)

    def _enqueue_in_place(self):
        """The r02 launch sequence: every GEMM reads its operands where the producing kernel left them (see __init__)."""
        st = K.current_stream()
        L, B, bf = len(self.layers), self.B, torch.bfloat16
        ws, wsn = self.ws.data_ptr(), self.ws.numel()
        lib, P = K.lib, K.ptr
        n = 0
        descs = [K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
                 for l in self.layers]
        main = torch.cuda.current_stream()
        side = self.comm_stream
        if self.side_prologue:             # fork BEFORE the input staging: the first prologue runs next to it, not after it
            side.wait_stream(main)
        K.check(lib.lbbnn_bf16_pack(P(self.x), None, K.PACK_SQUARE, B, self.sizes[0][0], P(self.x_bf, bf), P(self.x2_bf, bf),
                                    None, None, st)); n += 1

        def prologue(i, stream, finalize=True):   # mu, rho, lambda -> bf16 M, V (+ fp32 copies for the head's CUDA-core dX) + KL
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            M32 = d["mv32"]
            V32 = d["mv32"][K.lrt_mv_bytes(fi, fo) // 8:] if M32 is not None else None
            if finalize:
                K.check(lib.lbbnn_lrt_bf16_prologue(descs[i], l.cfg.priors, l.cfg.var_mode, P(d["M"], bf), P(d["V"], bf), None, None,
                                                    P(M32, True), P(V32, True), self.stats[1 + i:].data_ptr(), d["klws"].data_ptr(),
                                                    d["klws"].numel(), stream))
            else:                          # KL partials stay in the layer's workspace; kl_finalize(i) closes them later
                K.check(lib.lbbnn_lrt_bf16_prologue_parts(descs[i], l.cfg.priors, l.cfg.var_mode, P(d["M"], bf), P(d["V"], bf),
                                                          P(M32, True), P(V32, True), d["klws"].data_ptr(), d["klws"].numel(),
                                                          stream))

        def kl_finalize(i, stream, out=None):
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            out = self.stats[1 + i:] if out is None else out
            K.check(lib.lbbnn_lrt_kl_finalize(d["klws"].data_ptr(), int(lib.lbbnn_lrt_bf16_prologue_kl_parts(fi, fo)), descs[i],
                                              l.cfg.priors, out.data_ptr(), stream))

        carried = [d["carry"] or d["carry_side"] for d in self.tc]
        for i in range(L):                 # KL of the carried layers: computed at the end of the previous step
            if carried[i]:
                self.stats[1 + i:2 + i].copy_(self.kl_next[i:i + 1]); n += 1
        ready = [None] * L
        kl_done = None
        if self.side_prologue:             # prologues up front on the side stream; each forward GEMM waits for its own M, V
            with torch.cuda.stream(side):  # only; the scalar KL reductions follow once every layer's operands are out
                for i in range(L):
                    if carried[i]:
                        continue
                    prologue(i, K.current_stream(), finalize=False); n += 1
                    ready[i] = torch.cuda.Event()
                    ready[i].record(side)
                for i in range(L):
                    if not carried[i]:
                        kl_finalize(i, K.current_stream()); n += 1
                kl_done = torch.cuda.Event()     # they read the biases: before the first bias update of the backward
                kl_done.record(side)
        a, a2 = self.x_bf, self.x2_bf
        for i in range(L):
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            last = i == L - 1
            if carried[i]:
                pass                        # M, V were written at the end of the previous step (or by refresh_operands)
            elif self.side_prologue:
                main.wait_event(ready[i])
            else:
                prologue(i, st); n += 2
            K.check(lib.lbbnn_tc_lrt_fwd(P(a, bf), P(a2, bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo, P(l.bias_mu.data),
                                         P(l.bias_rho.data), self._noise(i), K.FLAG_SAMPLE | (0 if last else K.FLAG_RELU),
                                         P(d["act"], bf, True), P(d["act2"], bf, True), None, None, P(d["dsf"]),
                                         P(d["act32"], allow_none=True), st)); n += 1
            a, a2 = d["act"], d["act2"]
        dl = self.tc[-1]
        K.check(lib.lbbnn_logsoftmax_nll_f32(P(dl["act32"]), P(self.y, torch.int64), B, self.sizes[-1][1], None,
                                             self.stats.data_ptr(), P(dl["g32"]), 1.0,
                                             P(self.step_dev, torch.int64), ws, wsn, st)); n += 2 if B > 512 else 1
        klg_pre = 1.0 / (self.num_batches * self.world)    # KL added on every rank before a reduction of .grad
        klg_post = 1.0 / self.num_batches                  # KL added once (single GPU, or after the raw-gradient all-reduce)
        if self.fused_update:
            K.check(lib.lbbnn_adam_prepare(P(self.step_dev, torch.int64), self.lr, self.betas[0], self.betas[1],
                                           P(self.adam_coef), st)); n += 1
        if kl_done is not None:
            main.wait_event(kl_done)

        def grads_of(l):
            return K.LayerGrads(*[t.data_ptr() for t in (l.weight_mu.grad, l.weight_rho.grad, l.lambdal.grad,
                                                         l.bias_mu.grad, l.bias_rho.grad)], None)

        def dx(i):
            # ---- dx = dE M + 2 x (dS V) -> the layer below's dE, dS (+ bias partial sums) ----
            l, d, p = self.layers[i], self.tc[i], self.tc[i - 1]
            fi, fo = self.sizes[i]
            if d["head"]:
                M32, V32 = d["mv32"], d["mv32"][K.lrt_mv_bytes(fi, fo) // 8:]
                K.check(lib.lbbnn_tc_lrt_bwd_input_small(P(d["g32"]), P(d["dsf"]), P(M32), P(V32), B, fi, fo, P(p["act"], bf),
                                                         P(p["dsf"]), K.FLAG_SAMPLE | K.FLAG_MASK_DX, P(p["dE"], bf),
                                                         P(p["dS"], bf), None, None, P(p["colsum"]), ws, wsn, st))
                return 2
            K.check(lib.lbbnn_tc_lrt_bwd_input_mn(P(d["dE"], bf), P(d["dS"], bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo,
                                                  P(p["act"], bf), P(p["dsf"]), K.FLAG_SAMPLE | K.FLAG_MASK_DX,
                                                  P(p["dE"], bf), P(p["dS"], bf), P(p["colpart"]), st))
            return 1

        def dw(i, dx_first=False):
            """Layer i's bias sums, dM = dE^T x, dV = dS^T x^2 and the update.  Returns (launches, whether dx(i) was issued)."""
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            n, did_dx = 0, False
            xin, xin2 = (self.x_bf, self.x2_bf) if i == 0 else (self.tc[i - 1]["act"], self.tc[i - 1]["act2"])
            if i == L - 1:                 # fp32 upstream gradient of the loss head: stage dE, dS (+ K-major transposes for a
                # <= 12-output head, whose (batch, out) rows are too short for a TMA pitch) and the bias sums
                K.check(lib.lbbnn_bf16_pack(P(d["g32"]), P(d["dsf"]), K.PACK_SCALE, B, fo, P(d["dE"], bf), P(d["dS"], bf),
                                            P(d["dET"], bf, True), P(d["dST"], bf, True), st)); n += 1
                K.check(lib.lbbnn_colsum2(P(d["g32"]), P(d["dsf"]), 0, B, fo, P(d["colsum"]), ws, wsn, st)); n += 2
            elif d["colpart"] is not None:  # bias sums of this layer: partials written by the dX epilogue of the layer above
                K.check(lib.lbbnn_tc_colsum_reduce(P(d["colpart"]), B, fo, P(d["colsum"]), st)); n += 1
            if d["epi_update"]:            # chain rule + KL + Adam in the GEMM's epilogue; biases in a one-block kernel
                if d["carry"]:
                    if i > 0:              # the epilogue below overwrites M, V with the next step's: their last reader goes first
                        n += dx(i); did_dx = True
                    K.check(lib.lbbnn_tc_lrt_dw_adam_next(P(d["dE"], bf), P(d["dS"], bf), P(xin, bf), P(xin2, bf), descs[i], B,
                                                          l.cfg.priors, l.cfg.var_mode, klg_post, self._adam_state(l),
                                                          P(d["M"], bf), P(d["V"], bf), d["klpart"].data_ptr(), st)); n += 2
                else:
                    K.check(lib.lbbnn_tc_lrt_dw_adam(P(d["dE"], bf), P(d["dS"], bf), P(xin, bf), P(xin2, bf), descs[i], B,
                                                     l.cfg.priors, l.cfg.var_mode, klg_post, self._adam_state(l), st)); n += 1
                K.check(lib.lbbnn_lrt_f32_finalize_adam_bias(descs[i], P(d["colsum"]), l.cfg.priors, K.FLAG_SAMPLE, klg_post,
                                                             self._adam_state(l), st)); n += 1
                if d["carry"]:             # next step's KL of this layer: weight partials + the (updated) bias term
                    K.check(lib.lbbnn_lrt_kl_finalize(d["klpart"].data_ptr(), d["klpart"].numel(), descs[i], l.cfg.priors,
                                                      self.kl_next[i:].data_ptr(), st)); n += 1
                return n, did_dx
            if self.fused_update:
                dM, dV = d["raw"][:fo * fi], d["raw"][fo * fi:2 * fo * fi]
            else:
                dM, dV = self.dM, self.dV

            def gemm(stream):
                if d["head"]:          # A = dE^T, dS^T (out, batch) K-major; B = x, x^2 (batch, in) in place
                    K.check(lib.lbbnn_tc_dual_gemm_raw_ex(P(d["dET"], bf), P(d["dST"], bf), P(xin, bf), P(xin2, bf), fo, fi, B,
                                                          0, 1, P(dM), P(dV), stream))
                else:
                    K.check(lib.lbbnn_tc_dual_gemm_raw_ex(P(d["dE"], bf), P(d["dS"], bf), P(xin, bf), P(xin2, bf), fo, fi, B,
                                                          1, 1, P(dM), P(dV), stream))
            if self.fused_update and side is not None and self.overlap and d["head"] and i > 0:
                # the head's dW GEMM occupies 32 of 148 SMs: on the side stream, under the head's input-gradient kernel
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    gemm(K.current_stream()); n += 1
            else:
                gemm(st); n += 1
            if self.fused_update and self.dp_sharded:
                self._sharded_layer_update(i, descs[i], main); n += 1
            elif self.fused_update:
                self._fused_layer_update(i, descs[i], dM, dV, main); n += 1
            else:
                K.check(lib.lbbnn_lrt_f32_finalize(descs[i], P(dM), P(dV), P(d["colsum"]), l.cfg.priors, l.cfg.var_mode,
                                                   K.FLAG_SAMPLE, None, klg_pre, grads_of(l), st)); n += 1
            return n, did_dx

        for i in reversed(range(L)):
            if self.side_carry0 and i == 1:
                # layer 1's input gradient and layer 0's dW + update first; the freshly updated layer 0's operands and KL for
                # the NEXT step on the side stream, under layer 1's dW GEMM (the step's last)
                n += dx(1)
                n += dw(0)[0]
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    prologue(0, K.current_stream(), finalize=False); n += 1
                    kl_finalize(0, K.current_stream(), out=self.kl_next); n += 1
                n += dw(1)[0]
                break
            k, did_dx = dw(i)
            n += k
            if i > 0 and not did_dx:
                n += dx(i)
        if self.fused_update:
            if side is not None:
                main.wait_stream(side)
        else:
            if self.pg is not None:
                torch.distributed.all_reduce(self.gflat, group=self.pg)
            K.check(lib.lbbnn_adam_f32(P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq), self.n_flat,
                                       self.lr, self.betas[0], self.betas[1], self.eps, P(self.step_dev, torch.int64),
                                       P(self.adam_coef), st)); n += 2
        self.kernels_per_step = n

    def _enqueue(self):
        if self.in_place:
            return self._enqueue_in_place()
        st = K.current_stream()
        L, B, bf = len(self.layers), self.B, torch.bfloat16
        ws, wsn = self.ws.data_ptr(), self.ws.numel()
        lib, P = K.lib, K.ptr
        n = 0
        descs = [K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
                 for l in self.layers]
        # input staging: x, x^2 and their transposes in bf16
        K.check(lib.lbbnn_bf16_pack(P(self.x), None, K.PACK_SQUARE, B, self.sizes[0][0], P(self.x_bf, bf),
                                    P(self.x2_bf, bf), P(self.xT_bf, bf), P(self.x2T_bf, bf), st)); n += 1
        a, a2 = self.x_bf, self.x2_bf
        main = torch.cuda.current_stream()

        def fused_prologue(i, stream):     # mu, rho, lambda -> bf16 M, V (+ transposes) + KL in one pass
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            keep = d["mv32"] is not None
            M32 = d["mv32"] if keep else None
            V32 = d["mv32"][K.lrt_mv_bytes(fi, fo) // 8:] if keep else None
            K.check(lib.lbbnn_lrt_bf16_prologue(descs[i], l.cfg.priors, l.cfg.var_mode, P(d["M"], bf), P(d["V"], bf),
                                                P(d["MT"], bf, True), P(d["VT"], bf, True), P(M32, True), P(V32, True),
                                                self.stats[1 + i:].data_ptr(), d["klws"].data_ptr(), d["klws"].numel(), stream))

        ready = [None] * L
        if self.side_prologue:             # all prologues up front on the side stream; each forward GEMM waits for its own
            self.comm_stream.wait_stream(main)
            with torch.cuda.stream(self.comm_stream):
                for i in range(L):
                    fused_prologue(i, K.current_stream()); n += 2
                    ready[i] = torch.cuda.Event()
                    ready[i].record(self.comm_stream)
        for i in range(L):
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            last = i == L - 1
            if d["mv32"] is not None:      # keep the fp32 M,V of this layer for its SIMT input-gradient GEMM
                M32 = d["mv32"]
                V32 = d["mv32"][K.lrt_mv_bytes(fi, fo) // 8:]
            else:
                M32, V32 = self.M32, self.V32
            if self.side_prologue:
                main.wait_event(ready[i])
            elif self.fused_prologue:
                fused_prologue(i, st); n += 2
            else:
                K.check(lib.lbbnn_lrt_f32_prologue(descs[i], l.cfg.priors, l.cfg.var_mode, K.FLAG_SAMPLE, P(M32), P(V32),
                                                   self.stats[1 + i:].data_ptr(), ws, wsn, st)); n += 2
                K.check(lib.lbbnn_bf16_pack(P(M32), P(V32), K.PACK_PAIR, fo, fi, P(d["M"], bf), P(d["V"], bf),
                                            P(d["MT"], bf, True), P(d["VT"], bf, True), st)); n += 1
            if self.small_head and last and fo <= 12 and fi * fo * 4 <= 192 * 1024:
                K.check(lib.lbbnn_tc_lrt_fwd_small(P(a, bf), P(a2, bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo,
                                                   P(l.bias_mu.data), P(l.bias_rho.data), self._noise(i), K.FLAG_SAMPLE,
                                                   P(d["act32"]), P(d["dsf"]), st)); n += 1
            else:
                K.check(lib.lbbnn_tc_lrt_fwd(P(a, bf), P(a2, bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo, P(l.bias_mu.data),
                                             P(l.bias_rho.data), self._noise(i),
                                             K.FLAG_SAMPLE | (0 if last else K.FLAG_RELU),
                                             P(d["act"], bf, True), P(d["act2"], bf, True), P(d["actT"], bf, True),
                                             P(d["act2T"], bf, True), P(d["dsf"]), P(d["act32"], allow_none=True), st)); n += 1
            a, a2 = d["act"], d["act2"]
        dl = self.tc[-1]
        K.check(lib.lbbnn_logsoftmax_nll_f32(P(dl["act32"]), P(self.y, torch.int64), B, self.sizes[-1][1], None,
                                             self.stats.data_ptr(), P(dl["g32"]), 1.0,
                                             P(self.step_dev, torch.int64), ws, wsn, st)); n += 2 if B > 512 else 1
        klg = 1.0 / (self.num_batches * self.world)

        def grads_of(l):
            return K.LayerGrads(*[t.data_ptr() for t in (l.weight_mu.grad, l.weight_rho.grad, l.lambdal.grad,
                                                         l.bias_mu.grad, l.bias_rho.grad)], None)

        if self.fused_update:
            K.check(lib.lbbnn_adam_prepare(P(self.step_dev, torch.int64), self.lr, self.betas[0], self.betas[1],
                                           P(self.adam_coef), st)); n += 1
        for i in reversed(range(L)):
            l, d = self.layers[i], self.tc[i]
            fi, fo = self.sizes[i]
            if d["g32"] is not None:       # fp32 upstream gradient: stage dE, dS (+ transposes) and the bias sums
                K.check(lib.lbbnn_bf16_pack(P(d["g32"]), P(d["dsf"]), K.PACK_SCALE, B, fo, P(d["dE"], bf), P(d["dS"], bf),
                                            P(d["dET"], bf), P(d["dST"], bf), st)); n += 1
                K.check(lib.lbbnn_colsum2(P(d["g32"]), P(d["dsf"]), 0, B, fo, P(d["colsum"]), ws, wsn, st)); n += 2
            elif not (i + 1 < L and self.small_dx[i + 1]):     # (the fused head kernel already wrote this layer's column sums)
                K.check(lib.lbbnn_colsum2(P(d["dE"], bf), P(d["dS"], bf), 1, B, fo, P(d["colsum"]), ws, wsn, st)); n += 2
            xT, x2T = (self.xT_bf, self.x2T_bf) if i == 0 else (self.tc[i - 1]["actT"], self.tc[i - 1]["act2T"])
            # dM = dE^T x, dV = dS^T x^2: (out, B) x (in, B)^T
            if self.fused_update:
                dM, dV = d["raw"][:fo * fi], d["raw"][fo * fi:2 * fo * fi]
            else:
                dM, dV = self.dM, self.dV
            raw_gemm = lib.lbbnn_tc_dual_gemm_raw_small if (self.small_head and fo <= 12) else lib.lbbnn_tc_dual_gemm_raw
            if self.fused_update and self.comm_stream is not None and self.overlap and i > 0 and self.small_dx[i]:
                # the head's dW GEMM occupies 32 of 148 SMs: on the side stream, under the head's input-gradient kernel
                self.comm_stream.wait_stream(main)
                with torch.cuda.stream(self.comm_stream):
                    K.check(raw_gemm(P(d["dET"], bf), P(d["dST"], bf), P(xT, bf), P(x2T, bf), fo, fi, B, P(dM), P(dV),
                                     K.current_stream())); n += 1
            else:
                K.check(raw_gemm(P(d["dET"], bf), P(d["dST"], bf), P(xT, bf), P(x2T, bf), fo, fi, B, P(dM), P(dV), st)); n += 1
            if self.fused_update:
                self._fused_layer_update(i, descs[i], dM, dV, main); n += 1
            else:
                K.check(lib.lbbnn_lrt_f32_finalize(descs[i], P(dM), P(dV), P(d["colsum"]), l.cfg.priors,
                                                   l.cfg.var_mode, K.FLAG_SAMPLE, None, klg, grads_of(l), st)); n += 1
            if i == 0:
                continue
            p = self.tc[i - 1]
            if self.small_dx[i]:
                M32, V32 = d["mv32"], d["mv32"][K.lrt_mv_bytes(fi, fo) // 8:]
                K.check(lib.lbbnn_tc_lrt_bwd_input_small(P(d["g32"]), P(d["dsf"]), P(M32), P(V32), B, fi, fo, P(p["act"], bf),
                                                         P(p["dsf"]), K.FLAG_SAMPLE | K.FLAG_MASK_DX, P(p["dE"], bf),
                                                         P(p["dS"], bf), P(p["dET"], bf), P(p["dST"], bf), P(p["colsum"]),
                                                         ws, wsn, st)); n += 2
            elif self.simt_dx[i]:
                K.check(lib.lbbnn_lrt_f32_bwd_input(descs[i], P(p["act32"]), B, P(d["g32"]), P(d["dsf"]), l.cfg.priors,
                                                    l.cfg.var_mode, K.FLAG_SAMPLE | K.FLAG_MASK_DX, P(d["mv32"]),
                                                    P(p["g32"]), ws, wsn, st)); n += 2
            else:
                K.check(lib.lbbnn_tc_lrt_bwd_input(P(d["dE"], bf), P(d["dS"], bf), P(d["MT"], bf), P(d["VT"], bf), B, fi,
                                                   fo, P(p["act"], bf), P(p["dsf"]), K.FLAG_SAMPLE | K.FLAG_MASK_DX,
                                                   P(p["dE"], bf), P(p["dS"], bf), P(p["dET"], bf), P(p["dST"], bf),
                                                   st)); n += 1
        if self.fused_update:
            if self.comm_stream is not None:
                main.wait_stream(self.comm_stream)
        else:
            if self.pg is not None:
                torch.distributed.all_reduce(self.gflat, group=self.pg)
            K.check(lib.lbbnn_adam_f32(P(self.flat), P(self.gflat), P(self.exp_avg), P(self.exp_avg_sq), self.n_flat,
                                       self.lr, self.betas[0], self.betas[1], self.eps, P(self.step_dev, torch.int64),
                                       P(self.adam_coef), st)); n += 2
        self.kernels_per_step = n

    def _adam_state(self, l):
        st = K.AdamLayerState()
        for j, name in enumerate(_PARAM_NAMES):
            off = self.param_off[(id(l), name)]
            st.exp_avg[j] = self.exp_avg.data_ptr() + 4 * off
            st.exp_avg_sq[j] = self.exp_avg_sq.data_ptr() + 4 * off
        st.coef = self.adam_coef.data_ptr()
        st.beta1, st.beta2, st.eps = self.betas[0], self.betas[1], self.eps
        return st

    def _fused_layer_update(self, i, desc, dM, dV, main):
        """Layer i's raw gradients are complete on `main`: (all-reduce them and) run chain rule + KL + Adam over them.
        Single GPU: on `main`.  Data parallel: on the communication stream, overlapping the rest of the backward; the KL
        gradient is added once, after the reduction (SURVEY.md §8e)."""
        l, d = self.layers[i], self.tc[i]
        klg = 1.0 / self.num_batches
        if self.comm_stream is None:
            K.check(K.lib.lbbnn_lrt_f32_finalize_adam(desc, K.ptr(dM), K.ptr(dV), K.ptr(d["colsum"]), l.cfg.priors,
                                                      l.cfg.var_mode, K.FLAG_SAMPLE, None, klg, self._adam_state(l),
                                                      K.current_stream()))
            return
        self.comm_stream.wait_stream(main)
        with torch.cuda.stream(self.comm_stream):
            if self.pg is not None:
                torch.distributed.all_reduce(d["raw"], group=self.pg)
            K.check(K.lib.lbbnn_lrt_f32_finalize_adam(desc, K.ptr(dM), K.ptr(dV), K.ptr(d["colsum"]), l.cfg.priors,
                                                      l.cfg.var_mode, K.FLAG_SAMPLE, None, klg, self._adam_state(l),
                                                      K.current_stream()))

    _capture = LRTTrainer._capture
    _retarget_inputs = LRTTrainer._retarget_inputs
    _slot_graph = LRTTrainer._slot_graph
    step_device = LRTTrainer.step_device
    step = LRTTrainer.step
    _stats_dict = LRTTrainer._stats_dict
    step_async = LRTTrainer.step_async
    flush = LRTTrainer.flush
    h2d_bytes_per_step = LRTTrainer.h2d_bytes_per_step
    d2h_bytes_per_step = LRTTrainer.d2h_bytes_per_step


class MultiTensorAdam:
    """torch.optim.Adam(params, lr, betas, eps) (non-amsgrad) as ONE launch over the whole parameter list
    (lbbnn_adam_multi_f32): a device table names every (param, grad, exp_avg, exp_avg_sq, lr, decay) record.  `params` is
    what torch.optim takes: an iterable of tensors (MNF:352) or of parameter-group dicts {"params": ..., "lr": ...,
    "weight_decay": ...} -- the MF script's 33 groups with learning rates from 1e-5 to 0.1 (MF:520-553;
    `lbbnn.mf.reference_param_groups(net)`).  A group without "lr" / "weight_decay" uses the optimizer's.  A non-zero
    weight_decay makes that group's update torch.optim.AdamW's (decoupled: param *= 1 - lr * weight_decay first,
    variational_dropout.py:110); 0 (the default) is torch.optim.Adam exactly.  Gradient addresses are whatever autograd
    produced for this step: eager steps rewrite the table every call; under CUDA-graph capture the addresses (stable in the
    graph's private pool) are recorded and the table is written once after the capture (`finish_capture`)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.weight_decay = float(weight_decay)
        params = list(params)
        groups = params if (params and isinstance(params[0], dict)) else [{"params": params}]
        self.param_groups = []
        self.params, self.lr_scale, self.decay = [], [], []
        seen = set()
        # the launch takes ONE base learning rate (bias correction folded in on the device); groups carry a factor
        lrs = [float(g.get("lr", self.lr)) for g in groups]
        self.base_lr = self.lr if self.lr != 0.0 else (max(lrs) or 1.0)
        for g, glr in zip(groups, lrs):
            ps = g["params"]
            ps = [ps] if torch.is_tensor(ps) else list(ps)
            gwd = float(g.get("weight_decay", self.weight_decay))
            self.param_groups.append({"params": ps, "lr": glr, "weight_decay": gwd})
            for p in ps:
                if id(p) in seen:
                    raise ValueError("some parameters appear in more than one parameter group")
                seen.add(id(p))
                if p.requires_grad:
                    self.params.append(p)
                    self.lr_scale.append(glr / self.base_lr)
                    self.decay.append(glr * gwd)       # the table's decay: lr and weight decay are constant per group
        dev = self.params[0].device
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += _pad4(p.numel())
        self.offs = offs
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=dev)
        self.table = torch.zeros(len(self.params), 7, dtype=torch.int64, device=dev)
        self.coef = torch.zeros(2, dtype=torch.float32, device=dev)
        self.t_dev = torch.zeros(1, dtype=torch.int64, device=dev)      # 1-based index of the update being applied
        self._pending = None
        # early / late split (set_late_params): see there
        self._late_ids, self._early_n = None, 0
        self._early_table = self._early_stream = self._early_pending = None
        self._armed, self._early_seen, self._early_events, self._early_done = False, 0, [], False
        self.dp = None

    def data_parallel(self, process_group):
        """Data-parallel mode: the update applies the SUM over the ranks of `process_group` of every rank's gradients.
        Parameters (re-pointed here, so modules and state_dict() keep working) and the packed gradients live in one arena
        [parameters | packed gradients], each tensor at a 4-float aligned offset, its gradient `n_flat` floats after it;
        the early group (set_late_params, call that first) is laid out before the late one so that each group's gradients
        are one contiguous span.  Each update packs autograd's gradients into the arena (one launch), then
        LBBNN_DP_UPDATE = auto (default) | sharded | nccl:
          sharded  the arena is symmetric memory bound to an NVSwitch multicast object; between two cross-rank barriers each
                   rank reduces (in the switch), updates and multicasts ITS contiguous 1 / world of the table's blocks
                   (lbbnn_adam_multi_dp_f32) and keeps Adam moments for those only -- see owned_range();
          nccl     torch.distributed.all_reduce of the group's packed gradients, then the replicated update.
        auto takes sharded where the fabric has multicast.  Every rank must hold the same parameters (same order)."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        late = self._late_ids or set()
        order = [p for p in self.params if id(p) not in late] + [p for p in self.params if id(p) in late]
        scale = {id(p): (sc, dc) for p, sc, dc in zip(self.params, self.lr_scale, self.decay)}
        self.params, self.lr_scale, self.decay = order, [scale[id(p)][0] for p in order], [scale[id(p)][1] for p in order]
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += _pad4(p.numel())
        self.offs, self.n_flat = offs, total
        dev = self.params[0].device
        mode = os.environ.get("LBBNN_DP_UPDATE", "auto")
        if mode not in ("auto", "sharded", "nccl"):
            raise K.LbbnnError(f"LBBNN_DP_UPDATE={mode!r}: expected auto, sharded or nccl")
        arena = hdl = None
        if mode != "nccl":
            try:
                import torch.distributed._symmetric_memory as symm_mem
                arena = symm_mem.empty(2 * total, dtype=torch.float32, device=dev)
                arena.zero_()
                hdl = symm_mem.rendezvous(arena, process_group.group_name)
                if int(hdl.multicast_ptr) == 0:
                    raise RuntimeError("no multicast support on this fabric")
                hdl.barrier(channel=0)
                torch.cuda.synchronize()
            except Exception as e:  # noqa: BLE001
                if mode == "sharded":
                    raise
                self._dp_error, arena, hdl = repr(e), None, None
        if arena is None:
            arena = torch.zeros(2 * total, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, off in zip(self.params, offs):
                view = arena[off:off + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
        early_n = len(self.params) - len(late)
        spans = [(0, offs[early_n] if early_n < len(offs) else total), (offs[early_n] if early_n < len(offs) else total, total)]
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=dev)
        # pack rows [0, R) and, for the nccl form, the replicated update's rows (gradient = packed copy) [R, 2R)
        self.table = torch.zeros(2 * len(self.params), 7, dtype=torch.int64, device=dev)
        if self._late_ids is not None:
            self._early_table = torch.zeros(2 * early_n, 7, dtype=torch.int64, device=dev)
        self.dp = dict(pg=process_group, world=world, rank=rank, arena=arena, hdl=hdl, spans=spans, early_n=early_n,
                       mode="sharded" if hdl is not None else "nccl",
                       mc=int(hdl.multicast_ptr) if hdl is not None else 0)

    def owned_range(self, p):
        """Element range [lo, hi) of parameter `p` whose Adam moments (and update) THIS rank owns: all of it, except under
        the sharded data-parallel update, where each group's table is split into contiguous runs of blocks (shard_blocks)."""
        n = p.numel()
        if self.dp is None or self.dp["mode"] != "sharded":
            return 0, n
        late = self._late_ids is not None and id(p) in self._late_ids
        group = [q for q in self.params if (self._late_ids is not None and id(q) in self._late_ids) == late]
        first, total = 0, sum((q.numel() + 1023) // 1024 for q in group)
        for q in group:
            if q is p:
                break
            first += (q.numel() + 1023) // 1024
        lo, hi = shard_blocks(total, self.dp["world"], self.dp["rank"])
        lo, hi = max(lo, first) - first, min(hi, first + (n + 1023) // 1024) - first
        return (min(n, 1024 * lo), min(n, 1024 * hi)) if hi > lo else (0, 0)

    def set_late_params(self, late_params):
        """Update everything BUT `late_params` as soon as its gradients are final, in the middle of the backward: every
        other parameter gets a post-accumulate-grad hook that records an event on the stream its gradient was accumulated
        on; when the last of them has fired, the update of that whole group is launched on a private stream that waits for
        exactly those events, and step() only has the late group left.  For the MNF network the late group is the first
        layer's z flow and q0 parameters, whose gradients come out of the LAST node of the backward (a 34 us cluster launch
        at the end of the critical path): the 23 us update of the other 3.3 M parameters runs under it instead of after it.
        The group is the same on every step; a step in which some early parameter gets no gradient falls back to the one
        launch in step().  Contract: zero_grad(set_to_none=True), ONE backward pass, step() -- gradients accumulated over
        several backward passes would be consumed after the first (do not call this for such a loop)."""
        late = {id(p) for p in late_params}
        unknown = late - {id(p) for p in self.params}
        if unknown:
            raise ValueError("late parameters must belong to the optimizer")
        early = [p for p in self.params if id(p) not in late]
        if not early or not late:
            return
        self._late_ids, self._early_n = late, len(early)
        dev = self.params[0].device
        self._early_table = torch.zeros(len(early), 7, dtype=torch.int64, device=dev)
        self._early_stream = torch.cuda.Stream(device=dev)
        for p in early:
            p.register_post_accumulate_grad_hook(self._on_grad)

    def _on_grad(self, p):
        if not self._armed or self._early_done:
            return
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._early_events.append(ev)
        self._early_seen += 1
        if self._early_seen < self._early_n:
            return
        rows, blocks = self._rows(lambda q: id(q) not in self._late_ids)
        if len(rows) != self._early_n:
            return
        for ev in self._early_events:
            self._early_stream.wait_event(ev)
        with torch.cuda.stream(self._early_stream):
            self._launch(rows, blocks, self._early_table, "_early_pending", advance=True, group=0)
        self._early_done = True

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            if set_to_none:
                p.grad = None
            elif p.grad is not None:
                p.grad.zero_()
        # the early group's hooks count from here; gradients that are zeroed in place accumulate in several pieces, so only
        # the set_to_none form (one accumulation per parameter and backward) arms them
        self._armed = self._late_ids is not None and bool(set_to_none)
        self._early_seen, self._early_events, self._early_done = 0, [], False

    def _rows(self, keep=None):
        import struct
        rows, blocks = [], 0
        for p, off, sc, dc in zip(self.params, self.offs, self.lr_scale, self.decay):
            g = p.grad
            if g is None or (keep is not None and not keep(p)):
                continue
            if g.dtype != torch.float32 or not g.is_contiguous() or not p.is_contiguous():
                raise K.LbbnnError("MultiTensorAdam needs contiguous fp32 parameters and gradients")
            n = p.numel()
            lr_bits = struct.unpack("<q", struct.pack("<ff", sc, dc))[0]        # {float lr_scale; float decay}
            rows.append([p.data_ptr(), g.data_ptr(), self.exp_avg.data_ptr() + 4 * off,
                         self.exp_avg_sq.data_ptr() + 4 * off, n, blocks, lr_bits])
            blocks += (n + 1023) // 1024
        return rows, blocks

    def _table_rows(self, rows):
        if self.dp is None:
            return rows
        gdist = 4 * self.n_flat            # the replicated update of the nccl form reads the packed (all-reduced) copy
        return rows + [[r[0], r[0] + gdist] + r[2:] for r in rows]

    def _launch(self, rows, blocks, table, pending_attr, advance, group=None):
        """group (data parallel): 0 = the early group, 1 = the late group, None = every parameter."""
        if torch.cuda.is_current_stream_capturing():
            prev = getattr(self, pending_attr)
            if prev is not None and len(prev) != len(rows):
                raise K.LbbnnError("the set of parameters with gradients changed during capture")
            setattr(self, pending_attr, rows)
        else:
            table[:2 * len(rows) if self.dp is not None else len(rows)].copy_(torch.tensor(self._table_rows(rows), dtype=torch.int64))
        st = K.current_stream()
        if self.dp is not None:
            return self._launch_dp(rows, blocks, table, advance, group, st)
        if advance:                    # t_dev += 1 and the bias corrections of update t in the first of the two launches
            K.check(K.lib.lbbnn_adam_multi_step_f32(table.data_ptr(), len(rows), blocks, self.base_lr, self.betas[0],
                                                    self.betas[1], self.eps, K.ptr(self.t_dev, torch.int64), K.ptr(self.coef), st))
        else:                          # same update index: the early group's launch has advanced it
            K.check(K.lib.lbbnn_adam_multi_f32(table.data_ptr(), len(rows), blocks, self.base_lr, self.betas[0], self.betas[1],
                                               self.eps, K.ptr(self.t_dev, torch.int64), K.ptr(self.coef), st))

    def step(self):
        early_done, self._armed = self._early_done, False
        self._early_done = False
        if early_done:                 # the early group is being updated on its own stream: the late group after it
            torch.cuda.current_stream().wait_stream(self._early_stream)
            rows, blocks = self._rows(lambda q: id(q) in self._late_ids)
        else:
            rows, blocks = self._rows()
        if not rows:
            return
        self._launch(rows, blocks, self.table, "_pending", advance=not early_done, group=1 if early_done else None)

    def _launch_dp(self, rows, blocks, table, advance, group, st):
        D = self.dp
        n_group = {None: len(self.params), 0: D["early_n"], 1: len(self.params) - D["early_n"]}[group]
        if len(rows) != n_group:
            raise K.LbbnnError("data-parallel MultiTensorAdam: every parameter needs a gradient on every step")
        K.check(K.lib.lbbnn_adam_pack_f32(table.data_ptr(), len(rows), blocks, self.n_flat, st))
        tp = K.ptr(self.t_dev, torch.int64)
        if D["mode"] == "sharded":
            # group 0 (early, its own stream) and the late group are in flight at the same time: separate barrier channels.
            # First barrier: every rank has packed; second: every rank's multicast stores have landed (and no rank packs
            # the next step's gradients while a peer still reduces these)
            ch = 1 if group == 0 else 0
            lo, hi = shard_blocks(blocks, D["world"], D["rank"])
            D["hdl"].barrier(channel=ch)
            K.check(K.lib.lbbnn_adam_multi_dp_f32(table.data_ptr(), len(rows), lo, hi, D["arena"].data_ptr(), D["mc"], self.n_flat,
                                                  self.base_lr, self.betas[0], self.betas[1], self.eps, tp, K.ptr(self.coef),
                                                  1 if advance else 0, st))
            D["hdl"].barrier(channel=ch)
            return
        a, b = D["spans"][group] if group is not None else (0, self.n_flat)
        torch.distributed.all_reduce(D["arena"][self.n_flat + a:self.n_flat + b], group=D["pg"])
        upd = table.data_ptr() + table.stride(0) * 8 * len(rows)
        fn = K.lib.lbbnn_adam_multi_step_f32 if advance else K.lib.lbbnn_adam_multi_f32
        K.check(fn(upd, len(rows), blocks, self.base_lr, self.betas[0], self.betas[1], self.eps, tp, K.ptr(self.coef), st))

    def finish_capture(self):
        if self._pending is not None:
            rows = self._table_rows(self._pending)
            self.table[:len(rows)].copy_(torch.tensor(rows, dtype=torch.int64))
            self._pending = None
        if self._early_pending is not None:
            rows = self._table_rows(self._early_pending)
            self._early_table[:len(rows)].copy_(torch.tensor(rows, dtype=torch.int64))
            self._early_pending = None


class GraphedTrainer:
    """Whole training step of ANY of the drop-in networks (LRT, MNF, MF) as one CUDA-graph replay: forward through the
    modules' autograd Functions (liblbbnn kernels), the objective, backward and torch.optim.Adam(capturable=True) are
    captured once; a device step counter keys the native Philox noise so every replay draws fresh noise.

    Reference: the body of `train` for one minibatch -- LBBNN-GP-MF-MNF.py:263-275 (objective="kl": nll_loss(sum) +
    net.kl()/NUM_BATCHES) and LBBNN-GP-MF.py:325-343 (objective="elbo": net.sample_elbo).  The eager modules run the
    same kernels one Python call at a time (~8 ms per MNF step on B200, host-bound); the replay removes the host.  The
    optimizer is MultiTensorAdam by default: one launch instead of torch's ~40 multi_tensor_apply launches per step.

    Data parallel (process_group): each rank runs the captured step on its own `batch_size` rows of the minibatch and the
    optimizer applies the SUM over ranks of the gradients (the nll is a sum over rows, MNF:267-270 / MF:308), so the step
    is the single-GPU step on the concatenated minibatch.  The draws that depend on the parameters only -- MNF's z draw and
    flow masks and its KL branch's draws, MF's masks, sampled weights, bias noise and Gamma precisions -- are ONE draw per
    step for the whole minibatch in the reference, so every rank makes the same draw (same lbbnn / torch seeds, same
    modules built in the same order: checked at construction); the per-row activation noise of the LRT / MNF layers is
    disjoint across ranks (seed + 0x9E3779B97F4A7C15 * rank); the replicated scalar terms (MNF's kl, MF's log q and
    log prior) enter each rank's objective at 1 / world, so their gradient is counted once.  Rank 0's parameters are
    broadcast at construction; MultiTensorAdam.data_parallel does the exchange."""

    def __init__(self, net, batch_size, num_batches, objective="kl", lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                 in_features=None, optimizer=None, param_groups=None, fuse_objective=True, process_group=None):
        """optimizer: None = MultiTensorAdam (one launch for all parameters); "torch" = torch.optim.Adam(capturable=True);
        or any capturable torch optimizer instance over net.parameters().
        param_groups: torch.optim-style parameter groups with their own learning rates (the MF script's 33 groups,
        MF:520-553: `lbbnn.mf.reference_param_groups(net)`), for the first two optimizer choices.
        fuse_objective: objective="kl" through the one-launch loss head (_fused_objective) where the network allows it.
        process_group: data-parallel training over the ranks of this torch.distributed group (see the class docstring);
        needs optimizer=None.  batch_size is the rows of ONE rank."""
        K.require_device()
        self.net, self.B, self.num_batches, self.objective = net, int(batch_size), num_batches, objective
        params = list(net.parameters())
        dev = params[0].device
        if dev.type != "cuda":
            raise K.LbbnnError("GraphedTrainer needs the network on a CUDA device (no CPU fallback)")
        self.device = dev
        self.pg = process_group
        self.world = 1 if process_group is None else torch.distributed.get_world_size(process_group)
        self.rank = 0 if process_group is None else torch.distributed.get_rank(process_group)
        if process_group is not None:
            if optimizer is not None:
                raise K.LbbnnError("data-parallel GraphedTrainer runs the built-in MultiTensorAdam only (optimizer=None)")
            check_replicas(process_group, params, "data-parallel GraphedTrainer")
        in_features = in_features or net.sizes[0]
        self.x = torch.zeros(self.B, in_features, dtype=torch.float32, device=dev)
        self.y = torch.zeros(self.B, dtype=torch.int64, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        if optimizer is None:
            self.opt = MultiTensorAdam(param_groups if param_groups is not None else params, lr=lr, betas=betas, eps=eps)
            if hasattr(net, "late_grad_params") and os.environ.get("LBBNN_ADAM_SPLIT", "1") == "1":
                self.opt.set_late_params(net.late_grad_params())
            if process_group is not None:
                self.opt.data_parallel(process_group)
        elif isinstance(optimizer, str) and optimizer == "torch":
            self.opt = torch.optim.Adam(param_groups if param_groups is not None else params, lr=lr, betas=betas, eps=eps,
                                        capturable=True)
        else:
            self.opt = optimizer
        self.stats = torch.zeros(2, dtype=torch.float32, device=dev)      # [loss, nll]
        self.fuse_objective = bool(fuse_objective)
        self._dlogits = self._kl_grads = None
        self.stats_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        self.x_host = torch.zeros(self.B, in_features, dtype=torch.float32).pin_memory()
        self.y_host = torch.zeros(self.B, dtype=torch.int64).pin_memory()
        net.train()
        self._stream = torch.cuda.Stream(device=dev)
        self._stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._stream), K.graph_noise(self.step_dev), K.row_noise_rank(self.rank):
            for _ in range(3):                      # warm-up: sizes every workspace, creates the Adam state
                self._one_step()
        torch.cuda.current_stream().wait_stream(self._stream)
        torch.cuda.synchronize()
        self.opt.zero_grad(set_to_none=True)        # gradients are re-allocated from the graph's private pool
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self._stream), K.graph_noise(self.step_dev), K.row_noise_rank(self.rank):
            self._one_step()
        if isinstance(self.opt, MultiTensorAdam):
            self.opt.finish_capture()
        self.warmup_steps = 3

    def _fused_objective(self):
        """The objective through ONE launch (lbbnn_nll_kl_objective_f32) where the network exposes its logits and its
        per-layer scalar terms: loss = nll_loss(log_softmax(logits), y, 'sum') + sum_i scale_i term_i into self.stats together
        with d loss / d logits, and the backward started at the logits and the terms with those (constant) gradients -- no
        autograd nodes for log_softmax / nll_loss / the sums / the division (~20 launches of 1-6 us on the critical path).
        objective="kl" (MNF:267-270): terms = the layers' kl at 1 / num_batches.  objective="elbo" (MF:285-319 with
        samples = 1): terms = the layers' log q at + 1 / num_batches and log prior at - 1 / num_batches.
        Returns False when the network does not fit (the torch formulation runs instead)."""
        net = self.net
        if not (self.fuse_objective and hasattr(net, "_logits") and hasattr(net, "layers") and self.B <= 4096):
            return False
        if self.objective == "elbo":
            if not hasattr(net, "_elbo_terms"):
                return False
            logits, terms, signs = net._elbo_terms(self.x)
        else:
            logits = net._logits(self.x, sample=True)
            terms = [l.kl for l in net.layers]
            signs = [1.0] * len(terms)
        if not all(torch.is_tensor(k) and k.numel() == 1 and k.dtype == torch.float32 and k.requires_grad for k in terms) or \
                len(terms) > 16 or logits.dtype != torch.float32 or not logits.is_contiguous():
            raise K.LbbnnError("fused objective: the network's logits / scalar terms are not what the kernel takes")
        if self._dlogits is None or self._dlogits.shape != logits.shape:
            self._dlogits = torch.empty_like(logits)
            # d loss / d term_i; data parallel: the terms are replicated, each rank takes them at 1 / world
            self._kl_grads = [torch.full_like(k, sg / (self.num_batches * self.world)) for k, sg in zip(terms, signs)]
        ptrs = (C_void_p * len(terms))(*[k.data_ptr() for k in terms])
        scales = (C_float * len(terms))(*signs)
        K.check(K.lib.lbbnn_nll_kl_objective_f32(K.ptr(logits), K.ptr(self.y, torch.int64), logits.shape[0], logits.shape[1],
                                                 ptrs, scales, len(terms), 1.0 / (self.num_batches * self.world), K.ptr(self.stats),
                                                 K.ptr(self._dlogits), K.current_stream()))
        torch.autograd.backward([logits] + terms, [self._dlogits] + self._kl_grads)
        return True

    def _one_step(self):
        self.opt.zero_grad(set_to_none=True)
        if self._fused_objective():
            self.opt.step()
        else:
            if self.objective == "elbo":
                out = self.net.sample_elbo(self.x, self.y)
                loss, nll = out[0], out[3]
                if self.world > 1:         # loss = nll + (log q - log prior) / num_batches with the replicated terms at 1 / world
                    loss = nll + (out[2] - out[1]) / (self.net.num_batches * self.world)
            else:
                logp = self.net(self.x, sample=True)
                nll = torch.nn.functional.nll_loss(logp, self.y, reduction="sum")
                loss = nll + self.net.kl() / (self.num_batches * self.world)
            loss.backward()
            self.opt.step()
            self.stats.copy_(torch.stack([loss.detach(), nll.detach()]))
        K.check(K.lib.lbbnn_counter_inc(K.ptr(self.step_dev, torch.int64), K.current_stream()))

    def step_device(self):
        self.graph.replay()

    def step(self, x_host, y_host, read_loss=True):
        """One training step from HOST tensors: H2D, replay, D2H of [loss, nll]."""
        if x_host.is_pinned() and y_host.is_pinned() and x_host.is_contiguous():
            self.x.copy_(x_host.reshape(self.x.shape), non_blocking=True)
            self.y.copy_(y_host, non_blocking=True)
        else:
            self.x_host.copy_(x_host.reshape(self.x_host.shape))
            self.y_host.copy_(y_host)
            self.x.copy_(self.x_host, non_blocking=True)
            self.y.copy_(self.y_host, non_blocking=True)
        self.graph.replay()
        if not read_loss:
            return None
        self.stats_host.copy_(self.stats, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._stats_dict(self.stats_host)

    def _stats_dict(self, st):
        """[loss, nll] of the step.  Data parallel: THIS RANK's contribution (its rows' nll, the replicated terms at
        1 / world); the sum over ranks is the single-GPU value of the concatenated minibatch."""
        return {"loss": float(st[0]), "nll": float(st[1])}

    # the pipelined host-buffer step of the LRT trainers: upload of batch i+1 on a copy stream under step i, the [loss, nll]
    # of step i read at call i+1 (flush() delivers the last)
    step_async = LRTTrainer.step_async
    flush = LRTTrainer.flush
