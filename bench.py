#!/usr/bin/env python3
"""Benchmark of the variational-layer hot path (BASELINE.json metric: train samples/s & MC-predictive samples/s at
1/2/4/8 B200; % TC peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Default (`--workload headline`): the configuration the metric's "% TC peak" is quoted on -- BASELINE.json configs[4], the
widened LRT stack 4096-4096-4096-10 in bf16 at batch 8192 per GPU (tcgen05 / TMEM / TMA kernels; data-parallel over the N
ranks) -- timed for EXACTLY --steps steps, with two sub-records under "also" measured in the same process on the same
GPUs: `lrt_mnist` (configs[1], the reference's own MNIST-shape training step, fp32; data parallel) and `mf_mc_predict`
(configs[3], posterior-predictive averaging over 1024 MC weight samples x 1000 inputs, samples sharded over the N ranks).
One step = forward + loss + backward + Adam on one synthetic minibatch (LBBNN-GP-MF-LRT.py:217-229).
`--workload NAME` runs one workload alone.  `--impl reference` times the REFERENCE's own classes and `train` function
(oracle/_ref, built by oracle/make_ref.py from /root/reference) on the host cores.
Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for how every field is obtained.
`--dump-outputs DIR` (LRT training workloads): after the timed steps, rank 0 writes what the last of them left to the
caller -- the step statistics and the updated parameters -- as DIR/<name>.npy, so that two builds can be compared output
for output on identical inputs (same arguments, same seeds).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "bayesian-neural-nets_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np
import torch

SIZES = {"lrt_mnist": (784, 400, 600, 10), "lrt_wide": (4096, 4096, 4096, 10)}
BATCH = {"lrt_mnist": 100, "lrt_wide": 8192}
DTYPE = {"lrt_mnist": "f32", "lrt_wide": "bf16"}
POOLS = {"lrt_mnist": 512, "lrt_wide": 4}      # lrt_wide: one 134 MB batch already exceeds L2
NUM_BATCHES = 600
POOL = 512          # default number of distinct input batches (lrt_mnist: 512 x 313.6 KB = 160 MB > 126 MB L2)


NCU_SUMMARY = "r02_ncu_summary.json"     # {kernel key: {"dram_bytes_read": .., "dram_bytes_write": .., ...}}, written from this
                                         # round's `ncu --set full` captures by profiles/ncu_summary.py


def ncu_traffic(key):
    """DRAM bytes (read + write) per launch of kernel `key` from THIS round's ncu capture, or None (never a stale file)."""
    try:
        with open(os.path.join(ROOT, "profiles", NCU_SUMMARY)) as fh:
            d = json.load(fh)[key]
        return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"])
    except (OSError, KeyError, ValueError):
        return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# clocks sampler (NVML, polled from a thread during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.002):
        self.samples, self.period, self.stop_flag, self.ok = [], period, False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def start(self):
        if self.ok:
            self.th = threading.Thread(target=self._loop, daemon=True)
            self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.ok:
            self.th.join(timeout=1.0)

    def summary(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvml unavailable: " + self.err}
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        mask = 0
        for _, _, r in inside:
            mask |= r
        reasons = [n for b, n in self.REASONS.items() if mask & b and n != "gpu_idle"]
        return {"sm_mhz": statistics.median([s[1] for s in inside]) if inside else None,
                "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(inside)}


# ------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md §8d C2): x ~ U[0,1) (MNIST ToTensor range), y ~ randint(10)
# ------------------------------------------------------------------------------------------------
def make_pool(pool, batch, in_features, classes, seed):
    rng = np.random.default_rng(seed)
    x = torch.from_numpy(rng.random((pool, batch, in_features), dtype=np.float32))
    y = torch.from_numpy(rng.integers(0, classes, size=(pool, batch))).long()
    return x, y


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed, for output-for-output comparison of two builds
# ------------------------------------------------------------------------------------------------
DUMP_LIMIT = 64 << 20       # bytes written in all
DUMP_SAMPLE = 1 << 20       # entries kept of a larger parameter (the wide stack's 4096 x 4096 weights)


def training_outputs(tr, net):
    """The step statistics [nll, kl_1 .. kl_L] (`stats`) and every updated parameter of the network (`l1.weight_mu`, ...).
    A parameter of more than DUMP_SAMPLE entries is saved as `<name>.sample`: its flattened entries at DUMP_SAMPLE
    positions drawn with a fixed seed, the same positions in every run."""
    out = {"stats": tr.stats.cpu().numpy()}
    for name, p in net.named_parameters():
        flat = p.detach().reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_SAMPLE, replace=False))
            flat, name = flat[torch.from_numpy(pos).to(flat.device)], name + ".sample"
        out[name] = flat.float().cpu().numpy()
    return out


def dump_outputs(directory, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference step, timed on the host cores
# ------------------------------------------------------------------------------------------------
def _ref_modules():
    """oracle/_ref (the reference's own classes + train(), sliced at build time by oracle/make_ref.py) or None."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import make_ref
    return make_ref if make_ref.available() else None


def _ref_lrt_net(m, sizes):
    """The reference's BayesianNetwork (LRT:199-214).  Its layer sizes are hard-coded to 784-400-600-10; the widened stack
    of configs[4] composes the reference's own BayesianLinear exactly as LRT:206-214 does."""
    if tuple(sizes) == (784, 400, 600, 10):
        return m.BayesianNetwork()
    F = torch.nn.functional

    class WideNetwork(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.l1, self.l2, self.l3 = (m.BayesianLinear(i, o) for i, o in zip(sizes[:-1], sizes[1:]))

        def forward(self, x, sample=False):
            x = x.view(-1, sizes[0])
            x = F.relu(self.l1(x, sample))
            x = F.relu(self.l2(x, sample))
            return F.log_softmax(self.l3(x, sample), dim=1)

        def kl(self):
            return self.l1.kl + self.l2.kl + self.l3.kl

    return WideNetwork()


def cpu_reference_steps(workload, steps, warmup, budget_s=20.0):
    """The reference's training step on the host cores: `train(net, optimizer)` of LBBNN-GP-MF-LRT.py:217-229 (unmodified,
    from oracle/_ref) over one injected synthetic minibatch per call; falls back to the oracle port when oracle/_ref is
    absent (kind says which)."""
    sizes, B = SIZES[workload], BATCH[workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    rng = np.random.default_rng(0)
    nb = 8 if B <= 1000 else 1
    x = torch.from_numpy(rng.random((nb, B, sizes[0]), dtype=np.float32))
    y = torch.from_numpy(rng.integers(0, sizes[-1], size=(nb, B))).long()
    R = _ref_modules()
    if R is not None:
        m = R.load("ref_lrt")
        m.NUM_BATCHES = NUM_BATCHES
        torch.manual_seed(0)
        net = _ref_lrt_net(m, sizes)
        opt = m.optim.Adam(net.parameters(), lr=1e-3)          # LRT:358

        def one(i):
            m.train_loader = [(x[i % nb], y[i % nb])]
            return m.train(net, opt)[1]
        kind, what = "reference", "the reference's own BayesianLinear classes and train() (oracle/_ref, sliced from LBBNN-GP-MF-LRT.py)"
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import lbbnn_oracle as O
        layers = [{k: v.clone().requires_grad_(True) for k, v in O.init_lrt_params(rng, i, o).items()}
                  for i, o in zip(sizes[:-1], sizes[1:])]
        opt = torch.optim.Adam([v for p in layers for v in p.values()], lr=1e-3)

        def one(i):
            eps = [torch.randn(B, o) for o in sizes[1:]]            # LRT:174
            opt.zero_grad(set_to_none=True)
            loss, _, _, _ = O.lrt_net_loss(x[i % nb], y[i % nb], layers, eps, NUM_BATCHES)
            loss.backward()
            opt.step()
            return loss
        kind, what = "port", "oracle port (oracle/lbbnn_oracle.py; oracle/_ref absent)"

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        one(i)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": B * done / dt, "unit": "samples/s", "cores": cores, "kind": kind,
            "sample": f"{done} training steps (fwd+loss+bwd+Adam) of {workload} batch {B}: {what}, torch-CPU fp32, "
                      f"{cores} threads",
            "ms_per_step": dt / done * 1e3, "steps": done}


def reference_record(workload, args, steps, warmup, budget_s):
    r = cpu_reference_steps(workload, steps, warmup, budget_s=budget_s)
    return {"impl": "reference", "metric": "train_samples_per_sec", "value": r["value"], "unit": "samples/s",
            "n_gpus": args.gpus, "steps": r["steps"], "warmup": warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(workload, 1),  # the CPU reference computes in fp32, one process
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload != "headline":
        print(json.dumps(reference_record(args.workload, args, args.steps, args.warmup, 120.0)), flush=True)
        return
    # headline: the wide stack for (up to) --steps steps within ~2.5 minutes, then bounded samples of the two sub-records
    line = reference_record("lrt_wide", args, args.steps, min(args.warmup, 1), 150.0)
    line["also"] = {"lrt_mnist": reference_record("lrt_mnist", args, 200, 3, 20.0),
                    "mf_mc_predict": mc_reference_record(args, 20.0, 64)}
    if args.gpus == 1:
        line["also"]["mnf_mnist"] = module_reference_record("mnf_mnist", 1, 15.0, 200)
        line["also"]["mf_mnist"] = module_reference_record("mf_mnist", 1, 15.0, 200)
    print(json.dumps(line), flush=True)


def workload_config(workload, n_gpus):
    sizes, B = SIZES[workload], BATCH[workload]
    POOL = POOLS[workload]
    return {"workload": f"{workload}: LRT MLP {'-'.join(map(str, sizes))}, batch {B} per GPU, "
                        f"fwd+loss+bwd+Adam, NUM_BATCHES={NUM_BATCHES}",
            "batch_per_gpu": B, "global_batch": B * n_gpus,
            "parallelism": "single GPU" if n_gpus == 1 else f"dp{n_gpus} (all-reduce of the raw weight-moment gradients dM, dV + bias sums, then chain rule + Adam)",
            "l2": f"inputs rotate through a pool of {POOL} distinct batches "
                  f"({POOL * B * sizes[0] * 4 / 1e6:.0f} MB > 126 MB L2); parameters are the step's own working set"}


# ------------------------------------------------------------------------------------------------
# per-call timing of the step's C-ABI calls (cold L2), for the roofline of the dominant kernel
# ------------------------------------------------------------------------------------------------
def profile_calls(tr, reps=20):
    """Time every C-ABI call of one training step on its own: CUDA events on the launching stream around
    each call, L2 flushed (a 256 MB memset) before each, `reps` repetitions.  Returns a list of
    {name, us, bytes} with the ALGORITHMIC bytes of DESIGN.md §Kernels."""
    from lbbnn import _capi as K
    B, L = tr.B, len(tr.layers)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=tr.device)
    st = K.current_stream()
    ws, wsn = tr.ws.data_ptr(), tr.ws.numel()
    descs = [K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
             for l in tr.layers]
    calls = []
    for i, l in enumerate(tr.layers):
        K_, N_ = l.in_features, l.out_features
        xin = tr.x if i == 0 else tr.acts[i - 1]
        flags = K.FLAG_SAMPLE | K.FLAG_KL | (K.FLAG_RELU if i < L - 1 else 0)
        calls.append((f"lrt_f32_fwd[l{i + 1}] (prologue+gemm+epilogue)", 12 * K_ * N_ + 4 * B * K_ + 8 * B * N_,
                      lambda i=i, l=l, xin=xin, flags=flags: K.lib.lbbnn_lrt_f32_fwd(
                          descs[i], K.ptr(xin), B, tr._noise(i), l.cfg.priors, l.cfg.var_mode, flags,
                          K.ptr(tr.acts[i]), K.ptr(tr.dsf[i]), tr.stats[1 + i:].data_ptr(),
                          K.ptr(tr.mv[i], allow_none=True), ws, wsn, st)))
        g = l.weight_mu.grad, l.weight_rho.grad, l.lambdal.grad, l.bias_mu.grad, l.bias_rho.grad
        calls.append((f"lrt_f32_bwd_params[l{i + 1}] (gemm+finalize)", 24 * K_ * N_ + 4 * B * K_ + 8 * B * N_,
                      lambda i=i, l=l, xin=xin, g=g: K.lib.lbbnn_lrt_f32_bwd_params(
                          descs[i], K.ptr(xin), B, K.ptr(tr.gbuf[i]), K.ptr(tr.dsf[i]), l.cfg.priors,
                          l.cfg.var_mode, K.FLAG_SAMPLE, None, 1.0 / NUM_BATCHES,
                          K.LayerGrads(*[t.data_ptr() for t in g], None), ws, wsn, st)))
        if i > 0:
            calls.append((f"lrt_f32_bwd_input[l{i + 1}] (gemm+epilogue)", 8 * K_ * N_ + 8 * B * N_ + 8 * B * K_,
                          lambda i=i, l=l, xin=xin: K.lib.lbbnn_lrt_f32_bwd_input(
                              descs[i], K.ptr(xin), B, K.ptr(tr.gbuf[i]), K.ptr(tr.dsf[i]), l.cfg.priors,
                              l.cfg.var_mode, K.FLAG_SAMPLE | K.FLAG_MASK_DX, K.ptr(tr.mv[i]),
                              K.ptr(tr.gbuf[i - 1]), ws, wsn, st)))
    calls.append(("adam_f32 (flat)", 28 * tr.n_flat,
                  lambda: K.lib.lbbnn_adam_f32(K.ptr(tr.flat), K.ptr(tr.gflat), K.ptr(tr.exp_avg),
                                               K.ptr(tr.exp_avg_sq), tr.n_flat, 0.0, 0.9, 0.999, 1e-8,
                                               K.ptr(tr.step_dev, torch.int64), K.ptr(tr.adam_coef), st)))
    out = []
    for name, nbytes, fn in calls:
        times = []
        for _ in range(reps + 2):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            K.check(fn())
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) * 1e3)
        out.append({"name": name, "us": statistics.mean(times[2:]), "bytes": nbytes})
    return out


def profile_fused(tr, sizes, B, us_per_step, peaks, reps=20, replays=True):
    """Roofline of the persistent step kernel (the only kernel of the step).  Algorithmic bytes (DESIGN.md §4): per
    weight 12 B forward read of (mu,rho,lambda) + 12 B re-read in the backward + 12 B of gradient + Adam's 28 B x 3
    tensors (read p,g,m,v, write p,m,v), plus the activations each phase exchanges.  Duration: (a) the average launch
    inside the timed region (= ms_per_step: one launch per step; the input copies are included, so it is an upper
    bound), (b) the same launch alone after a 256 MB L2 flush (cold: the 27 MB of state come from HBM)."""
    from lbbnn import _capi as K  # noqa: F401
    pairs = list(zip(sizes[:-1], sizes[1:]))
    nparam = sum(3 * i * o + 2 * o for i, o in pairs)
    path = sum(36 * i * o + (4 * B * i + 8 * B * o) * 2 + (8 * B * (i + o) if li else 0) for li, (i, o) in enumerate(pairs))
    nbytes = path + 28 * nparam
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=tr.device) if replays else None
    cold = []
    for _ in range(reps + 2 if replays else 0):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tr.step_device()
        e1.record()
        e1.synchronize()
        cold.append(e0.elapsed_time(e1) * 1e3)
    us_cold = statistics.mean(cold[2:]) if replays else None
    us_warm = None
    if replays:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(200):
            tr.step_device()
        e1.record()
        e1.synchronize()
        us_warm = e0.elapsed_time(e1) * 1e3 / 200
    ach = nbytes / (us_per_step * 1e-6) / 1e9
    # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of THIS round's kernel, else null
    traffic = ncu_traffic("lrt_step_kernel")
    roof = {"bound": "hbm", "kernel": "lrt_step_kernel (persistent: fwd + loss + bwd + KL + Adam of the whole stack)",
            "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": traffic,
            "traffic_note": "ncu replays flush the caches, so this is the cold-L2 DRAM traffic of one launch "
                            f"(profiles/{NCU_SUMMARY}); in steady state the 27 MB of state stay in L2",
            "peak_source": peaks["source"], "us_per_launch": us_per_step, "bytes_per_launch": nbytes,
            "us_per_launch_back_to_back": us_warm, "us_per_launch_cold_l2": us_cold,
            "timing": "average launch over the timed region (CUDA events, one launch per step, inputs rotate through a "
                      "pool > L2); back_to_back = 200 replays on resident inputs; cold = alone after a 256 MB L2 flush",
            "note": "the 27 MB of parameters + Adam state are L2-resident between steps; the kernel is bound by phase "
                    "latency (grid barriers + fp32 FFMA tiles), not by HBM"}
    flops = sum(4.0 * B * i * o * (3 if li else 2) for li, (i, o) in enumerate(pairs))
    step_roof = {"bytes_per_step": nbytes, "hbm_floor_us": nbytes / peaks["hbm_gbs"] / 1e3,
                 "frac_of_hbm_floor": (nbytes / peaks["hbm_gbs"] / 1e3) / us_per_step,
                 "flops_per_step": flops, "fp32_tflops": flops / (us_per_step * 1e-6) / 1e12,
                 "schedule": tr.schedule}
    kern = [{"name": "lrt_step_kernel", "us": round(us_per_step, 2), "us_back_to_back": us_warm and round(us_warm, 2),
             "us_cold_l2": us_cold and round(us_cold, 2), "bytes": nbytes, "gbps": round(ach, 1)}]
    return roof, step_roof, kern


def profile_calls_wide(tr, reps=5):
    """Tensor-core GEMM calls of one wide step timed on their own (CUDA events, operands > L2): FLOPs are the
    ALGORITHMIC 2 GEMMs x 2 B in out per call (DESIGN.md §Kernels).  Layer 2 of the stack (4096 x 4096, batch 8192)."""
    from lbbnn import _capi as K
    bf, st, B = torch.bfloat16, K.current_stream(), tr.B
    P = K.ptr
    out = []
    i = 1 if len(tr.layers) > 2 else 0
    l, d = tr.layers[i], tr.tc[i]
    fi, fo = tr.sizes[i]
    a, a2 = (tr.x_bf, tr.x2_bf) if i == 0 else (tr.tc[i - 1]["act"], tr.tc[i - 1]["act2"])
    desc = K.make_layer(l.weight_mu.data, l.weight_rho.data, l.lambdal.data, l.bias_mu.data, l.bias_rho.data)
    if tr.in_place:
        calls = [(f"tc_lrt_fwd[l{i + 1}] (tcgen05 dual GEMM + eps/sqrt/relu epilogue)", lambda: K.lib.lbbnn_tc_lrt_fwd(
            P(a, bf), P(a2, bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo, P(l.bias_mu.data), P(l.bias_rho.data), tr._noise(i),
            K.FLAG_SAMPLE | K.FLAG_RELU, P(d["act"], bf), P(d["act2"], bf), None, None, P(d["dsf"]), None, st))]
        if d["epi_update"]:
            calls.append((f"tc_lrt_dw_adam[l{i + 1}] (dM, dV from operands in place + chain rule + KL + Adam epilogue)",
                          lambda: K.lib.lbbnn_tc_lrt_dw_adam(P(d["dE"], bf), P(d["dS"], bf), P(a, bf), P(a2, bf), desc, B,
                                                             l.cfg.priors, l.cfg.var_mode, 1.0 / NUM_BATCHES, tr._adam_state(l), st)))
        else:
            dM, dV = d["raw"][:fo * fi], d["raw"][fo * fi:2 * fo * fi]
            calls.append((f"tc_dual_gemm_raw_ex[l{i + 1}] (dM, dV from operands in place)", lambda: K.lib.lbbnn_tc_dual_gemm_raw_ex(
                P(d["dE"], bf), P(d["dS"], bf), P(a, bf), P(a2, bf), fo, fi, B, 1, 1, P(dM), P(dV), st)))
        if i > 0:
            p = tr.tc[i - 1]
            calls.append((f"tc_lrt_bwd_input_mn[l{i + 1}] (dx + relu mask + next dE/dS + bias partial sums epilogue)",
                          lambda: K.lib.lbbnn_tc_lrt_bwd_input_mn(
                              P(d["dE"], bf), P(d["dS"], bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo, P(p["act"], bf), P(p["dsf"]),
                              K.FLAG_SAMPLE | K.FLAG_MASK_DX, P(p["dE"], bf), P(p["dS"], bf), P(p["colpart"], True), st)))
    else:
        xT, x2T = (tr.xT_bf, tr.x2T_bf) if i == 0 else (tr.tc[i - 1]["actT"], tr.tc[i - 1]["act2T"])
        dM, dV = (d["raw"][:fo * fi], d["raw"][fo * fi:2 * fo * fi]) if tr.fused_update else (tr.dM, tr.dV)
        calls = [(f"tc_lrt_fwd[l{i + 1}] (tcgen05 dual GEMM + eps/sqrt/relu epilogue)", lambda: K.lib.lbbnn_tc_lrt_fwd(
            P(a, bf), P(a2, bf), P(d["M"], bf), P(d["V"], bf), B, fi, fo, P(l.bias_mu.data), P(l.bias_rho.data), tr._noise(i),
            K.FLAG_SAMPLE | K.FLAG_RELU, P(d["act"], bf), P(d["act2"], bf), P(d["actT"], bf), P(d["act2T"], bf), P(d["dsf"]),
            P(d["act32"], allow_none=True), st)),
            (f"tc_dual_gemm_raw[l{i + 1}] (dM, dV)", lambda: K.lib.lbbnn_tc_dual_gemm_raw(
                P(d["dET"], bf), P(d["dST"], bf), P(xT, bf), P(x2T, bf), fo, fi, B, P(dM), P(dV), st))]
        if i > 0:
            p = tr.tc[i - 1]
            calls.append((f"tc_lrt_bwd_input[l{i + 1}] (dx + relu mask + next dE/dS epilogue)", lambda: K.lib.lbbnn_tc_lrt_bwd_input(
                P(d["dE"], bf), P(d["dS"], bf), P(d["MT"], bf), P(d["VT"], bf), B, fi, fo, P(p["act"], bf), P(p["dsf"]),
                K.FLAG_SAMPLE | K.FLAG_MASK_DX, P(p["dE"], bf), P(p["dS"], bf), P(p["dET"], bf), P(p["dST"], bf), st)))
    flops = 2 * 2.0 * B * fi * fo
    for name, fn in calls:
        for _ in range(2):
            K.check(fn())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            K.check(fn())
        e1.record()
        e1.synchronize()
        out.append({"name": name, "key": name.split(" ")[0], "us": e0.elapsed_time(e1) / reps * 1e3, "flops": flops})
    return out


# ------------------------------------------------------------------------------------------------
def _mark(msg):
    if os.environ.get("LBBNN_BENCH_VERBOSE"):
        print(f"[bench rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


class Ctx:
    """Process-wide state of one bench run: rank / device / process group, created once for all workloads of the run."""

    def __init__(self, args):
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.pg = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.pg = dist.group.WORLD

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def shutdown(self):
        """Leave the process group cleanly: every captured graph that holds NCCL / symmetric-memory kernels has been
        dropped by its workload, the device is idle, all ranks are here.  destroy_process_group() is given 30 s (it was
        seen to block on one box while graphs were still alive); a watchdog then ends the process, the JSON line being
        already flushed."""
        if self.world == 1:
            return
        import gc
        gc.collect()
        torch.cuda.synchronize()
        torch.distributed.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        t = threading.Timer(30.0, lambda: os._exit(0))
        t.daemon = True
        t.start()
        torch.distributed.destroy_process_group()
        t.cancel()


def bench_lrt(ctx, workload, steps, warmup, unfused=False, cpu_budget_s=15.0, dump_dir=None):
    """One LRT training workload (lrt_mnist / lrt_wide) on this run's GPUs; returns the record on rank 0, None elsewhere.
    dump_dir: rank 0 writes training_outputs() of the last timed step there."""
    import lbbnn
    if os.environ.get("LBBNN_HANG_DUMP"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["LBBNN_HANG_DUMP"]), exit=True)
    rank, local_rank, world, dev, pg = ctx.rank, ctx.local_rank, ctx.world, ctx.dev, ctx.pg
    args = argparse.Namespace(steps=steps, warmup=warmup, unfused=unfused)

    sizes, B, POOL = SIZES[workload], BATCH[workload], POOLS[workload]
    wide = workload == "lrt_wide"
    torch.manual_seed(0)                       # identical initial parameters on every rank
    lbbnn.manual_seed(1234)
    net = lbbnn.BayesianNetwork(sizes).to(dev)
    _mark("process group up, building trainer")
    if wide:
        tr = lbbnn.LRTTensorCoreTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-3, process_group=pg,
                                        fused_update=not args.unfused,
                                        in_place=False if os.environ.get("LBBNN_WIDE_R01") else None,
                                        carry_operands=os.environ.get("LBBNN_WIDE_CARRY", "0") == "1")
    else:   # the fused persistent step kernel unless --unfused; gradients stay in registers (no .grad written)
        tr = lbbnn.LRTTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-3, process_group=pg,
                              fused=not args.unfused, materialize_grads=args.unfused)
    _mark("trainer captured")

    pool_x_host, pool_y_host = make_pool(POOL, B, sizes[0], sizes[-1], seed=1000 + rank)
    pool_x_host, pool_y_host = pool_x_host.pin_memory(), pool_y_host.pin_memory()
    pool_x, pool_y = pool_x_host.to(dev), pool_y_host.to(dev)

    barrier = ctx.barrier

    # ---- device-resident throughput ("value") ---------------------------------------------------------
    def dev_step(i):
        tr.x.copy_(pool_x[i % POOL], non_blocking=True)
        tr.y.copy_(pool_y[i % POOL], non_blocking=True)
        tr.step_device()

    for i in range(args.warmup):
        dev_step(i)
    _mark("warmup done")
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        dev_step(args.warmup + i)
    e1.record()
    barrier()
    t1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    _mark(f"timed region done: {ms / args.steps * 1e3:.1f} us/step")
    if dump_dir and rank == 0:      # now: the end-to-end steps below go on training the same network
        dump_outputs(dump_dir, training_outputs(tr, net))

    # ---- end to end through the public API with host buffers ("e2e") ----------------------------------
    # trainer.step_async(x_host, y_host): every step uploads its batch from pinned host memory (H2D) and its
    # [nll, kl_1..kl_L] are read back on the host (D2H); the read of step i is returned by call i+1, so the host
    # never idles the GPU.  The timed region ends after flush() has delivered the last step's statistics.
    for i in range(min(args.warmup, 5)):
        tr.step(pool_x_host[i % POOL], pool_y_host[i % POOL])
    for i in range(3):                                   # warm the pipelined path too (its device slots, copy stream)
        tr.step_async(pool_x_host[i % POOL], pool_y_host[i % POOL])
    tr.flush()
    barrier()
    te0 = time.perf_counter()
    n_read = 0
    for i in range(args.steps):
        out = tr.step_async(pool_x_host[(i + 7) % POOL], pool_y_host[(i + 7) % POOL])
        n_read += out is not None
    out = tr.flush()
    n_read += 1
    barrier()
    te1 = time.perf_counter()
    assert n_read == args.steps + 1     # every timed step's statistics + the re-read of the last warm-up step
    e2e_ms = (te1 - te0) * 1e3
    # the fully synchronous form (upload, step, read back, host sync every step), for reference
    ts0 = time.perf_counter()
    for i in range(min(args.steps, 200)):
        tr.step(pool_x_host[(i + 3) % POOL], pool_y_host[(i + 3) % POOL])
    torch.cuda.synchronize()
    e2e_sync_us = (time.perf_counter() - ts0) / min(args.steps, 200) * 1e6
    _mark("e2e done")
    sampler.stop()
    clocks = sampler.summary(t0, te1)

    if world > 1:
        tms = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(tms, op=torch.distributed.ReduceOp.MAX)
        ms, e2e_ms = tms.tolist()
    assert out["loss"] == out["loss"], "loss is NaN"

    if rank == 0:
        peaks = load_peaks()
        if wide:
            prof = profile_calls_wide(tr)
            top = max(prof, key=lambda r: r["us"])
            ach = top["flops"] / (top["us"] * 1e-6) / 1e12
            step_flops = sum(2 * 2.0 * B * i * o * (3 if li > 0 else 2) for li, (i, o) in enumerate(zip(sizes[:-1], sizes[1:])))
            traffic = ncu_traffic(top["key"])
            traffic_note = (f"dram__bytes_read + dram__bytes_write of this round's ncu --set full capture of this call "
                            f"(profiles/{NCU_SUMMARY})") if traffic is not None else None
            roof = {"bound": "tensor", "kernel": top["name"], "achieved": ach, "peak": peaks["bf16_tflops"],
                    "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"], "traffic": traffic, "traffic_note": traffic_note,
                    "peak_source": peaks["source"], "us_per_launch": top["us"], "flops_per_launch": top["flops"],
                    "timing": "kernel alone, operands larger than L2, CUDA events, mean of 5; burst peak"}
            step_roof = {"flops_per_step": step_flops, "achieved_tflops": step_flops / (ms / args.steps * 1e-3) / 1e12,
                         "frac_of_sustained_peak": step_flops / (ms / args.steps * 1e-3) / 1e12 / (peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"])}
            kern = [{"name": r["name"], "us": round(r["us"], 1), "tflops": round(r["flops"] / r["us"] / 1e6, 1)} for r in prof]
        elif tr.fused:
            # extra replays are collective under data parallelism (NCCL all-reduce inside the step): single GPU only
            roof, step_roof, kern = profile_fused(tr, sizes, B, ms / args.steps * 1e3, peaks, replays=(world == 1))
        else:
            prof = profile_calls(tr)
            top = max(prof, key=lambda r: r["us"])
            achieved = top["bytes"] / (top["us"] * 1e-6) / 1e9
            step_bytes = sum(r["bytes"] for r in prof)
            roof = {"bound": "hbm", "kernel": top["name"], "achieved": achieved, "peak": peaks["hbm_gbs"],
                    "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": None,
                    "peak_source": peaks["source"], "us_per_launch": top["us"], "bytes_per_launch": top["bytes"],
                    "timing": "cold L2 (256 MB memset before each launch), CUDA events, mean of 20"}
            step_roof = {"bytes_per_step": step_bytes, "hbm_floor_us": step_bytes / peaks["hbm_gbs"] / 1e3,
                         "sum_of_calls_us_cold": sum(r["us"] for r in prof),
                         "frac_of_hbm_floor": (step_bytes / peaks["hbm_gbs"] / 1e3) / (ms / args.steps * 1e3)}
            kern = [{"name": r["name"], "us": round(r["us"], 2), "bytes": r["bytes"],
                     "gbps": round(r["bytes"] / r["us"] / 1e3, 1)} for r in prof]
        cpu = None
        if world == 1 and cpu_budget_s > 0:
            cpu = cpu_reference_steps(workload, steps=2 if wide else 60, warmup=1 if wide else 3, budget_s=cpu_budget_s)
        line = {
            "metric": "train_samples_per_sec", "value": B * world * args.steps / (ms * 1e-3), "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[workload], "data": "synthetic",
            "config": workload_config(workload, world),
            "e2e": {"value": B * world * args.steps / (e2e_ms * 1e-3), "unit": "samples/s",
                    "h2d_bytes_per_step": tr.h2d_bytes_per_step, "d2h_bytes_per_step": tr.d2h_bytes_per_step,
                    "ms_per_step": e2e_ms / args.steps, "api": "LRTTrainer.step_async (pipelined: stats of step i read at call i+1)",
                    "sync_api_us_per_step": e2e_sync_us},
            "gpu_launches": tr.kernels_per_step * args.steps, "allreduce": getattr(tr, "allreduce", None),
            "kernels_per_step": tr.kernels_per_step,
            "roofline": roof, "step_roofline": step_roof, "kernels": kern,
            "clocks": clocks, "timed_region_s": ms * 1e-3,
            "last_loss": out["loss"],
        }
        if cpu is not None:
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    else:
        line = None
    # captured NCCL / symmetric-memory work must be gone before the process group is torn down
    tr.graph = None
    del tr, pool_x, pool_y, pool_x_host, pool_y_host
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------------------------------------------
# MC posterior-predictive workload (BASELINE.json configs[3]): MF net, S = 1024 weight samples over a
# 1000-input test batch, samples sharded across the GPUs, one all-reduce of the accumulators.
# ------------------------------------------------------------------------------------------------
MC_SAMPLES, MC_BATCH, MC_SIZES = 1024, 1000, (784, 400, 600, 10)


def _mc_net_params(rng):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lbbnn_oracle as O
    layers = [O.init_mf_params(rng, i, o) for i, o in zip(MC_SIZES[:-1], MC_SIZES[1:])]
    for p in layers:   # trained-like inclusion probabilities spanning (0,1) (SURVEY.md §8d C4)
        p["lambdal"] = torch.from_numpy(rng.normal(0.0, 2.0, size=tuple(p["lambdal"].shape)).astype(np.float32))
    return layers, O


def cpu_reference_mc(budget_s=15.0, max_samples=64):
    """The per-sample body of the reference's test_ensemble loop (LBBNN-GP-MF.py:367-406) with the reference's own MF
    classes (oracle/_ref): refresh alpha, draw the statistics masks, the stochastic forward with fresh masks, the density
    masks, and the host-side row-normalised expit accumulation; gamma.exact = True as the driver sets it (MF:612-627).
    Falls back to the oracle port when oracle/_ref is absent."""
    rng = np.random.default_rng(0)
    layers, O = _mc_net_params(rng)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    x = torch.from_numpy(rng.random((MC_BATCH, MC_SIZES[0]), dtype=np.float32))
    R = _ref_modules()
    if R is not None:
        from scipy.special import expit
        m = R.load("ref_mf")
        m.BATCH_SIZE = MC_BATCH
        net = m.BayesianNetwork()
        with torch.no_grad():
            for l, p in zip((net.l1, net.l2, net.l3), layers):
                for k, v in p.items():
                    getattr(l, k).copy_(v)
        net.eval()
        ls = (net.l1, net.l2, net.l3)
        for l in ls:
            l.gamma.exact = True
        state = {"means": None, "sum": torch.zeros(MC_BATCH, MC_SIZES[-1]), "spars": 0.0, "dens": 0.0}
        ntot = float(sum(i * o for i, o in zip(MC_SIZES[:-1], MC_SIZES[1:])))

        def one():
            for l in ls:                                                             # MF:369-374
                l.alpha = 1 / (1 + torch.exp(-l.lambdal))
                l.gamma.alpha = l.alpha
            g = [l.gamma.rsample() for l in ls]                                      # MF:377-379
            state["spars"] += sum(torch.sum(t > 0.5).cpu().detach().numpy() for t in g) / ntot   # MF:382-385
            out = net.forward(x, sample=True, medimean=False, g1=net.l1.gamma.rsample(), g2=net.l2.gamma.rsample(),
                              g3=net.l3.gamma.rsample())                             # MF:389-390
            g = [l.gamma.rsample() for l in ls]                                      # MF:391-393
            state["dens"] += torch.cat([t.flatten() for t in g]).mean().item()       # MF:394-395
            tmp = expit(out.detach().cpu().numpy())                                  # MF:398-406
            for j in range(MC_BATCH):
                tmp[j] /= np.sum(tmp[j])
            state["means"] = tmp if state["means"] is None else state["means"] + tmp
            state["sum"] += out
        kind, what = "reference", "the reference's own MF classes (oracle/_ref, sliced from LBBNN-GP-MF.py), loop body MF:367-406"
    else:
        acc = torch.zeros(MC_BATCH, MC_SIZES[-1])

        def one():
            h = x
            for i, p in enumerate(layers):
                alpha = O.alpha_of(p["lambdal"])
                g = torch.bernoulli(alpha)                                        # gamma.exact = True (MF:113)
                nz = {"eps_w": torch.randn_like(alpha), "eps_b": torch.randn(alpha.shape[0])}
                h, _, _ = O.mf_forward(h, p, g, nz, calc_log_probs=False)
                h = torch.relu(h) if i < len(layers) - 1 else torch.log_softmax(h, 1)
            acc.add_(h)
        kind, what = "port", "oracle port (oracle/_ref absent)"
    done, t0 = 0, None
    with torch.no_grad():
        one()                                                                      # warm-up
        t0 = time.perf_counter()
        while done < max_samples and (done < 2 or time.perf_counter() - t0 < budget_s):
            one()
            done += 1
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "MC weight-samples/s", "cores": cores, "kind": kind, "steps": done,
            "ms_per_step": dt / done * 1e3,
            "sample": f"{done} MC weight samples (masks+weights+bias sampled, forward over {MC_BATCH} inputs, accumulate) "
                      f"of the MF 784-400-600-10 net: {what}, torch-CPU fp32, {cores} threads"}


def mc_reference_record(args, budget_s, max_samples):
    r = cpu_reference_mc(budget_s=budget_s, max_samples=max_samples)
    return {"impl": "reference", "metric": "mc_predictive_samples_per_sec", "value": r["value"],
            "unit": r["unit"], "n_gpus": args.gpus, "steps": r["steps"], "warmup": 1,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": mc_config(1),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def _mc_traffic():
    return ncu_traffic("tc_linear_tf32x3_pair[l1]")


def mc_config(world):
    return {"workload": f"mf_mc_predict: MF MLP 784-400-600-10 posterior-predictive averaging, {MC_SAMPLES} MC weight samples "
                        f"x {MC_BATCH}-input batch per step, gamma.exact=True",
            "mc_samples": MC_SAMPLES, "test_batch": MC_BATCH,
            "parallelism": "single GPU" if world == 1 else f"MC samples sharded over {world} GPUs, one fp64 all-reduce per batch",
            "l2": "each step re-samples all 559,600 weights 1024 times from Philox; inputs rotate through 8 test batches; "
                  "the 6.7 MB of parameters are the step's own working set"}


def run_mc(args):
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(mc_reference_record(args, 60.0, max(8, args.steps))), flush=True)
        return
    ctx = Ctx(args)
    line = bench_mc(ctx, args, args.steps, args.warmup)
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)
    ctx.shutdown()


def bench_mc(ctx, args, steps, warmup, cpu_budget_s=15.0):
    """configs[3] on this run's GPUs; a step = 1024 MC weight samples over one 1000-input test batch, samples sharded over
    the ranks, one fp64 all-reduce of the accumulators.  Returns the record on rank 0, None elsewhere."""
    import lbbnn
    rank, local_rank, world, dev, pg = ctx.rank, ctx.local_rank, ctx.world, ctx.dev, ctx.pg
    args = argparse.Namespace(steps=steps, warmup=warmup, mc_batch=args.mc_batch, mc_gemm=args.mc_gemm, mc_lanes=args.mc_lanes)
    rng = np.random.default_rng(0)
    layers, _ = _mc_net_params(rng)
    net = lbbnn.mf.BayesianNetwork(MC_SIZES).to(dev)
    with torch.no_grad():
        for l, p in zip(net.layers, layers):
            for k, v in p.items():
                getattr(l, k).copy_(v)
    mc = lbbnn.mf.MCPredictor(net, batch=MC_BATCH, seed=4321, process_group=pg, samples_per_launch=args.mc_batch,
                              gemm=args.mc_gemm, lanes=args.mc_lanes)
    first, count = lbbnn.mf.shard_samples(MC_SAMPLES, world, rank)
    xs_host = torch.from_numpy(rng.random((8, MC_BATCH, MC_SIZES[0]), dtype=np.float32)).pin_memory()
    xs = xs_host.to(dev)
    pred_host = torch.zeros(MC_BATCH, dtype=torch.int64).pin_memory()

    barrier = ctx.barrier

    def step(i, host):
        mc.run((xs_host if host else xs)[i % 8], count, first_sample=first)
        res = mc.result(MC_SAMPLES)
        if host:
            pred_host.copy_(res["pred"], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return res

    for i in range(args.warmup):
        step(i, False)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        step(i, False)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    te0 = time.perf_counter()
    for i in range(args.steps):
        step(i, True)
    barrier()
    te1 = time.perf_counter()
    e2e_ms = (te1 - te0) * 1e3
    sampler.stop()
    clocks = sampler.summary(t0, te1)
    if world > 1:
        tms = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(tms, op=torch.distributed.ReduceOp.MAX)
        ms, e2e_ms = tms.tolist()
    if rank == 0:
        from lbbnn import _capi as K
        peaks = load_peaks()
        # kernels of the layer-1 stage timed alone (CUDA events, cold L2): the batched sampler (ALU-bound Philox; HBM
        # side: 12 B read per weight + 4 or 8 B written per weight and sample) and the layer's GEMM over SB samples
        l = net.layers[0]
        SB = mc.SB
        tc = mc.n_tc >= 2
        desc = mc._desc(0)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        times = {"s": [], "g": []}
        st = K.current_stream()
        stride = mc.NSTREAMS * len(net.layers)
        lane = mc.lanes[0]
        if tc:
            sample = lambda: K.lib.lbbnn_mc_sample_split(desc, SB, K.ptr(lane.counter, torch.int64), 4321, 0, stride, 1,
                                                         K.ptr(lane.w[0]), K.ptr(lane.w_lo[0]), K.ptr(lane.b[0]), st)
            gemm = lambda: K.lib.lbbnn_tc_linear_tf32x3(K.ptr(mc.x_hi), K.ptr(mc.x_lo), 784, 0, K.ptr(lane.w[0]),
                                                        K.ptr(lane.w_lo[0]), K.ptr(lane.b[0]), 1, MC_BATCH, SB * 400, 784,
                                                        K.FLAG_RELU, None, K.ptr(lane.h_hi[0]), K.ptr(lane.h_lo[0]), SB * 400,
                                                        400, st)
            gname = f"tc_linear_tf32x3[l1] (3xTF32 on tcgen05, fp32 accuracy, {SB} weight samples per launch)"
        else:
            sample = lambda: K.lib.lbbnn_mc_sample_split(desc, SB, K.ptr(lane.counter, torch.int64), 4321, 0, stride, 1,
                                                         K.ptr(lane.w[0]), None, K.ptr(lane.b[0]), st)
            gemm = lambda: K.lib.lbbnn_linear_f32_batched(K.ptr(mc.x), 0, K.ptr(lane.w[0]), K.ptr(lane.b[0]), SB, MC_BATCH,
                                                          784, 400, K.FLAG_RELU, K.ptr(lane.h[0]), st)
            gname = f"sgemm_tn_batched[l1] (fp32 SIMT, {SB} weight samples per launch)"
        for _ in range(8):
            for name, fn in (("s", sample), ("g", gemm)):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); K.check(fn()); b.record(); b.synchronize()
                times[name].append(a.elapsed_time(b) * 1e3)
        us_s = statistics.mean(times["s"][2:])
        us_g = statistics.mean(times["g"][2:])
        nbytes = (12 + (8 if tc else 4) * SB) * 784 * 400   # parameters read once (L2 serves the other samples) + SB x w written
        gflop = 2.0 * MC_BATCH * 784 * 400 * SB / 1e9        # ALGORITHMIC flops: one fp32 product per (input, weight)
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12   # nominal CUDA-core FFMA peak, TFLOP/s
        cpu = cpu_reference_mc(budget_s=cpu_budget_s) if (world == 1 and cpu_budget_s > 0) else None
        ach = gflop * 1e9 / (us_g * 1e-6) / 1e12     # TFLOP/s
        launches_per_step = sum((count // SB) // len(mc.lanes) + (1 if j < (count // SB) % len(mc.lanes) else 0)
                                for j in range(len(mc.lanes))) + (1 if count % SB else 0)
        note = ("fp32 parity mode (1e-5 vs the oracle, argmax bit-exact): every fp32 product is three kind::tf32 MMAs "
                "(hi*hi + hi*lo + lo*hi) at half the bf16 rate, so 1/6 of the bf16 tensor peak is the ceiling of this "
                "algorithmic-flops fraction; `mma_tflops` counts the MMAs actually issued") if tc else (
                "fp32 parity mode keeps this GEMM on the CUDA cores; the fraction of the bf16 tensor peak is quoted because "
                "the contract asks for it")
        line = {"metric": "mc_predictive_samples_per_sec", "value": MC_SAMPLES * args.steps / (ms * 1e-3),
                "unit": "MC weight-samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": dict(mc_config(world), samples_per_launch=SB, lanes=len(mc.lanes),
                               gemm="3xTF32 tcgen05 (layers 1-2) + fp32 SIMT (10-wide head)" if tc else "fp32 SIMT"),
                "e2e": {"value": MC_SAMPLES * args.steps / (e2e_ms * 1e-3), "unit": "MC weight-samples/s",
                        "h2d_bytes_per_step": MC_BATCH * MC_SIZES[0] * 4, "d2h_bytes_per_step": MC_BATCH * 8,
                        "ms_per_step": e2e_ms / args.steps},
                "gpu_launches": int((mc.kernels_per_launch * launches_per_step + 4) * args.steps),
                "kernels_per_sample": mc.kernels_per_sample,
                "input_samples_per_sec": MC_SAMPLES * MC_BATCH * args.steps / (ms * 1e-3),
                "roofline": {"bound": "tensor", "kernel": gname,
                             "achieved": ach, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"],
                             "traffic": _mc_traffic() if tc else None, "peak_source": peaks["source"], "us_per_launch": us_g,
                             "flops_per_launch": gflop * 1e9,
                             "timing": "kernel alone, cold L2 (256 MB memset before each launch), CUDA events, mean of 6",
                             "note": note},
                "sampling_roofline": {"bound": "hbm", "kernel": f"mc_sample[l1] (mask + weights + bias, {SB} samples per launch)",
                                      "achieved": nbytes / (us_s * 1e-6) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                      "frac": nbytes / (us_s * 1e-6) / 1e9 / peaks["hbm_gbs"], "us_per_launch": us_s,
                                      "bytes_per_launch": nbytes},
                "timed_region_s": ms * 1e-3,
                "kernels": [{"name": "mc_sample[l1]", "us": round(us_s, 2)},
                            {"name": gname.split(" ")[0], "us": round(us_g, 2), "tflops": round(ach, 2)}],
                "clocks": clocks}
        if tc:
            line["roofline"]["mma_tflops"] = 3 * ach
            line["roofline"]["frac_of_3xtf32_ceiling"] = ach / (peaks["bf16_tflops"] / 6)
        else:
            line["roofline"]["frac_of_fp32_cuda_core_peak"] = ach / fp32_peak
            line["roofline"]["fp32_cuda_core_peak_tflops"] = fp32_peak
        if cpu is not None:
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    else:
        line = None
    mc.graph = None
    del mc
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------------------------------------------
# MNF / MF training steps through the drop-in modules (BASELINE.json configs[2] and the MF train loop, MF:325-343):
# the reference's own `train` body -- forward (flows / weight sampling), objective, backward, optim.Adam.step -- with
# the modules of this repo; every kernel of the layers is liblbbnn's, the glue (autograd tape, Adam) is torch's.
# ------------------------------------------------------------------------------------------------
def _module_oracle_step(kind):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lbbnn_oracle as O
    import cases as C
    rng = np.random.default_rng(0)
    sizes = list(zip(MC_SIZES[:-1], MC_SIZES[1:]))
    B = 100
    x = torch.from_numpy(rng.random((B, 784), dtype=np.float32))
    y = torch.from_numpy(rng.integers(0, 10, size=(B,))).long()
    if kind == "vd_mnist":
        x = (x - 0.1307) / 0.3081                      # the script normalises MNIST (variational_dropout.py:38-40)
        layers = [{k: v.clone().requires_grad_(k == "theta") for k, v in O.init_vd_params(rng, n, m).items()} for n, m in C.VD_SIZES]
        opt = torch.optim.AdamW([p["theta"] for p in layers], lr=1e-4)

        def one():
            zetas = [torch.randn(B, m) for _, m in C.VD_SIZES]
            opt.zero_grad(set_to_none=True)
            loss = O.vd_net_loss(x, y, layers, zetas, NUM_BATCHES)[0]
            loss.backward()
            opt.step()
    elif kind == "mnf_mnist":
        named = [{k: v.clone().requires_grad_(True) for k, v in C.flat_named(O.init_mnf_params(rng, i, o)).items()} for i, o in sizes]
        tmpl = [O.init_mnf_params(np.random.default_rng(1), i, o) for i, o in sizes]
        layers = [C.unflatten_like(t_, n) for t_, n in zip(tmpl, named)]
        opt = torch.optim.Adam([v for n in named for v in n.values()], lr=1e-3)

        def one():
            noises = [C.mnf_noise(rng, B, i, o) for i, o in sizes]
            opt.zero_grad(set_to_none=True)
            loss, _, _, _ = O.mnf_net_loss(x, y, layers, noises, NUM_BATCHES)
            loss.backward()
            opt.step()
    else:
        layers = [{k: v.clone().requires_grad_(True) for k, v in O.init_mf_params(rng, i, o).items()} for i, o in sizes]
        opt = torch.optim.Adam([v for p in layers for v in p.values()], lr=1e-3)

        def one():
            noises = [{"eps_w": torch.randn(o, i), "eps_b": torch.randn(o), "g0_w": torch._standard_gamma(torch.full((1,), 1.05)),
                       "g0_b": torch._standard_gamma(torch.full((o,), 1.05))} for i, o in sizes]
            us = [torch.rand(o, i) for i, o in sizes]
            opt.zero_grad(set_to_none=True)
            loss = O.mf_net_elbo(x, y, layers, noises, us, NUM_BATCHES)[0]
            loss.backward()
            opt.step()
    return one, B


# the 33 Adam parameter groups of LBBNN-GP-MF.py:520-553 (name -> learning rate), for the reference's own network
_MF_REF_LRS = (("bias_mu", 1e-4), ("bias_rho", 1e-4), ("weight_mu", 1e-4), ("weight_rho", 1e-4), ("pa", 1e-3), ("pb", 1e-3),
               ("weight_a", 1e-5), ("weight_b", 1e-5), ("bias_a", 1e-5), ("bias_b", 1e-5), ("lambdal", 0.1))


def _module_reference_step(kind):
    """One minibatch of the reference's own `train()` (oracle/_ref: LBBNN-GP-MF-MNF.py:263-275 over its BayesianNetwork with
    optim.Adam(net.parameters(), lr=1e-4), MNF:416; LBBNN-GP-MF.py:325-343 with the script's 33 parameter groups, MF:520-553)
    or None when oracle/_ref does not hold that script."""
    R = _ref_modules()
    if R is None or kind not in ("mnf_mnist", "mf_mnist"):
        return None
    try:
        m = R.load("ref_mnf" if kind == "mnf_mnist" else "ref_mf")
    except Exception:
        return None
    m.NUM_BATCHES = NUM_BATCHES
    rng = np.random.default_rng(0)
    B = 100
    x = torch.from_numpy(rng.random((8, B, 784), dtype=np.float32))
    y = torch.from_numpy(rng.integers(0, 10, size=(8, B))).long()
    torch.manual_seed(0)
    net = m.BayesianNetwork()
    if kind == "mnf_mnist":
        opt = m.optim.Adam(net.parameters(), lr=1e-4)
        step = lambda: m.train(net, opt)                                    # noqa: E731
    else:
        opt = m.optim.Adam([{"params": getattr(l, name), "lr": lr} for name, lr in _MF_REF_LRS for l in (net.l1, net.l2, net.l3)],
                           lr=1e-4)
        step = lambda: m.train(net, opt, 0, 0)                              # noqa: E731
    state = {"i": 0}

    def one():
        m.train_loader = [(x[state["i"] % 8], y[state["i"] % 8])]
        state["i"] += 1
        step()
    return one, B


def cpu_reference_module(kind, budget_s=15.0, max_steps=60):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = _module_reference_step(kind)
    if ref is not None:
        one, B = ref
        who, what = "reference", ("the reference's own classes and train() (oracle/_ref, sliced from "
                                  + ("LBBNN-GP-MF-MNF.py" if kind == "mnf_mnist" else "LBBNN-GP-MF.py, 33 Adam groups") + ")")
    else:
        one, B = _module_oracle_step(kind)
        who, what = "port", "oracle port"
    one()
    done, t0 = 0, time.perf_counter()
    while done < max_steps and (done < 2 or time.perf_counter() - t0 < budget_s):
        one()
        done += 1
    dt = time.perf_counter() - t0
    return {"value": B * done / dt, "unit": "samples/s", "cores": cores, "kind": who, "steps": done,
            "ms_per_step": dt / done * 1e3,
            "sample": f"{done} training steps (fwd+objective+bwd+Adam) of {kind} batch {B}: {what}, torch-CPU fp32, {cores} threads"}


def module_config(kind):
    if kind == "vd_mnist":
        return {"workload": "vd_mnist: variational-dropout MLP 784-1200-1200-1200-10 (variational_dropout.py), batch 100, "
                            "fwd+loss_fn+bwd+AdamW(lr 1e-4), theta trained / alpha fixed at 0.2 as in the reference",
                "batch_per_gpu": 100, "parallelism": "single GPU",
                "l2": "inputs rotate through a pool of 512 distinct batches (161 MB > 126 MB L2)"}
    what = ("MNF MLP 784-400-600-10 (2 RNVP transforms, h=75x4, z flow + auxiliary r flow KL)" if kind == "mnf_mnist"
            else "MF MLP 784-400-600-10 (relaxed-Bernoulli gamma, full weight sampling, GaussGamma/BetaBinomial log-probs)")
    return {"workload": f"{kind}: {what}, batch 100, fwd+objective+bwd+Adam through the drop-in modules (eager autograd)",
            "batch_per_gpu": 100, "parallelism": "single GPU",
            "l2": "inputs rotate through a pool of 512 distinct batches (161 MB > 126 MB L2)"}


def module_reference_record(kind, n_gpus, budget_s, max_steps):
    r = cpu_reference_module(kind, budget_s=budget_s, max_steps=max_steps)
    return {"impl": "reference", "metric": "train_samples_per_sec", "value": r["value"], "unit": r["unit"],
            "n_gpus": n_gpus, "steps": r["steps"], "warmup": 1, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": module_config(kind),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def run_module(args):
    kind = args.workload
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        print(json.dumps(module_reference_record(kind, args.gpus, 60.0, max(8, args.steps))), flush=True)
        return
    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit(f"{kind} is a single-GPU workload (replicas only)")
    print(json.dumps(bench_module(kind, args.steps, args.warmup, eager=args.eager)), flush=True)


def bench_module(kind, steps, warmup, eager=False, cpu_budget_s=15.0):
    """One module-level training workload (mnf_mnist / mf_mnist / vd_mnist) on cuda:<current device>; returns the record."""
    import lbbnn
    args = argparse.Namespace(steps=steps, warmup=warmup, eager=eager)
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    lbbnn.manual_seed(99)
    B, POOL = 100, 512
    net = (lbbnn.vd.BNN() if kind == "vd_mnist" else
           lbbnn.mnf.BayesianNetwork() if kind == "mnf_mnist" else lbbnn.mf.BayesianNetwork()).to(dev)
    net.train()
    px_h, py_h = make_pool(POOL, B, 784, 10, seed=1000)
    if kind == "vd_mnist":
        px_h = (px_h - 0.1307) / 0.3081
    px_h, py_h = px_h.pin_memory(), py_h.pin_memory()
    px, py = px_h.to(dev), py_h.to(dev)
    tr = None
    if args.eager:
        opt = (torch.optim.AdamW(net.parameters(), lr=1e-4) if kind == "vd_mnist" else
               torch.optim.Adam(lbbnn.mf.reference_param_groups(net), lr=1e-4) if kind == "mf_mnist" else
               torch.optim.Adam(net.parameters(), lr=1e-3))

        def dev_step(x, y):
            opt.zero_grad(set_to_none=True)
            if kind == "vd_mnist":
                loss = lbbnn.vd.loss_fn(net(x), y, net, NUM_BATCHES)
            elif kind == "mnf_mnist":
                logp = net(x, sample=True)
                loss = torch.nn.functional.nll_loss(logp, y, reduction="sum") + net.kl() / NUM_BATCHES
            else:
                loss = net.sample_elbo(x, y)[0]
            loss.backward()
            opt.step()
            return loss

        def host_step(xh, yh):
            return dev_step(xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True)).item()
    else:   # the whole step (modules' autograd Functions + objective + backward + Adam) as one CUDA-graph replay
        if kind == "vd_mnist":      # C-ABI calls on preallocated buffers (no autograd), captured once
            tr = lbbnn.vd.VDTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-4)
        else:
            if kind == "mf_mnist":   # the reference's own optimizer: 33 parameter groups, lr 1e-5 .. 0.1 (MF:520-553)
                tr = lbbnn.GraphedTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-4, objective="elbo",
                                          param_groups=lbbnn.mf.reference_param_groups(net))
            else:
                tr = lbbnn.GraphedTrainer(net, batch_size=B, num_batches=NUM_BATCHES, lr=1e-3, objective="kl")

        def dev_step(x, y):
            tr.x.copy_(x, non_blocking=True)
            tr.y.copy_(y, non_blocking=True)
            tr.step_device()

        if hasattr(tr, "step_async"):          # pipelined: upload of batch i+1 under step i, statistics read one call late
            last = {}

            def host_step(xh, yh):
                out = tr.step_async(xh, yh)
                if out is not None:
                    last.update(out)
                return last.get("loss")
        else:
            def host_step(xh, yh):
                return tr.step(xh, yh)["loss"]

    for i in range(args.warmup):
        dev_step(px[i % POOL], py[i % POOL])
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        dev_step(px[(args.warmup + i) % POOL], py[(args.warmup + i) % POOL])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    te0 = time.perf_counter()
    for i in range(args.steps):
        lv = host_step(px_h[(i + 7) % POOL], py_h[(i + 7) % POOL])
    if tr is not None and hasattr(tr, "flush"):
        lv = tr.flush()["loss"]               # the last step's statistics (inside the timed region)
    torch.cuda.synchronize()
    te1 = time.perf_counter()
    sampler.stop()
    cpu = cpu_reference_module(kind, budget_s=cpu_budget_s) if cpu_budget_s > 0 else None
    peaks = load_peaks()
    nparam = sum(p.numel() for p in net.parameters())
    # algorithmic bytes of a step: every parameter read in forward and backward, gradient written, Adam 28 B/param
    nbytes = nparam * (4 + 4 + 4 + 28)
    us = ms / args.steps * 1e3
    line = {"metric": "train_samples_per_sec", "value": B * args.steps / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": module_config(kind),
            "e2e": {"value": B * args.steps / (te1 - te0), "unit": "samples/s", "h2d_bytes_per_step": B * 784 * 4 + B * 8,
                    "d2h_bytes_per_step": 8 if (tr is not None and hasattr(tr, "step_async")) else 4,
                    "ms_per_step": (te1 - te0) / args.steps * 1e3,
                    "api": ("GraphedTrainer.step_async (pipelined: [loss, nll] of step i read at call i+1)"
                            if (tr is not None and hasattr(tr, "step_async")) else "step(x_host, y_host)")},
            "gpu_launches": (tr.kernels_per_step * args.steps if kind == "vd_mnist" and tr is not None else None),
            "mode": "eager" if args.eager else "cuda-graph replay of the whole step",
            "roofline": {"bound": "hbm", "kernel": "whole step (all kernels of one replay)", "achieved": nbytes / (us * 1e-6) / 1e9,
                         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": nbytes / (us * 1e-6) / 1e9 / peaks["hbm_gbs"],
                         "traffic": None, "peak_source": peaks["source"], "bytes_per_launch": nbytes, "us_per_launch": us,
                         "note": "a step is ~10^2 small launches (flow GEMVs, prologue/finalize, Adam): latency-bound, reported "
                                 "against HBM because the contract asks for one bound"},
            "clocks": sampler.summary(t0, te1), "last_loss": lv, "n_parameters": nparam}
    if cpu is not None:
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if tr is not None:
        tr.graph = None
    del tr, net, px, py
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return line


def run_headline(args):
    """lrt_wide for exactly --steps steps, plus bounded runs of lrt_mnist and mf_mc_predict on the same GPUs (`also`)."""
    ctx = Ctx(args)
    line = bench_lrt(ctx, "lrt_wide", args.steps, args.warmup, unfused=args.unfused, dump_dir=args.dump_outputs)
    small = bench_lrt(ctx, "lrt_mnist", 2000, 50)
    mc = bench_mc(ctx, args, 8, 3)
    also = {"lrt_mnist": small, "mf_mc_predict": mc}
    if ctx.world == 1:     # the module-level training loops of the other two scripts (single-GPU workloads: replicas only)
        also["mnf_mnist"] = bench_module("mnf_mnist", 500, 20, cpu_budget_s=10.0)
        also["mf_mnist"] = bench_module("mf_mnist", 300, 20, cpu_budget_s=10.0)
    if ctx.rank == 0:
        line["also"] = also
        print(json.dumps(line), flush=True)
    ctx.shutdown()


def run_ours(args):
    ctx = Ctx(args)
    line = bench_lrt(ctx, args.workload, args.steps, args.warmup, unfused=args.unfused, dump_dir=args.dump_outputs)
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)
    ctx.shutdown()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mc-batch", type=int, default=32, help="mf_mc_predict: weight samples per launch")
    ap.add_argument("--mc-gemm", default="auto", choices=("auto", "simt", "tc"),
                    help="mf_mc_predict: GEMMs on the tensor cores as 3xTF32 (auto / tc) or on the CUDA cores (simt)")
    ap.add_argument("--mc-lanes", type=int, default=None, help="mf_mc_predict: concurrent launch sequences per GPU")
    ap.add_argument("--eager", action="store_true", help="mnf_mnist / mf_mnist: eager modules instead of the graphed step")
    ap.add_argument("--unfused", action="store_true", help="lrt_*: per-layer launch sequence / separate update passes")
    ap.add_argument("--workload", default="headline",
                    choices=["headline"] + sorted(SIZES) + ["mf_mc_predict", "mnf_mnist", "mf_mnist", "vd_mnist"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="headline / lrt_*: write the statistics and updated parameters of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ["headline"] + sorted(SIZES)):
        ap.error("--dump-outputs covers the LRT training workloads (headline, lrt_mnist, lrt_wide) of --impl ours")
    big = args.workload in ("headline", "lrt_wide")
    if args.steps is None:
        args.steps = 100 if big else (20 if args.workload == "mf_mc_predict" else 2000)
    if args.warmup is None:
        args.warmup = 5 if big or args.workload == "mf_mc_predict" else 50
    if args.workload == "mf_mc_predict":
        run_mc(args)
    elif args.workload in ("mnf_mnist", "mf_mnist", "vd_mnist"):
        run_module(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.workload == "headline":
        run_headline(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
