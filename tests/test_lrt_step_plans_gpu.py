"""The one-launch LRT training step (csrc/lrt_step.cu, lrt_step_kernel: forward, loss, backward, chain rule, KL and Adam) in
every kind of schedule its host planner can pick, against the float64 oracle (lbbnn_oracle.lrt_forward / lrt_kl, per-layer
var_mode and priors) driving torch.optim.Adam in float64:
  - forward split-K sums of 1, 8 (sum_splits2 without a tail), 9 (a tail of one) and the auto plan's 20-28 partials, in the
    hidden-layer epilogue and in the tiled head's loss_epilogue;
  - thread groups per CTA (TileCfg.G, the contraction split inside a CTA) of 1 (batch 128, bn 64) and 8 (bn 8, batch 16);
  - ragged shapes: K % 4 != 0 (unvectorised loaders), N % 4 != 0 (st4_clip's scalar stores), in*out % 4 != 0
    (update_quad<false, ..>), N < 8, edge tiles in every phase; batch 1, 7 and 128;
  - more work items than CTAs in a forward and in a backward phase (a second item whose weight tiles were not staged);
  - dX straight through the relu mask (xsplits 1) and through the Xe phase (xsplits > 1) on the same layer;
  - the small head (last_fwd_loss / last_bwd) at 10 and 32 classes, the tiled head at 33 classes and forced by
    LBBNN_STEP_GENERIC_HEAD with 8 and 9 splits; one layer with either head, and eight layers;
  - var_mode "exact" (moments4's exact branch, update_quad<.., REF=false, ..>) and different non-default priors per layer;
  - injected and native (Philox) noise;
and, on whole launches: phases 1 then 2 bit-identical to phases 3, bit-identical repeats, LBBNN_STEP_OVERLAP_UPDATE, the plan
cache following the overrides, and the limits.
Plans are forced through LBBNN_STEP_PLAN_L<i> = "bn,fsplits,rn,ck,bk,xsplits" (0 = free), and every run asserts from the
trainer's schedule string that the forced plan and head ran.  Item counts in the comments are for 148 SMs (296 CTAs).
Tolerances as test_trainer_step_matches_oracle_plus_torch_adam: nll and KL (total and per layer) 1e-5 relative; every
gradient 1e-5 (max|a-b|/max|b|); parameters and both Adam moments 2e-6 after each of 3 steps.  Each step restarts the fp64
side from the kernel's fp32 parameters, and Adam is driven with the kernel's own gradients."""
import ctypes
import re
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import cases as C
import lbbnn_oracle as O

TOL = 1e-5
PTOL = 2e-6
NAMES = ["weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho"]
SEED = 4242
PLAN_RE = re.compile(r"l(\d+)\((\d+)->(\d+)\) F bn=(\d+) kc=(\d+) items=(\d+)x(\d+) \| W (\d+)x(\d+) items=(\d+) \| "
                     r"X bk=(\d+) nc=(\d+) items=(\d+)x(\d+); ")
HEAD_RE = re.compile(r"head=(small|tiled) smem=\d+$")
# layer l of a configuration with priors gets PRIORS[(l + 1) % 3]: neighbouring layers differ, layer 0 is not the default
PRIORS = [dict(mu_prior=0.0, sigma_prior=1.0, alpha_prior=0.05, bias_mu_prior=0.0, bias_sigma_prior=1.0),
          dict(mu_prior=0.1, sigma_prior=0.5, alpha_prior=0.25, bias_mu_prior=-0.1, bias_sigma_prior=2.0),
          dict(mu_prior=-0.05, sigma_prior=1.3, alpha_prior=0.6, bias_mu_prior=0.2, bias_sigma_prior=0.7)]


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


@dataclass
class Cfg:
    id: str
    sizes: tuple
    batch: int
    plan: dict = field(default_factory=dict)     # layer -> "bn,fsplits,rn,ck,bk,xsplits"
    generic_head: bool = False
    exact: tuple = ()                             # layers with var_mode "exact"
    priors: bool = False
    native: bool = False
    seed: int = 0        # of the case: parameters, inputs, labels, injected noise

    @property
    def head(self):
        return "tiled" if self.generic_head or self.sizes[-1] > 32 else "small"

    def env(self):
        e = {f"LBBNN_STEP_PLAN_L{l}": v for l, v in self.plan.items()}
        if self.generic_head:
            e["LBBNN_STEP_GENERIC_HEAD"] = "1"
        return e


MNIST = (784, 400, 600, 10)
CONFIGS = [
    # auto plan at the MNIST shape: 28 / 20 forward splits summed by the hidden epilogue, dX of l1 through Xe (25 splits),
    # small head; exact variance on l0 and l2, reference on l1; per-layer priors; native noise
    Cfg("mnist-auto", MNIST, 100, exact=(0, 2), priors=True, native=True),
    # the same network with the tiled head: 8 splits (sum_splits2 with an empty tail) walked by loss_epilogue, dX of the head
    # straight through l1's relu mask (75x1 items)
    Cfg("mnist-tiled-head-8-splits", MNIST, 100, {2: "8,8,0,0,0,0"}, generic_head=True, seed=2),
    # ... 9 splits: a tail of one partial
    Cfg("mnist-tiled-head-9-splits", MNIST, 100, {2: "8,9,0,0,0,0"}, generic_head=True, exact=(1,), seed=3),
    # 9 splits summed by the hidden-layer epilogue (tail of one), G = 3; small head
    Cfg("hidden-9-splits", (100, 600, 10), 32, {0: "64,9,0,0,0,0"}, priors=True),
    # 8 splits in the hidden epilogue, 9 in the tiled head, the head's dX in 3 splits (Xe into l0)
    Cfg("hidden-8-splits-head-xe", (120, 600, 10), 32, {0: "64,8,0,0,0,0", 1: "8,9,0,0,0,3"}, generic_head=True,
        native=True),
    # forward of l0: bn 8 -> 300 tiles x 1 split > 296 CTAs (four CTAs run a second, unstaged item); G = 8; batch 16
    Cfg("fwd-items-exceed-grid", (64, 2400, 10), 16, {0: "8,0,0,0,0,0"}, seed=1),
    # batch 128: l0 forward bn 64 -> G = 1; l1 backward 256 dW + 128 dX (xsplits 4) items > 296 CTAs
    Cfg("bwd-items-exceed-grid-b128", (96, 256, 128, 10), 128, {0: "64,0,0,0,0,0", 1: "0,0,8,16,8,4"}, exact=(0, 1, 2),
        seed=3),
    # the same layer (256 -> 64 at batch 128) with dX in 4 splits through Xe, and straight through the relu mask
    Cfg("dx-xe-4-splits", (96, 256, 64, 10), 128, {1: "0,0,8,16,8,4"}),
    Cfg("dx-direct", (96, 256, 64, 10), 128, {1: "0,0,8,16,8,1"}, priors=True),
    # ragged, every layer tiled: K 37 / 23 / 6, N 23 / 6 / 3 (N % 4 != 0, N < 8), in*out 851 / 138 / 18 (update_quad<false>);
    # edge tiles in F (16 of 23, 2 splits of 23), W (8 x 16 of 23 x 37 and 6 x 23) and X (16 of 23, 2 splits of 6)
    Cfg("ragged-tiled", (37, 23, 6, 3), 7, {0: "16,3,8,16,0,0", 1: "8,2,8,16,16,2", 2: "0,0,0,0,8,1"}, generic_head=True,
        exact=(1,), priors=True),
    # ragged, batch 1, small head of 5 classes
    Cfg("ragged-b1", (37, 23, 5), 1, exact=(0, 1)),
    # the small head at its limit (32 classes) and the tiled head one class past it
    Cfg("head-32-small", (128, 72, 32), 100),
    Cfg("head-33-tiled", (128, 72, 33), 100, priors=True),
    # one layer: the small head alone (no generic phase, Lg == 0) and the tiled head alone
    Cfg("one-layer-small-head", (20, 3), 7, native=True),
    Cfg("one-layer-tiled-head", (64, 40), 1, exact=(0,)),
    # eight layers (the maximum), ragged widths
    Cfg("eight-layers", (48, 40, 36, 33, 32, 24, 17, 12, 10), 7, exact=(1, 4, 7), priors=True),
]


def _grid():
    """CTAs of the step kernel's grid: 2 per SM (148 SMs on a B200; the library assumes 148 without a GPU)."""
    return 2 * (torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148)


def _parse(schedule):
    layers = []
    for m in PLAN_RE.finditer(schedule):
        l, K_, N, bn, kc, ft, fs, rn, ck, nw, bk, nc, xt, xs = map(int, m.groups())
        layers.append(dict(K=K_, N=N, bn=bn, kc=kc, f_items=ft * fs, fsplits=fs, rn=rn, ck=ck, w_items=nw, bk=bk,
                           x_items=xt * xs, xsplits=xs))
    head = HEAD_RE.search(schedule)
    assert head and len(layers) >= 1, schedule
    return layers, head.group(1)


def _assert_plan(schedule, cfg):
    """The schedule string shows every forced value and the head kind the configuration asks for."""
    layers, head = _parse(schedule)
    assert [(y["K"], y["N"]) for y in layers] == list(zip(cfg.sizes[:-1], cfg.sizes[1:])), schedule
    assert head == cfg.head, schedule
    for l, spec in cfg.plan.items():
        for name, v in zip(("bn", "fsplits", "rn", "ck", "bk", "xsplits"), map(int, spec.split(","))):
            assert v == 0 or layers[l][name] == v, (cfg.id, l, name, schedule)
    return layers, head


def _describe(K, sizes, batch):
    """lbbnn_lrt_step_describe of a stack (host code: works without a GPU)."""
    st = K.Step()
    st.n_layers, st.batch = len(sizes) - 1, batch
    off = 0
    for i, (k, n) in enumerate(zip(sizes[:-1], sizes[1:])):
        sl = st.layer[i]
        sl.in_features, sl.out_features = k, n
        nk, n4 = (k * n + 3) // 4 * 4, (n + 3) // 4 * 4
        sl.off_weight_mu, sl.off_weight_rho, sl.off_lambdal = off, off + nk, off + 2 * nk
        sl.off_bias_mu, sl.off_bias_rho = off + 3 * nk, off + 3 * nk + n4
        off += 3 * nk + 2 * n4
        sl.priors, sl.var_mode = K.Priors(0, 1, 0.05, 0, 1), 0
    buf = ctypes.create_string_buffer(4096)
    if K.lib.lbbnn_lrt_step_describe(st, buf, 4096) != 0:
        raise K.LbbnnError(K.lib.lbbnn_last_error().decode())
    return buf.value.decode()


def _fwd_groups(B, bn, N, kc, nt=256):
    """Host copy of make_cfg(B, min(bn, N), kc, NT).G in csrc/lrt_step.cu: thread groups that split a forward item's
    contraction inside the CTA."""
    RP, CP = (B + 3) & ~3, (min(bn, N) + 7) & ~7
    g = max(1, min(nt // ((RP >> 2) * (CP >> 3)), 8, kc))
    kpg = ((kc + g - 1) // g + 3) & ~3
    return (kc + kpg - 1) // kpg


def _set_env(monkeypatch, env):
    for k in ("LBBNN_STEP_GENERIC_HEAD", "LBBNN_STEP_OVERLAP_UPDATE") + tuple(f"LBBNN_STEP_PLAN_L{l}" for l in range(8)):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def test_configurations_reach_their_paths(monkeypatch):
    """Host-only: the planner gives every configuration above its forced plan, and together they reach every path the module
    docstring lists (so a change of the cost model cannot quietly move them off it)."""
    from lbbnn import _capi as K
    G = _grid()
    seen = {}
    for cfg in CONFIGS:
        _set_env(monkeypatch, cfg.env())
        layers, head = _assert_plan(_describe(K, cfg.sizes, cfg.batch), cfg)
        L = len(layers)
        generic = layers if head == "tiled" else layers[:-1]
        for l, y in enumerate(generic):
            tags = {f"fsplits={y['fsplits']}" if y["fsplits"] <= 9 else "fsplits>9",
                    f"G={_fwd_groups(cfg.batch, y['bn'], y['N'], y['kc'])}"}
            if y["f_items"] > G:
                tags.add("fwd items > grid")
            if l > 0:
                tags.add("xsplits=1" if y["xsplits"] == 1 else "xsplits>1")
                if y["w_items"] + y["x_items"] > G:
                    tags.add("bwd items > grid")
            if l == L - 1 and y["fsplits"] > 1:
                tags.add("tiled head split")
            for cond, tag in ((y["K"] % 4, "K%4"), (y["N"] % 4, "N%4"), ((y["K"] * y["N"]) % 4, "KN%4"), (y["N"] < 8, "N<8")):
                if cond:
                    tags.add(tag)
            for t in tags:
                seen.setdefault(t, set()).add(cfg.id)
        seen.setdefault(f"head={head} N={cfg.sizes[-1]}", set()).add(cfg.id)
        seen.setdefault(f"L={L} head={head}", set()).add(cfg.id)
        seen.setdefault(f"B={cfg.batch}", set()).add(cfg.id)
    for tag in ("fsplits=1", "fsplits=8", "fsplits=9", "fsplits>9", "G=1", "G=8", "fwd items > grid", "bwd items > grid",
                "xsplits=1", "xsplits>1", "tiled head split", "K%4", "N%4", "KN%4", "N<8", "head=small N=10",
                "head=tiled N=10", "head=small N=32", "head=tiled N=33", "L=1 head=small", "L=1 head=tiled",
                "L=8 head=small", "B=1", "B=7", "B=128"):
        assert tag in seen, (tag, sorted(seen))
    # dX straight through the relu mask and through Xe on the same layer
    assert {"dx-xe-4-splits", "dx-direct"} <= seen["xsplits>1"] | seen["xsplits=1"]
    assert sum(len(c.exact) > 0 for c in CONFIGS) >= 3 and sum(c.native for c in CONFIGS) >= 2
    assert sum(c.priors for c in CONFIGS) >= 3


def test_plan_cache_follows_the_overrides(monkeypatch):
    """Host-only: the planner caches one plan per shape; setting an override replans, clearing it restores the cost model's
    plan (auto, forced, auto), and likewise for the head switch (small, tiled, small)."""
    from lbbnn import _capi as K
    _set_env(monkeypatch, {})
    auto = _describe(K, MNIST, 100)
    monkeypatch.setenv("LBBNN_STEP_PLAN_L0", "8,0,0,0,0,0")
    forced = _describe(K, MNIST, 100)
    monkeypatch.delenv("LBBNN_STEP_PLAN_L0")
    again = _describe(K, MNIST, 100)
    assert forced != auto and again == auto
    assert _parse(forced)[0][0]["bn"] == 8 and _parse(auto)[0][0]["bn"] != 8
    heads = []
    for env in ({}, {"LBBNN_STEP_GENERIC_HEAD": "1"}, {}):
        _set_env(monkeypatch, env)
        heads.append(_parse(_describe(K, MNIST, 100))[1])
    assert heads == ["small", "tiled", "small"]


def _case(cfg):
    rng = np.random.default_rng(sum(cfg.sizes) * 7 + cfg.batch + 1000 * cfg.seed)
    layers = []
    for i, o in zip(cfg.sizes[:-1], cfg.sizes[1:]):
        p = O.init_lrt_params(rng, i, o)
        p["lambdal"] = C.t(rng.normal(0.0, 2.0, size=(o, i)))     # alpha spans (0, 1): the KL gradient's log terms matter
        layers.append(p)
    x = C.t(rng.uniform(0.0, 1.0, size=(cfg.batch, cfg.sizes[0])))
    y = torch.from_numpy(rng.integers(0, cfg.sizes[-1], size=(cfg.batch,))).long()
    return layers, x, y, rng


def _layer_kwargs(cfg, l):
    kw = dict(PRIORS[(l + 1) % 3]) if cfg.priors else {}
    return dict(kw, var_mode="exact" if l in cfg.exact else "reference")


def _trainer(lb, cfg, layers, **kw):
    net = lb.BayesianNetwork(cfg.sizes).cuda()
    with torch.no_grad():
        for l, (layer, p) in enumerate(zip(net.layers, layers)):
            for k, v in p.items():
                getattr(layer, k).copy_(v)
            layer.cfg = lb.LayerConfig(**_layer_kwargs(cfg, l))
    tr = lb.LRTTrainer(net, batch_size=cfg.batch, num_batches=C.NUM_BATCHES, lr=1e-3, seed=SEED, use_graph=False,
                       fused=True, materialize_grads=True, **kw)
    assert tr.fused and tr.kernels_per_step == 1
    return net, tr


def _reference(cfg, x, y, layers64, eps):
    """fp64 nll and per-layer KL of the step, gradients into layers64; also the smallest |hidden pre-activation| relative
    to its layer's largest (a relu mask bit within fp32 rounding of zero would be a property of the case, not the kernel)."""
    h, margin, L = x.double(), 1.0, len(layers64)
    for l, p in enumerate(layers64):
        h = O.lrt_forward(h, p, eps[l].double(), True, var_mode=_layer_kwargs(cfg, l)["var_mode"])
        if l < L - 1:
            a = h.detach().abs()
            margin = min(margin, (a.min() / a.max()).item())
            h = F.relu(h)
    nll = F.nll_loss(F.log_softmax(h, dim=1), y, reduction="sum")
    kls = []
    for l, p in enumerate(layers64):
        kw = _layer_kwargs(cfg, l)
        kls.append(O.lrt_kl(p, O.Priors(kw.get("mu_prior", 0.0), kw.get("sigma_prior", 1.0), kw.get("alpha_prior", 0.05),
                                        kw.get("bias_mu_prior", 0.0), kw.get("bias_sigma_prior", 1.0))))
    (nll + sum(kls) / C.NUM_BATCHES).backward()
    return nll.item(), [k.item() for k in kls], margin


def _run_against_oracle(lb, cfg, monkeypatch, extra_env=None, steps=3):
    _set_env(monkeypatch, dict(cfg.env(), **(extra_env or {})))
    layers, x, y, rng = _case(cfg)
    net, tr = _trainer(lb, cfg, layers, inject_noise=not cfg.native)
    _assert_plan(tr.schedule, cfg)
    L = len(layers)
    layers64 = [{k: v.double().clone().requires_grad_(True) for k, v in p.items()} for p in layers]
    # the step takes lr, betas and eps as C floats: the fp64 Adam runs with those values (1 - float(0.999) is 1.3e-5 off
    # 1e-3, which would show in exp_avg_sq)
    f32 = lambda v: float(np.float32(v))  # noqa: E731
    opt = torch.optim.Adam([v for p in layers64 for v in p.values()], lr=f32(1e-3), betas=(f32(0.9), f32(0.999)),
                           eps=f32(1e-8))
    for step in range(steps):
        if cfg.native:      # the streams the kernel draws: layer l of step s is stream l + s * L
            eps = [lb.philox_normal((cfg.batch, o), SEED, l + step * L).cpu() for l, o in enumerate(cfg.sizes[1:])]
        else:
            eps = [C.t(rng.standard_normal(size=(cfg.batch, o))) for o in cfg.sizes[1:]]
            for buf, e in zip(tr.eps_in, eps):
                buf.copy_(e)
        out = tr.step(x, y)
        kl_dev = tr.stats_host[1:].tolist()
        opt.zero_grad()
        nll, kls, margin = _reference(cfg, x, y, layers64, eps)
        # the case seeds keep this margin >= 2e-6 on the injected-noise cases: far from the kernels' fp32 rounding
        at = f"{cfg.id} step {step} (smallest hidden |pre-activation| / largest {margin:.1e})"
        assert abs(out["nll"] - nll) <= TOL * abs(nll), (at, out["nll"], nll)
        assert abs(out["kl"] - sum(kls)) <= TOL * abs(sum(kls)), (at, out["kl"], sum(kls))
        for l in range(L):
            assert abs(kl_dev[l] - kls[l]) <= TOL * abs(kls[l]), (at, l, kl_dev[l], kls[l])
        for l, (layer, p) in enumerate(zip(net.layers, layers64)):
            for k in NAMES:
                g = getattr(layer, k).grad
                assert C.rel_err(g, p[k].grad) <= TOL, (at, l, k, "grad", C.rel_err(g, p[k].grad))
                p[k].grad = g.detach().cpu().double().clone()      # Adam driven by the kernel's own gradient
        opt.step()
        for l, (layer, p) in enumerate(zip(net.layers, layers64)):
            for k in NAMES:
                par = getattr(layer, k)
                off, n = tr._offsets[(id(layer), k)], par.numel()
                st = opt.state[p[k]]
                for what, got, ref in (("param", par.data, p[k].data), ("exp_avg", tr.exp_avg[off:off + n], st["exp_avg"]),
                                       ("exp_avg_sq", tr.exp_avg_sq[off:off + n], st["exp_avg_sq"])):
                    e = C.rel_err(got.reshape(ref.shape), ref)
                    assert e <= PTOL, (at, l, k, what, e)
                with torch.no_grad():          # the next step starts from the kernel's fp32 parameters on both sides
                    p[k].copy_(par.data.detach().cpu().double())
    return tr


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c.id for c in CONFIGS])
def test_step_plan_matches_fp64_oracle(lb, monkeypatch, cfg):
    _run_against_oracle(lb, cfg, monkeypatch)


# layer 0's dW phase leaves >= 1/8 of the grid idle, so the other layers are updated during it
OVERLAP_CONFIGS = [Cfg("mnist", MNIST, 100, exact=(1,), priors=True, seed=3),
                   Cfg("b128-xe", (96, 256, 128, 10), 128, {0: "64,0,0,0,0,0", 1: "0,0,8,16,8,4"}, native=True)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", OVERLAP_CONFIGS, ids=[c.id for c in OVERLAP_CONFIGS])
def test_overlap_update_matches_fp64_oracle(lb, monkeypatch, cfg):
    """LBBNN_STEP_OVERLAP_UPDATE=1: layers >= 1 are updated by the CTAs without a layer-0 dW tile during that phase.  It sums
    the KL partials in another order than the default, so it is compared with the oracle, not bit for bit."""
    tr = _run_against_oracle(lb, cfg, monkeypatch, {"LBBNN_STEP_OVERLAP_UPDATE": "1"})
    assert _parse(tr.schedule)[0][0]["w_items"] * 8 <= 7 * _grid(), tr.schedule


# phases 1 then 2 against 3: a tiled network with an Xe phase, the small head alone (Lg == 0), the tiled head alone
LAUNCH_CONFIGS = [Cfg("b128-xe", (96, 256, 128, 10), 128, {0: "64,0,0,0,0,0", 1: "0,0,8,16,8,4"}, exact=(1,)),
                  Cfg("one-layer-small-head", (20, 3), 7, priors=True),
                  Cfg("one-layer-tiled-head", (64, 40), 7),
                  Cfg("tiled-head-9-splits", (120, 600, 10), 32, {0: "64,8,0,0,0,0", 1: "8,9,0,0,0,3"}, generic_head=True)]


def _state(tr):
    return [t.clone() for t in (tr.flat, tr.exp_avg, tr.exp_avg_sq, tr.gflat, tr.stats, tr.step_dev)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", LAUNCH_CONFIGS, ids=[c.id for c in LAUNCH_CONFIGS])
def test_two_launch_step_equals_one_launch(lb, monkeypatch, cfg):
    """Forward + backward (phases 1) then the update (phases 2), the launch pair of data-parallel training, on one GPU: the
    parameters, Adam state, gradients and stats are bit-identical to the one-launch step (phases 3), native noise, 3 steps."""
    K = lb._capi
    _set_env(monkeypatch, cfg.env())
    layers, x, y, _ = _case(cfg)
    trs = [_trainer(lb, cfg, layers)[1] for _ in range(2)]
    for tr in trs:
        _assert_plan(tr.schedule, cfg)
        tr.x.copy_(x)
        tr.y.copy_(y)
    for _ in range(3):
        for tr, phases in zip(trs, ((3,), (1, 2))):
            for ph in phases:
                K.check(K.lib.lbbnn_lrt_step_f32(tr._step_desc, ph, tr.ws.data_ptr(), tr.ws.numel(), K.current_stream()))
        torch.cuda.synchronize()
        a, b = _state(trs[0]), _state(trs[1])
        assert all(torch.equal(u, v) for u, v in zip(a, b)), cfg.id
    assert int(trs[0].step_dev) == 3 and torch.isfinite(trs[0].stats).all()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [CONFIGS[0], CONFIGS[4]], ids=[CONFIGS[0].id, CONFIGS[4].id])
def test_step_is_bit_identical_on_repeat(lb, monkeypatch, cfg):
    """Fixed-order reductions throughout: two trainers with the same plan and native noise agree bit for bit over 3 steps."""
    _set_env(monkeypatch, cfg.env())
    layers, x, y, _ = _case(cfg)
    runs = []
    for _ in range(2):
        _, tr = _trainer(lb, cfg, layers)
        _assert_plan(tr.schedule, cfg)
        stats = [tr.step(x, y) for _ in range(3)]
        runs.append((stats, _state(tr)))
    assert runs[0][0] == runs[1][0]
    assert all(torch.equal(u, v) for u, v in zip(runs[0][1], runs[1][1]))


@pytest.mark.gpu
def test_step_limits_fail_loudly(lb, monkeypatch):
    """An override that fits nothing or does not parse, batch 129 and nine layers are rejected when the trainer is built."""
    _set_env(monkeypatch, {})
    ok = Cfg("ok", (20, 3), 7)
    layers, x, y, _ = _case(ok)
    for var, spec, match in (("LBBNN_STEP_PLAN_L1", "0,0,0,0,0,1", "no backward schedule fits layer 1"),
                             ("LBBNN_STEP_PLAN_L0", "8,0,0,0,0,0,", "expected bn,fsplits,rn,ck,bk,xsplits"),
                             ("LBBNN_STEP_PLAN_L0", "0,0,0,0,8,0", "layer 0 has no dX phase"),
                             ("LBBNN_STEP_PLAN_L0", "7,0,0,0,0,0", "no forward schedule fits layer 0")):
        monkeypatch.setenv(var, spec)
        cfg = Cfg("bad", MNIST, 128)
        with pytest.raises(lb.LbbnnError, match=match):
            _trainer(lb, cfg, _case(cfg)[0])
        monkeypatch.delenv(var)
    for sizes, batch in (((20, 3), 129), ((8,) * 9 + (3,), 7)):
        net = lb.BayesianNetwork(sizes).cuda()
        with pytest.raises(lb.LbbnnError, match="fused step kernel needs batch <= 128 and <= 8 layers"):
            lb.LRTTrainer(net, batch_size=batch, num_batches=C.NUM_BATCHES, fused=True, use_graph=False)
    K = lb._capi
    st = K.Step()
    st.n_layers, st.batch = 9, 7
    assert K.lib.lbbnn_lrt_step_workspace_bytes(st) == 0 and b"n_layers" in K.lib.lbbnn_last_error()
    torch.cuda.synchronize()           # nothing was launched: the context is healthy
    _, tr = _trainer(lb, ok, layers)    # and the limits themselves are fine (batch 128 and 8 layers: CONFIGS above)
    assert np.isfinite(tr.step(x, y)["loss"])
