"""LRTReplicaTrainer: R LRT networks trained side by side in one launch of the persistent step kernel (lrt_step_kernel's
replica instantiation, csrc/lrt_step.cuh), against
  - the float64 oracle per replica, driving a float64 Adam with the kernel's own gradients, with the bounds of
    test_lrt_step_plans_gpu.py: nll and KL (total and per layer) 1e-5 relative, every gradient 1e-5, parameters and both
    Adam moments 2e-6 after each of 3 steps;
  - the single-network kernel (LRTTrainer) bit for bit under one plan, and R = 1 on the auto plan;
  - itself: permuted replicas, graph replay against eager launches, repeats."""
import re

import numpy as np
import pytest
import torch

import cases as C
import test_lrt_step_plans_gpu as S

MNIST = S.MNIST
ITEMS_RE = re.compile(r"l(\d+)\((\d+)->(\d+)\) F bn=\d+ kc=\d+ items=(\d+)x(\d+) \| W \d+x\d+ items=(\d+) \| X bk=\d+ nc=\d+ "
                      r"items=(\d+)x(\d+); ")


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def _net(lb, cfg, layers):
    net = lb.BayesianNetwork(cfg.sizes).cuda()
    with torch.no_grad():
        for l, (layer, p) in enumerate(zip(net.layers, layers)):
            for k, v in p.items():
                getattr(layer, k).copy_(v)
            layer.cfg = lb.LayerConfig(**S._layer_kwargs(cfg, l))
    return net


def _replica_cases(cfg, R, shared):
    """R cases with distinct parameters (and, unless shared, distinct minibatches and labels)."""
    out = []
    for r in range(R):
        layers, x, y, rng = S._case(S.Cfg(cfg.id, cfg.sizes, cfg.batch, seed=cfg.seed + 11 * r + 1))
        out.append([layers, x, y, rng])
    if shared:
        for o in out[1:]:
            o[1], o[2] = out[0][1], out[0][2]
    return out


SEEDS = lambda R: [S.SEED + 1000 * r + 7 for r in range(R)]  # noqa: E731


@pytest.mark.gpu
@pytest.mark.parametrize("cfg, R, shared, check", [
    (S.Cfg("mnist-injected", MNIST, 100, seed=5), 3, False, None),
    (S.Cfg("mnist-shared-native", MNIST, 100, exact=(0, 2), priors=True, native=True, seed=6), 3, True, None),
    (S.Cfg("ragged-tiled", (37, 23, 6, 3), 7, {0: "16,3,8,16,0,0", 1: "8,2,8,16,16,2", 2: "0,0,0,0,8,1"},
           generic_head=True, exact=(1,), priors=True, seed=7), 5, False, None),
    # case seed 13: the checked replicas' smallest hidden |pre-activation| is >= 3e-6 of the largest (no relu bit within
    # fp32 rounding of zero)
    (S.Cfg("mnist-r32", MNIST, 100, seed=13), 32, False, (0, 17, 31)),
], ids=["mnist-r3-injected", "mnist-r3-shared-native-priors-exact", "ragged-r5-tiled-head", "mnist-r32"])
def test_replicas_match_fp64_oracle(lb, monkeypatch, cfg, R, shared, check):
    S._set_env(monkeypatch, cfg.env())
    cases = _replica_cases(cfg, R, shared)
    nets = [_net(lb, cfg, c[0]) for c in cases]
    tr = lb.LRTReplicaTrainer(nets, batch_size=cfg.batch, num_batches=C.NUM_BATCHES, seeds=SEEDS(R), shared_batch=shared,
                              use_graph=False, inject_noise=not cfg.native)
    head = S.HEAD_RE.search(tr.schedule.replace(f" replicas={R}", ""))
    assert head and head.group(1) == ("tiled" if cfg.generic_head or R * cfg.batch > 8 * S._grid() else "small"), tr.schedule
    if R == 32:   # more head rows than 8 per CTA, and more forward and backward items than CTAs
        G = S._grid()
        items = [tuple(map(int, m.groups())) for m in ITEMS_RE.finditer(tr.schedule)]
        assert R * cfg.batch > 8 * G and head.group(1) == "tiled"
        assert any(R * ft * fs > G for _, _, _, ft, fs, _, _, _ in items), tr.schedule
        assert any(R * (nw + xt * xs) > G for l, _, _, _, _, nw, xt, xs in items if l > 0), tr.schedule
    check = range(R) if check is None else check
    L = len(cfg.sizes) - 1
    f32 = lambda v: float(np.float32(v))  # noqa: E731
    side = {}
    for r in check:
        layers64 = [{k: v.double().clone().requires_grad_(True) for k, v in p.items()} for p in cases[r][0]]
        opt = torch.optim.Adam([v for p in layers64 for v in p.values()], lr=f32(1e-3), betas=(f32(0.9), f32(0.999)),
                               eps=f32(1e-8))
        side[r] = (layers64, opt)
    xs = torch.stack([c[1] for c in cases]) if not shared else cases[0][1]
    ys = torch.stack([c[2] for c in cases]) if not shared else cases[0][2]
    for step in range(3):
        if cfg.native:
            eps = [[lb.philox_normal((cfg.batch, o), SEEDS(R)[r], l + step * L).cpu() for l, o in enumerate(cfg.sizes[1:])]
                   for r in range(R)]
        else:
            eps = [[C.t(c[3].standard_normal(size=(cfg.batch, o))) for o in cfg.sizes[1:]] for c in cases]
            for l, buf in enumerate(tr.eps_in):
                buf.copy_(torch.stack([eps[r][l] for r in range(R)]))
        out = tr.step(xs, ys)
        kl_dev = tr.stats_host[:, 1:]
        for r in check:
            layers64, opt = side[r]
            opt.zero_grad()
            nll, kls, margin = S._reference(cfg, cases[r][1], cases[r][2], layers64, eps[r])
            at = f"{cfg.id} replica {r} step {step} (margin {margin:.1e})"
            assert abs(out["nll"][r] - nll) <= S.TOL * abs(nll), (at, out["nll"][r], nll)
            assert abs(out["kl"][r] - sum(kls)) <= S.TOL * abs(sum(kls)), (at, out["kl"][r], sum(kls))
            for l in range(L):
                assert abs(kl_dev[r, l].item() - kls[l]) <= S.TOL * abs(kls[l]), (at, l)
            for l, (layer, p) in enumerate(zip(nets[r].layers, layers64)):
                for k in S.NAMES:
                    g = getattr(layer, k).grad
                    assert C.rel_err(g, p[k].grad) <= S.TOL, (at, l, k, "grad", C.rel_err(g, p[k].grad))
                    p[k].grad = g.detach().cpu().double().clone()
            opt.step()
            for l, (layer, p) in enumerate(zip(nets[r].layers, layers64)):
                for k in S.NAMES:
                    par = getattr(layer, k)
                    off, n = tr._offsets[(l, k)], par.numel()
                    st = opt.state[p[k]]
                    for what, got, ref in (("param", par.data, p[k].data), ("exp_avg", tr.exp_avg[r, off:off + n], st["exp_avg"]),
                                           ("exp_avg_sq", tr.exp_avg_sq[r, off:off + n], st["exp_avg_sq"])):
                        e = C.rel_err(got.reshape(ref.shape), ref)
                        assert e <= S.PTOL, (at, l, k, what, e)
                    with torch.no_grad():
                        p[k].copy_(par.data.detach().cpu().double())
    assert int(tr.step_dev) == 3


def _plan_env(schedule):
    """LBBNN_STEP_PLAN_L<i> values that force a schedule string's plan on every layer."""
    env = {}
    for m in re.finditer(r"l(\d+)\(\d+->\d+\) F bn=(\d+) kc=\d+ items=\d+x(\d+) \| W (\d+)x(\d+) items=\d+ \| X bk=(\d+) nc=\d+ "
                         r"items=\d+x(\d+); ", schedule):
        l, bn, fs, rn, ck, bk, xs = map(int, m.groups())
        env[f"LBBNN_STEP_PLAN_L{l}"] = f"{bn},{fs},{rn},{ck},{bk if l else 0},{xs if l else 0}"
    return env


def _single(lb, cfg, layers, seed):
    net = _net(lb, cfg, layers)
    return net, lb.LRTTrainer(net, batch_size=cfg.batch, num_batches=C.NUM_BATCHES, seed=seed, use_graph=False, fused=True)


def _assert_replica_equals_single(tr, r, single, what):
    for name, a, b in (("flat", tr.flat[r], single.flat), ("exp_avg", tr.exp_avg[r], single.exp_avg),
                       ("exp_avg_sq", tr.exp_avg_sq[r], single.exp_avg_sq), ("grad", tr.gflat[r], single.gflat)):
        assert torch.equal(a, b), (what, r, name, (a - b).abs().max().item())


@pytest.mark.gpu
def test_replicas_equal_the_single_network_kernel_bit_for_bit(lb, monkeypatch):
    """R = 4, native noise, one plan forced on both sides: after 3 steps every replica's parameters, moments and gradients are
    LRTTrainer(net_r, seed=seeds[r])'s bit for bit; nll and KL agree to 1e-6 (their cross-CTA sums run in another order)."""
    cfg, R = S.Cfg("mnist", MNIST, 100, exact=(1,), priors=True, native=True, seed=9), 4
    S._set_env(monkeypatch, {})
    cases = _replica_cases(cfg, R, False)
    _, probe = _single(lb, cfg, cases[0][0], 0)
    S._set_env(monkeypatch, _plan_env(probe.schedule))
    singles = [_single(lb, cfg, c[0], s)[1] for c, s in zip(cases, SEEDS(R))]
    tr = lb.LRTReplicaTrainer([_net(lb, cfg, c[0]) for c in cases], batch_size=cfg.batch, num_batches=C.NUM_BATCHES,
                              seeds=SEEDS(R), use_graph=False)
    assert tr.schedule == probe.schedule + f" replicas={R}" and all(s.schedule == probe.schedule for s in singles)
    xs, ys = torch.stack([c[1] for c in cases]), torch.stack([c[2] for c in cases])
    for _ in range(3):
        out = tr.step(xs, ys)
        for r, s in enumerate(singles):
            o = s.step(xs[r], ys[r])
            for k in ("nll", "kl"):
                assert abs(out[k][r] - o[k]) <= 1e-6 * abs(o[k]), (r, k, out[k][r], o[k])
    torch.cuda.synchronize()
    for r, s in enumerate(singles):
        _assert_replica_equals_single(tr, r, s, "R=4 forced plan")


@pytest.mark.gpu
def test_one_replica_is_the_single_network_step(lb, monkeypatch):
    """R = 1 on the auto plan: the same schedule string as LRTTrainer, bit-identical parameters, moments and gradients."""
    cfg = S.Cfg("mnist", MNIST, 100, exact=(0, 2), priors=True, native=True, seed=10)
    S._set_env(monkeypatch, {})
    (layers, x, y, _), = _replica_cases(cfg, 1, False)
    _, single = _single(lb, cfg, layers, 77)
    tr = lb.LRTReplicaTrainer([_net(lb, cfg, layers)], batch_size=cfg.batch, num_batches=C.NUM_BATCHES, seeds=[77],
                              use_graph=False)
    assert tr.schedule == single.schedule
    for _ in range(3):
        out, o = tr.step(x[None], y[None]), single.step(x, y)
        assert abs(out["loss"][0] - o["loss"]) <= 1e-6 * abs(o["loss"])
    torch.cuda.synchronize()
    _assert_replica_equals_single(tr, 0, single, "R=1 auto plan")


def _state(tr):
    return [t.clone() for t in (tr.flat, tr.exp_avg, tr.exp_avg_sq, tr.gflat, tr.stats, tr.step_dev)]


@pytest.mark.gpu
def test_replicas_are_independent_and_deterministic(lb, monkeypatch):
    """Permuting the nets and seeds permutes parameters, moments and gradients bit for bit (nll and KL to 1e-6); a graph
    replay equals an eager launch bit for bit, and a repeat is bit-identical."""
    cfg, R = S.Cfg("mnist", MNIST, 100, native=True, seed=12), 5
    S._set_env(monkeypatch, {})
    cases = _replica_cases(cfg, R, False)
    xs, ys = torch.stack([c[1] for c in cases]), torch.stack([c[2] for c in cases])
    perm = [3, 0, 4, 1, 2]

    def run(order, use_graph):
        tr = lb.LRTReplicaTrainer([_net(lb, cfg, cases[r][0]) for r in order], batch_size=cfg.batch,
                                  num_batches=C.NUM_BATCHES, seeds=[SEEDS(R)[r] for r in order], use_graph=use_graph)
        outs = [tr.step(xs[order], ys[order]) for _ in range(3)]
        return tr, outs, _state(tr)

    tr0, out0, st0 = run(list(range(R)), False)
    _, out1, st1 = run(perm, False)
    for a, b in zip(st0[:4], st1[:4]):
        assert torch.equal(a[perm], b)
    for k in ("nll", "kl"):
        for i, r in enumerate(perm):
            assert abs(out1[-1][k][i] - out0[-1][k][r]) <= 1e-6 * abs(out0[-1][k][r])
    _, out2, st2 = run(list(range(R)), True)     # graph replay
    _, out3, st3 = run(list(range(R)), False)    # repeat
    for st in (st2, st3):
        assert all(torch.equal(a, b) for a, b in zip(st0, st))
    assert out2 == out0 and out3 == out0
    assert int(tr0.step_dev) == 3 and np.isfinite(out0[-1]["loss"]).all()
