"""The fused coupling-flow kernels (csrc/flows.cu) in every launch configuration they pick at run time, against the float64
oracle (flows2.py RNVP / IAF-style 'MNF' transform, lbbnn_oracle.propagate_flow):
  - the cluster width C = 1, 2, 4, 8 (cluster_for(D)) on both sides of each switch, and at D that no C divides, so the
    per-CTA slices of the output dims do not start on a quad boundary;
  - the narrow (every hidden layer <= 80) and the wide kernel instantiation, RNVP with 1 to 6 hidden layers, IAF;
  - 1, 3 and 8 transforms, 1 to 7 rows (and 300 rows forward only), one-sided backward (dz_out or dlogdet NULL);
  - the native masks through mask_quad's per-element path (rows that do not start on a quad boundary);
  - bit-identical repeats at every C, and the limits.
Tolerances as in test_mnf_gpu.py: 1e-5 (max|a-b|/max|b|) on outputs and log-dets, 5e-5 on dz, and on every parameter
gradient the larger of 5e-5 and four times the fp32 oracle's own distance from the fp64 truth."""
import numpy as np
import pytest
import torch

import cases as C
import lbbnn_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5
GTOL = 5e-5


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def cluster_width(D):
    """Host copy of cluster_for() in csrc/flows.cu."""
    c = 1
    while c < 8 and D // (2 * c) >= 48:
        c *= 2
    return c


def _flow(lb, kind, D, T, h_sizes, hidden, named):
    kw = dict(h_sizes=h_sizes) if kind == "RNVP" else dict(hidden=hidden)
    flow = lb.flows.PropagateFlow(kind, D, T, **kw)
    flow.load_state_dict({k[len("z_flow."):]: v for k, v in named.items()})
    return flow.cuda()


def _oracle(z0, masks, tmpl, named, kind, gz, gl, dtype, backward=True):
    """Oracle forward (per-row log-dets for both kinds: the IAF kind sums over rows, so it runs one row at a time) and, if
    asked, the gradients of sum(gz * z_out) + sum(gl * logdet)."""
    nm = {k: v.to(dtype).clone().requires_grad_(backward) for k, v in named.items()}
    tps = C.unflatten_like({"z_flow": tmpl}, nm)["z_flow"]
    z = z0.to(dtype).clone().requires_grad_(backward)
    ms = [m.to(dtype) for m in masks]
    if kind == "RNVP":
        zo, ld = O.propagate_flow(z, ms, tps, kind)
    else:
        outs = [O.propagate_flow(z[r:r + 1], [m[r:r + 1] for m in ms], tps, kind) for r in range(z.shape[0])]
        zo, ld = torch.cat([o[0] for o in outs]), torch.stack([o[1] for o in outs])
    if not backward:
        return zo, ld, None, None
    ((zo * gz.to(dtype)).sum() + (ld * gl.to(dtype)).sum()).backward()
    return zo.detach(), ld.detach(), z.grad, {k: v.grad for k, v in nm.items()}


def _case(kind, D, rows, T, h_sizes, hidden, seed):
    rng = np.random.default_rng(seed)
    tmpl = O.init_flow_params(rng, D, T, h_sizes or (75,) * 4, kind, hidden=hidden)
    named = C.flat_named({"z_flow": tmpl})
    z0 = C.t(rng.standard_normal(size=(rows, D)))
    masks = C._masks(rng, T, rows, D)
    gz = C.t(rng.standard_normal(size=(rows, D)))
    gl = C.t(rng.standard_normal(size=(rows,)))
    return tmpl, named, z0, masks, gz, gl


def _check_grads(zgrad, pgrads, t64, t32):
    assert C.rel_err(zgrad, t64[2]) < GTOL
    for k, ref in t64[3].items():
        bound = max(GTOL, 4 * C.rel_err(t32[3][k], ref))
        assert C.rel_err(pgrads[k], ref) < bound, k


# (kind, D, rows, T, h_sizes (RNVP) / hidden (IAF)); the comment gives the cluster width and the kernel instantiation
CONFIGS = [
    ("RNVP", 95, 2, 2, (80,)),             # C 1, narrow at its limit, the only hidden layer is the last
    ("RNVP", 96, 2, 3, (81,)),             # C 2, wide just past the limit
    ("RNVP", 191, 1, 1, (128, 128)),       # C 2, widest hidden layers
    ("RNVP", 192, 7, 2, (33, 128)),        # C 4, wide
    ("RNVP", 383, 2, 3, (64,) * 6),        # C 4, narrow, deepest conditioner
    ("RNVP", 384, 1, 8, (80,)),            # C 8, narrow, most transforms
    ("RNVP", 193, 2, 2, (75, 75)),         # C 4, ragged: slices start at 49, 98, 147
    ("RNVP", 201, 7, 3, (81,)),            # C 4, ragged, wide
    ("RNVP", 785, 2, 2, (75,) * 4),        # C 8, ragged
    ("RNVP", 37, 1, 1, (128,)),            # C 1, wide, one hidden layer
    ("RNVP", 600, 7, 2, (80, 80)),         # C 8, narrow
    ("MNF", 96, 2, 2, 64),                 # C 2, narrow IAF
    ("MNF", 201, 7, 3, 128),               # C 4, wide IAF, ragged
    ("MNF", 384, 1, 1, 64),                # C 8, narrow IAF
    ("MNF", 785, 2, 2, 128),               # C 8, wide IAF, ragged
    ("MNF", 95, 7, 8, 100),                # C 1, IAF at the reference's width, most transforms
]


def _cfg_id(c):
    kind, D, rows, T, h = c
    return f"{kind}-D{D}-C{cluster_width(D)}-r{rows}-T{T}-h{'x'.join(map(str, h)) if kind == 'RNVP' else h}"


@pytest.mark.parametrize("cfg", CONFIGS, ids=[_cfg_id(c) for c in CONFIGS])
def test_flow_config_matches_fp64_oracle(lb, cfg):
    kind, D, rows, T, h = cfg
    h_sizes, hidden = (h, 100) if kind == "RNVP" else (None, h)
    tmpl, named, z0, masks, gz, gl = _case(kind, D, rows, T, h_sizes, hidden, seed=D * 31 + rows * 7 + T)
    t64 = _oracle(z0, masks, tmpl, named, kind, gz, gl, torch.float64)
    t32 = _oracle(z0, masks, tmpl, named, kind, gz, gl, torch.float32)
    flow = _flow(lb, kind, D, T, h_sizes, hidden, named)
    z = z0.cuda().requires_grad_(True)
    zo, ld = flow(z, [m.cuda() for m in masks], per_row=True)
    ((zo * gz.cuda()).sum() + (ld * gl.cuda()).sum()).backward()
    assert C.rel_err(zo.detach(), t64[0]) < TOL and C.rel_err(ld.detach(), t64[1]) < TOL
    _check_grads(z.grad, {"z_flow." + k: v.grad for k, v in flow.named_parameters()}, t64, t32)


@pytest.mark.parametrize("kind,D,h", [("RNVP", 201, (75,) * 4), ("MNF", 385, 100)])
def test_flow_forward_many_rows(lb, kind, D, h):
    """300 rows in one launch (the ensemble predictor batches its flow evaluations as rows)."""
    rows, T = 300, 2
    h_sizes, hidden = (h, 100) if kind == "RNVP" else (None, h)
    tmpl, named, z0, masks, gz, gl = _case(kind, D, rows, T, h_sizes, hidden, seed=D + 1)
    zo64, ld64, _, _ = _oracle(z0, masks, tmpl, named, kind, gz, gl, torch.float64, backward=False)
    flow = _flow(lb, kind, D, T, h_sizes, hidden, named)
    with torch.no_grad():
        zo, ld = flow(z0.cuda(), [m.cuda() for m in masks], per_row=True)
    assert C.rel_err(zo, zo64) < TOL and C.rel_err(ld, ld64) < TOL


def _flow_capi(lb, flow, z, masks, dz, dld):
    """lbbnn_flow_fwd / lbbnn_flow_bwd called directly, so that an absent output gradient reaches the kernel as NULL (the
    autograd path materialises it as zeros).  Returns z_out, logdet, dz_in and {name: gradient}."""
    K = lb._capi
    R, D = z.shape
    params = [p.detach().contiguous() for p in flow._params()]
    f = lb.flows._build_flow(flow.kind, D, len(flow.transforms), flow.n_hidden, params)
    zo, ld = torch.empty_like(z), torch.empty(R, device=z.device)
    save = torch.empty(int(K.lib.lbbnn_flow_save_floats(f, R)), device=z.device)
    noise = K.make_noise(None, 1, 2)
    K.check(K.lib.lbbnn_flow_fwd(f, K.ptr(z), R, K.ptr(masks), noise, K.ptr(zo), K.ptr(ld), K.ptr(save), K.current_stream()))
    gbuf = torch.empty(R, sum(p.numel() for p in params), device=z.device)
    gt, offs = lb.mnf._flow_grad_table(f, params, gbuf)
    dzi = torch.empty_like(z)
    K.check(K.lib.lbbnn_flow_bwd(f, gt, R, K.ptr(masks), noise, K.ptr(dz, allow_none=True), K.ptr(dld, allow_none=True),
                                 K.ptr(save), K.ptr(dzi), K.current_stream()))
    g = gbuf.sum(0)
    names = [n for n, _ in flow.named_parameters()]
    return zo, ld, dzi, {"z_flow." + n: g[offs[j]:offs[j + 1]].view_as(params[j]) for j, n in enumerate(names)}


@pytest.mark.parametrize("kind,D,h,side", [("RNVP", 201, (75, 75), "z"), ("RNVP", 201, (75, 75), "logdet"),
                                           ("MNF", 193, 64, "z"), ("MNF", 96, 128, "logdet")])
def test_flow_one_sided_backward(lb, kind, D, h, side):
    """A loss on z_out only (dlogdet == NULL) or on the log-dets only (dz_out == NULL)."""
    rows, T = 2, 2
    h_sizes, hidden = (h, 100) if kind == "RNVP" else (None, h)
    tmpl, named, z0, masks, gz, gl = _case(kind, D, rows, T, h_sizes, hidden, seed=D + 2)
    if side == "z":
        gl = torch.zeros_like(gl)
    else:
        gz = torch.zeros_like(gz)
    t64 = _oracle(z0, masks, tmpl, named, kind, gz, gl, torch.float64)
    t32 = _oracle(z0, masks, tmpl, named, kind, gz, gl, torch.float32)
    flow = _flow(lb, kind, D, T, h_sizes, hidden, named)
    m = torch.stack(masks).cuda()
    zo, ld, dz, pg = _flow_capi(lb, flow, z0.cuda(), m, gz.cuda() if side == "z" else None,
                                gl.cuda() if side == "logdet" else None)
    assert C.rel_err(zo, t64[0]) < TOL and C.rel_err(ld, t64[1]) < TOL
    _check_grads(dz, pg, t64, t32)
    # the NULL gradient acts exactly as a zero one
    zo2, ld2, dz2, pg2 = _flow_capi(lb, flow, z0.cuda(), m, gz.cuda(), gl.cuda())
    assert torch.equal(dz, dz2) and all(torch.equal(pg[k], pg2[k]) for k in pg)


@pytest.mark.parametrize("kind,D,h", [("RNVP", 37, (75, 75)), ("RNVP", 201, (81,)), ("MNF", 201, 64)])
def test_flow_native_masks_per_element_path(lb, kind, D, h):
    """D % 4 != 0 with 5 rows: rows 1.. do not start on a quad boundary, so the kernels draw those rows' masks element by
    element.  The masks rebuilt from the exported Philox uniforms, injected, reproduce the native forward and backward
    bit for bit, and the fp64 oracle fed the same masks agrees."""
    rows, T = 5, 2
    h_sizes, hidden = (h, 100) if kind == "RNVP" else (None, h)
    tmpl, named, z0, _, gz, gl = _case(kind, D, rows, T, h_sizes, hidden, seed=D + 3)
    lb.manual_seed(91)
    flow = _flow(lb, kind, D, T, h_sizes, hidden, named)
    z = z0.cuda().requires_grad_(True)
    zo, ld = flow(z, per_row=True)
    ((zo * gz.cuda()).sum() + (ld * gl.cuda()).sum()).backward()
    seed, stream = flow.last_noise_key
    native = (zo.detach(), ld.detach(), z.grad.clone(), [p.grad.clone() for p in flow.parameters()])
    masks = [(lb.philox_uniform(rows * D, seed, stream + t, device="cuda") < 0.5).float().view(rows, D) for t in range(T)]
    assert 0.4 < torch.stack(masks).mean().item() < 0.6
    flow.zero_grad()
    z = z0.cuda().requires_grad_(True)
    zo, ld = flow(z, masks, per_row=True)
    ((zo * gz.cuda()).sum() + (ld * gl.cuda()).sum()).backward()
    assert torch.equal(zo.detach(), native[0]) and torch.equal(ld.detach(), native[1])
    assert torch.equal(z.grad, native[2]) and all(torch.equal(p.grad, g) for p, g in zip(flow.parameters(), native[3]))
    cpu_masks = [m.cpu() for m in masks]
    t64 = _oracle(z0, cpu_masks, tmpl, named, kind, gz, gl, torch.float64)
    t32 = _oracle(z0, cpu_masks, tmpl, named, kind, gz, gl, torch.float32)
    assert C.rel_err(native[0], t64[0]) < TOL and C.rel_err(native[1], t64[1]) < TOL
    _check_grads(native[2], {"z_flow." + k: v.grad for k, v in flow.named_parameters()}, t64, t32)


@pytest.mark.parametrize("D", [60, 150, 300, 500])
def test_flow_bit_identical_repeats(lb, D):
    """The kernels sum the cluster's log-det partials and the all-reduced conditioner gradient in a fixed order: two
    identical calls agree bit for bit at every cluster width (a missing cluster barrier shows up here first)."""
    C_ = cluster_width(D)
    assert C_ == {60: 1, 150: 2, 300: 4, 500: 8}[D]
    rows, T = 3, 3
    tmpl, named, z0, masks, gz, gl = _case("RNVP", D, rows, T, (75, 75), 100, seed=D + 4)
    flow = _flow(lb, "RNVP", D, T, (75, 75), 100, named)
    runs = []
    for _ in range(2):
        flow.zero_grad()
        z = z0.cuda().requires_grad_(True)
        zo, ld = flow(z, [m.cuda() for m in masks], per_row=True)
        ((zo * gz.cuda()).sum() + (ld * gl.cuda()).sum()).backward()
        runs.append([zo.detach(), ld.detach(), z.grad] + [p.grad.clone() for p in flow.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*runs))


def test_flow_limits_fail_loudly(lb):
    z = torch.randn(2, 40, device="cuda")
    for flow in (lb.flows.PropagateFlow("RNVP", 40, 2, h_sizes=(75, 129)), lb.flows.PropagateFlow("MNF", 40, 2, hidden=129)):
        with pytest.raises(lb.LbbnnError, match="bad hidden layer"):
            flow.cuda()(z)
    torch.cuda.synchronize()           # the rejected calls launched nothing: the context is healthy
    with pytest.raises(ValueError):
        lb.flows.PropagateFlow("RNVP", 40, 9)
    with pytest.raises(ValueError):
        lb.flows.PropagateFlow("MNF", 40, 9)
    with pytest.raises(ValueError):
        lb.flows.PropagateFlow("RNVP", 40, 2, h_sizes=(20,) * 7)
    ok = lb.flows.PropagateFlow("RNVP", 40, 8, h_sizes=(20,) * 6).cuda()     # the largest stack the kernels take
    zo, ld = ok(z, per_row=True)
    assert torch.isfinite(zo).all() and torch.isfinite(ld).all()


@pytest.mark.parametrize("kind,i,o,T", [("RNVP", 150, 11, 3), ("RNVP", 203, 9, 1), ("MNF", 203, 9, 3), ("MNF", 150, 11, 1)])
def test_mnf_layer_flow_depths_match_fp64_oracle(lb, kind, i, o, T):
    """lbbnn.mnf.BayesianLinear with 1 or 3 transforms per flow, at in_features 150 (C 2) and 203 (C 4, ragged slices)."""
    case = C.mnf_layer_case(i * 10 + T, 6, i, o, T=T, kind=kind)
    named64 = {k: v.double().clone().requires_grad_(True) for k, v in C.flat_named(case["p"]).items()}
    p64 = C.unflatten_like(case["p"], named64)
    x64 = case["x"].double().clone().requires_grad_(True)
    nz64 = {k: ([m.double() for m in v] if isinstance(v, list) else v.double()) for k, v in case["noise"].items()}
    act64, kl64 = O.mnf_forward(x64, p64, nz64, kind=kind)
    ((act64 * case["gout"].double()).sum() + kl64 / C.NUM_BATCHES).backward()

    layer = lb.mnf.BayesianLinear(i, o, T, z_flow_type=kind, r_flow_type=kind)
    layer.load_state_dict(C.flat_named(case["p"]))
    layer = layer.cuda().train()
    x = case["x"].cuda().requires_grad_(True)
    noise = {k: ([m.cuda() for m in v] if isinstance(v, list) else v.cuda()) for k, v in case["noise"].items()}
    act = layer(x, noise=noise)
    ((act * case["gout"].cuda()).sum() + layer.kl / C.NUM_BATCHES).backward()
    assert C.rel_err(act.detach(), act64.detach()) < TOL
    assert abs(layer.kl.item() - kl64.item()) / abs(kl64.item()) < TOL
    assert C.rel_err(x.grad, x64.grad) < TOL
    got = dict(layer.named_parameters())
    assert set(got) == set(named64)
    for name, v in named64.items():
        assert got[name].grad is not None, name
        assert C.rel_err(got[name].grad, v.grad) < GTOL, name
