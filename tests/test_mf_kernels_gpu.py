"""The MF weight-sampling kernels of csrc/mf.cu through the C-ABI, against a float64 torch restatement of what they compute:
  w  = g (mu + sigma eps)   (g = gamma; alpha_stale or alpha for the joint mean; ws = mu for the two means)
  s0 = sum g_wp   s1 = sum wl^2   s2 = sum lgamma(1 + pb - g_gp) - lgamma(2 - g_gp)
  s3 = sum log(g N(wl; mu, sigma) + (1 - g) + 1e-8)   s4 = sum g_b log(alpha + 1e-8) + (1 - g_b) log(1 - alpha + 1e-8)
(wl = ws with LP_ON_WS, else w; g_x = round(g) under the matching EXACT_* flag) and the derivatives of
sum(dw w) + sum_k c_k s_k, by autograd.  w within 1e-5 (max|a-b|/max|b|); the elementwise gradients within the larger of
1e-5 and four times the distance of the same expressions in fp32 torch from the fp64 truth, and the sums and dpb within the
larger of 1e-5 and that multiple, entry by entry.

Covered: sizes from one element to past the grid cap (grid-stride loop, many-block ticket reduction), every mode and flag
combination, unaligned operands, the three per-thread widths (LBBNN_MF_SPLIT, read once per process, so widths 1 and 4 run
in a subprocess: this file is also that subprocess's script), the ticket entry points eager and in a CUDA graph, the
native Philox draws at odd sizes, and the one-block prior kernels.

    python tests/test_mf_kernels_gpu.py OUT.npz       writes the width cases with this process's LBBNN_MF_SPLIT"""
import itertools
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases as C

pytestmark = pytest.mark.gpu
TOL = 1e-5
SUM_FLOOR = 1e-5
K_TINY = 1.1754943508222875e-38           # torch.finfo(float32).tiny: the relaxed draw's lower clip
K_EPS = 1.1920928955078125e-07            # torch.finfo(float32).eps: its upper clip is 1 - eps
SEED, STREAM = 1234, 77
GRAPH_STRIDE = 0x9E3779B1


def _capi():
    from lbbnn import _capi as K
    K.require_device()
    return K


def big_n():
    """Twice the capped grid (8 blocks per SM, 256 threads) at four elements per thread, plus 3: the grid-stride loop and
    a ragged tail at every width."""
    return 2 * 8 * torch.cuda.get_device_properties(0).multi_processor_count * 256 * 4 + 3


def _size(spec):
    return big_n() if spec == "big" else spec


def _flags(K):
    """LOGPROBS with every combination of the four modifier flags."""
    mods = (K.MF_FLAG_LP_ON_WS, K.MF_FLAG_EXACT_GAMMA, K.MF_FLAG_EXACT_WPRIOR, K.MF_FLAG_EXACT_GPRIOR)
    return [K.MF_FLAG_LOGPROBS | sum(c) for r in range(5) for c in itertools.combinations(mods, r)]


def _inputs(n, seed, offset=0):
    """fp32 CUDA operands of n elements.  Relaxed gammas over (0, 1), every 7th from the 4th at the lower clip and every 7th
    from the 5th at the upper clip; pb = 0.05.  offset > 0: every operand is a contiguous view at that storage offset, so
    that alignment alone rules out the float4 path."""
    rng = np.random.default_rng(seed)
    g = rng.uniform(0.0, 1.0, size=n)
    g[3::7] = K_TINY
    g[4::7] = 1.0 - K_EPS
    lam = rng.normal(0.0, 2.0, size=n)
    host = {"mu": rng.uniform(-0.2, 0.2, size=n), "rho": rng.uniform(-3.5, -1.0, size=n), "lam": lam, "gamma": g,
            "alpha_stale": 1.0 / (1.0 + np.exp(-(lam + rng.normal(0.0, 0.3, size=n)))), "eps": rng.standard_normal(size=n),
            "dw": rng.standard_normal(size=n)}
    out = {}
    for k, v in host.items():
        buf = torch.empty(n + offset, dtype=torch.float32, device="cuda")
        buf[offset:] = C.t(v).cuda()
        out[k] = buf[offset:]
    out["pb"] = torch.tensor([0.05], device="cuda")
    out["c"] = C.t(rng.standard_normal(size=5)).cuda()
    return out


def _native_eps(n, step=0):
    from lbbnn import philox_normal
    return philox_normal(n, SEED, (STREAM + step * GRAPH_STRIDE) % 2 ** 64)


def _noise(K, x, native, step_dev=None):
    if native:
        return K.make_noise(None, SEED, STREAM, step_dev, GRAPH_STRIDE if step_dev is not None else 0)
    return K.make_noise(x["eps"])


def _fwd(K, x, mode, flags, native=False, ticket=None, stale=True, out=None, step_dev=None):
    n = x["mu"].numel()
    o = out or {"w": torch.full((n,), float("nan"), device="cuda"), "sums": torch.full((5,), float("nan"), device="cuda")}
    ws = torch.empty(int(K.lib.lbbnn_mf_workspace_bytes(n)), dtype=torch.uint8, device="cuda")
    o["_keep"] = ws
    gamma = None if mode == K.MF_JOINTMEAN else x["gamma"]
    stale_t = x["alpha_stale"] if mode == K.MF_JOINTMEAN and stale else None
    args = [K.ptr(x["mu"]), K.ptr(x["rho"]), K.ptr(x["lam"]), K.ptr(gamma, True), K.ptr(stale_t, True), K.ptr(x["pb"]), n,
            _noise(K, x, native, step_dev), mode, flags, K.ptr(o["w"]), K.ptr(o["sums"]), ws.data_ptr(), ws.numel()]
    if ticket is None:
        K.check(K.lib.lbbnn_mf_sample_fwd(*args, K.current_stream()))
    else:
        K.check(K.lib.lbbnn_mf_sample_fwd_ticket(*args, ticket.data_ptr(), K.current_stream()))
    return o


def _bwd(K, x, flags, native=False, ticket=None, use_dw=True, use_c=True, want_dgamma=True, out=None, step_dev=None):
    n = x["mu"].numel()
    o = out or {k: torch.full((n,), float("nan"), device="cuda") for k in ("dmu", "drho", "dlam", "dgamma")}
    if out is None:
        o["dpb"] = torch.full((1,), float("nan"), device="cuda")
    ws = torch.empty(int(K.lib.lbbnn_mf_workspace_bytes(n)), dtype=torch.uint8, device="cuda")
    o["_keep"] = ws
    args = [K.ptr(x["mu"]), K.ptr(x["rho"]), K.ptr(x["lam"]), K.ptr(x["gamma"]), K.ptr(x["pb"]), n,
            _noise(K, x, native, step_dev), flags, K.ptr(x["dw"]) if use_dw else None, K.ptr(x["c"]) if use_c else None,
            K.ptr(o["dmu"]), K.ptr(o["drho"]), K.ptr(o["dlam"]), K.ptr(o["dgamma"]) if want_dgamma else None, K.ptr(o["dpb"]),
            ws.data_ptr(), ws.numel()]
    if ticket is None:
        K.check(K.lib.lbbnn_mf_sample_bwd(*args, K.current_stream()))
    else:
        K.check(K.lib.lbbnn_mf_sample_bwd_ticket(*args, ticket.data_ptr(), K.current_stream()))
    return o


def _ref(K, x, mode, flags, dtype, stale=True, eps=None, grad=False, use_dw=True, use_c=True):
    """The kernels' arithmetic restated in torch at `dtype`: (w, [s0..s4]) and, with grad, the derivatives of
    sum(dw w) + sum_k c_k s_k wrt mu, rho, lambda, gamma, pb."""
    v = {k: x[k].detach().to(dtype).clone().requires_grad_(grad and k in ("mu", "rho", "lam", "gamma", "pb"))
         for k in ("mu", "rho", "lam", "gamma", "alpha_stale", "pb")}
    e = (x["eps"] if eps is None else eps).to(dtype)
    sg = torch.log1p(torch.exp(v["rho"]))
    al = torch.sigmoid(v["lam"])
    ws = v["mu"] + sg * e if mode == K.MF_SAMPLE else v["mu"]
    g = v["gamma"] if mode != K.MF_JOINTMEAN else (v["alpha_stale"] if stale else al)
    w = g * ws
    wl = ws if flags & K.MF_FLAG_LP_ON_WS else w
    pick = lambda f: torch.round(g) if flags & f else g          # noqa: E731  (round: no gradient, like the kernels)
    g_b, g_wp, g_gp = pick(K.MF_FLAG_EXACT_GAMMA), pick(K.MF_FLAG_EXACT_WPRIOR), pick(K.MF_FLAG_EXACT_GPRIOR)
    pb = v["pb"]
    logn = -0.5 * math.log(2 * math.pi) - torch.log(sg) - (wl - v["mu"]) ** 2 / (2 * sg * sg)
    s = torch.stack([g_wp.sum(), (wl * wl).sum(), (torch.lgamma(1 + pb - g_gp) - torch.lgamma(2 - g_gp)).sum(),
                     torch.log(g * torch.exp(logn) + (1 - g) + 1e-8).sum(),
                     (g_b * torch.log(al + 1e-8) + (1 - g_b) * torch.log(1 - al + 1e-8)).sum()])
    if not grad:
        return w.detach(), s.detach()
    loss = 0
    if use_dw:
        loss = loss + (x["dw"].to(dtype) * w).sum()
    if use_c:
        loss = loss + (x["c"].to(dtype) * s).sum()
    gr = torch.autograd.grad(loss, [v[k] for k in ("mu", "rho", "lam", "gamma", "pb")], allow_unused=True)
    gr = [torch.zeros_like(v[k]) if t is None else t for t, k in zip(gr, ("mu", "rho", "lam", "gamma", "pb"))]
    return dict(zip(("dmu", "drho", "dlam", "dgamma", "dpb"), gr))


def _scalar_ok(got, r64, r32, floor=SUM_FLOOR):
    """Each entry within max(floor, 4 x the fp32 restatement's error) of the fp64 truth (relative to that entry)."""
    got, r64, r32 = (torch.as_tensor(t).double().cpu().reshape(-1) for t in (got, r64, r32))
    for k in range(r64.numel()):
        den = max(abs(r64[k].item()), 1e-30)
        e, e32 = abs(got[k].item() - r64[k].item()) / den, abs(r32[k].item() - r64[k].item()) / den
        if not e < max(floor, 4 * e32):
            return f"entry {k}: {got[k].item()!r} vs {r64[k].item()!r} (err {e:.2e}, fp32 torch {e32:.2e})"
    return None


def _check_fwd(K, o, x, mode, flags, stale=True, eps=None, what=""):
    w64, s64 = _ref(K, x, mode, flags, torch.float64, stale, eps)
    assert C.rel_err(o["w"], w64) < TOL, what
    if flags & K.MF_FLAG_LOGPROBS:
        _, s32 = _ref(K, x, mode, flags, torch.float32, stale, eps)
        bad = _scalar_ok(o["sums"], s64, s32)
        assert bad is None, f"{what}: sums {bad}"


def _check_bwd(K, o, x, flags, eps=None, what="", use_dw=True, use_c=True, want_dgamma=True):
    r64 = _ref(K, x, K.MF_SAMPLE, flags, torch.float64, eps=eps, grad=True, use_dw=use_dw, use_c=use_c)
    r32 = _ref(K, x, K.MF_SAMPLE, flags, torch.float32, eps=eps, grad=True, use_dw=use_dw, use_c=use_c)
    for k in ("dmu", "drho", "dlam") + (("dgamma",) if want_dgamma else ()):
        # 1e-5 unless fp32 itself cannot get there: at a single element with gamma close to alpha, d lambda is the
        # difference of two nearly equal terms
        assert C.rel_err(o[k], r64[k]) < max(TOL, 4 * C.rel_err(r32[k], r64[k])), f"{what}: {k}"
    bad = _scalar_ok(o["dpb"], r64["dpb"], r32["dpb"])
    assert bad is None, f"{what}: dpb {bad}"


@pytest.mark.parametrize("n", [1, 3, 5, 1023, 4096, "big"])
def test_mf_sample_every_mode_and_flag_matches_fp64(n):
    K = _capi()
    n = _size(n)
    x = _inputs(n, seed=n % 100003)
    modes = [(K.MF_SAMPLE, True), (K.MF_MEDIMEAN, True), (K.MF_JOINTMEAN, True), (K.MF_JOINTMEAN, False)]
    for mode, stale in modes:
        for flags in [0] + _flags(K):
            o = _fwd(K, x, mode, flags, stale=stale)
            _check_fwd(K, o, x, mode, flags, stale, what=f"n={n} mode={mode} stale={stale} flags={flags}")
    for flags in _flags(K):
        o = _bwd(K, x, flags)
        _check_bwd(K, o, x, flags, what=f"n={n} bwd flags={flags}")
    # absent dL/dw, absent dL/dsums (dpb = 0), no dgamma wanted
    for use_dw, use_c, want_dg in ((False, True, True), (True, False, True), (True, True, False)):
        o = _bwd(K, x, K.MF_FLAG_LOGPROBS, use_dw=use_dw, use_c=use_c, want_dgamma=want_dg)
        _check_bwd(K, o, x, K.MF_FLAG_LOGPROBS, what=f"n={n} dw={use_dw} c={use_c} dgamma={want_dg}", use_dw=use_dw,
                   use_c=use_c, want_dgamma=want_dg)
        if not want_dg:
            assert torch.isnan(o["dgamma"]).all()        # not written
        if not use_c:
            assert o["dpb"].item() == 0.0


def test_mf_sample_unaligned_operands_match_aligned():
    """n % 4 == 0, every operand one float off a 16-byte boundary: the scalar-load path, same results bit for bit."""
    K = _capi()
    n = 4096
    a, u = _inputs(n, seed=11), _inputs(n, seed=11, offset=1)
    assert u["mu"].data_ptr() % 16 != 0 and u["mu"].is_contiguous()
    for flags in (K.MF_FLAG_LOGPROBS, _flags(K)[-1]):
        for mode in (K.MF_SAMPLE, K.MF_JOINTMEAN):
            oa, ou = _fwd(K, a, mode, flags), _fwd(K, u, mode, flags)
            assert torch.equal(oa["w"], ou["w"]) and torch.equal(oa["sums"], ou["sums"])
            _check_fwd(K, ou, u, mode, flags, what=f"unaligned mode={mode} flags={flags}")
        ba, bu = _bwd(K, a, flags), _bwd(K, u, flags)
        for k in ("dmu", "drho", "dlam", "dgamma", "dpb"):
            assert torch.equal(ba[k], bu[k]), k
        _check_bwd(K, bu, u, flags, what=f"unaligned bwd flags={flags}")


# ---- per-thread widths (LBBNN_MF_SPLIT) ----------------------------------------------------------------------------------
WIDTH_CASES = [(n, fi, native) for n in (5, 1023, "big") for fi in (0, 7, 15) for native in (False, True)]
WIDTH_KEYS = ("w", "sums", "dmu", "drho", "dlam", "dgamma", "dpb")


def _width_results():
    """Every WIDTH_CASES forward and backward with this process's width: {f"{case}_{key}": array}."""
    K = _capi()
    res = {}
    for i, (n, fi, native) in enumerate(WIDTH_CASES):
        n = _size(n)
        x = _inputs(n, seed=100 + i)
        flags = _flags(K)[fi]
        o = _fwd(K, x, K.MF_SAMPLE, flags, native=native)
        o.update(_bwd(K, x, flags, native=native))
        for k in WIDTH_KEYS:
            res[f"{i}_{k}"] = o[k].cpu().numpy()
    torch.cuda.synchronize()
    return res


def _width_run(width, tmp_path):
    if width == int(os.environ.get("LBBNN_MF_SPLIT", "2")):
        return _width_results()
    out = os.path.join(str(tmp_path), f"width{width}.npz")
    env = dict(os.environ, LBBNN_MF_SPLIT=str(width))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), out], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    with np.load(out) as z:
        return dict(z)


def test_mf_sample_widths_1_and_4_bit_identical_to_2(tmp_path):
    """Widths 1 and 4 (two and four threads share a Philox group / one thread takes a whole group) against the default 2:
    the elementwise results bit for bit, with injected and native eps; every width's sums and dpb against the fp64 truth."""
    K = _capi()
    base = _width_run(2, tmp_path)
    got = {w: _width_run(w, tmp_path) for w in (1, 4)}
    for i, (n, fi, native) in enumerate(WIDTH_CASES):
        n = _size(n)
        flags = _flags(K)[fi]
        x = _inputs(n, seed=100 + i)
        eps = _native_eps(n) if native else None
        what = f"case {i} (n={n}, flags={flags}, native eps={native})"
        o = {k: torch.from_numpy(base[f"{i}_{k}"]) for k in WIDTH_KEYS}
        _check_fwd(K, o, x, K.MF_SAMPLE, flags, eps=eps, what=what)
        _check_bwd(K, o, x, flags, eps=eps, what=what)
        _, s64 = _ref(K, x, K.MF_SAMPLE, flags, torch.float64, eps=eps)
        _, s32 = _ref(K, x, K.MF_SAMPLE, flags, torch.float32, eps=eps)
        p64 = _ref(K, x, K.MF_SAMPLE, flags, torch.float64, eps=eps, grad=True)["dpb"]
        p32 = _ref(K, x, K.MF_SAMPLE, flags, torch.float32, eps=eps, grad=True)["dpb"]
        for w, r in got.items():
            for k in ("w", "dmu", "drho", "dlam", "dgamma"):
                assert np.array_equal(r[f"{i}_{k}"], base[f"{i}_{k}"]), f"width {w}, {what}: {k}"
            bad = _scalar_ok(r[f"{i}_sums"], s64, s32) or _scalar_ok(r[f"{i}_dpb"], p64, p32)
            assert bad is None, f"width {w}, {what}: sums / dpb {bad}"


# ---- ticket entry points -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [5, 4096, "big"])
def test_mf_ticket_paths_equal_two_launch_paths_and_leave_ticket_zero(n):
    K = _capi()
    n = _size(n)
    x = _inputs(n, seed=23)
    tk = torch.zeros(2, dtype=torch.int32, device="cuda")
    for flags in (K.MF_FLAG_LOGPROBS, _flags(K)[-1], _flags(K)[5]):
        for native in (False, True):
            a, b = _fwd(K, x, K.MF_SAMPLE, flags, native=native), _fwd(K, x, K.MF_SAMPLE, flags, native=native, ticket=tk[0:1])
            assert torch.equal(a["w"], b["w"]) and torch.equal(a["sums"], b["sums"]), (flags, native)
            a, b = _bwd(K, x, flags, native=native), _bwd(K, x, flags, native=native, ticket=tk[1:2])
            for k in ("dmu", "drho", "dlam", "dgamma", "dpb"):
                assert torch.equal(a[k], b[k]), (flags, native, k)
            assert tk.tolist() == [0, 0]
    # captured once, replayed three times: same results, tickets back at zero
    flags = _flags(K)[-1]
    eager_f, eager_b = _fwd(K, x, K.MF_SAMPLE, flags), _bwd(K, x, flags)
    of = {"w": torch.empty(n, device="cuda"), "sums": torch.empty(5, device="cuda")}
    ob = {k: torch.empty(n, device="cuda") for k in ("dmu", "drho", "dlam", "dgamma")}
    ob["dpb"] = torch.empty(1, device="cuda")
    _fwd(K, x, K.MF_SAMPLE, flags, ticket=tk[0:1], out=of)          # warm-up outside the capture
    _bwd(K, x, flags, ticket=tk[1:2], out=ob)
    torch.cuda.synchronize()
    graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(graph, stream=side):
        _fwd(K, x, K.MF_SAMPLE, flags, ticket=tk[0:1], out=of)
        _bwd(K, x, flags, ticket=tk[1:2], out=ob)
    for t in list(of.values()) + list(ob.values()):
        if t.dtype == torch.float32:
            t.fill_(float("nan"))
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    assert tk.tolist() == [0, 0]
    assert torch.equal(of["w"], eager_f["w"]) and torch.equal(of["sums"], eager_f["sums"])
    for k in ("dmu", "drho", "dlam", "dgamma", "dpb"):
        assert torch.equal(ob[k], eager_b[k]), k


# ---- native draws ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1, 1), (3, 5), (7, 13), (37, 1001)])
@pytest.mark.parametrize("step", [None, 5])
def test_mf_native_draws_equal_exported_philox(shape, step):
    """lbbnn_mf_sample_predict (hard mask [u < alpha], weights and bias drawn in one launch) and the sampler's native eps at
    odd sizes (the last Philox group of four is partial), with and without a device step counter: the oracle evaluated on
    lbbnn.philox_uniform / philox_normal of the same streams."""
    from lbbnn import philox_normal, philox_uniform
    K = _capi()
    o_, i_ = shape
    n = o_ * i_
    rng = np.random.default_rng(n)
    f32 = lambda a: C.t(a).cuda()      # noqa: E731
    mu, rho, lam = f32(rng.uniform(-0.2, 0.2, (o_, i_))), f32(rng.uniform(-5, -2, (o_, i_))), f32(rng.normal(0, 2, (o_, i_)))
    bmu, brho = f32(rng.uniform(-0.2, 0.2, o_)), f32(rng.uniform(-5, -2, o_))
    step_dev = torch.tensor([step], dtype=torch.int64, device="cuda") if step is not None else None
    eff = lambda s: (s + (step or 0) * GRAPH_STRIDE) % 2 ** 64     # noqa: E731
    nz = [K.make_noise(None, SEED, STREAM + k, step_dev, GRAPH_STRIDE if step is not None else 0) for k in range(3)]
    w, bias = torch.empty(o_, i_, device="cuda"), torch.empty(o_, device="cuda")
    K.check(K.lib.lbbnn_mf_sample_predict(K.make_layer(mu, rho, lam, bmu, brho), nz[0], nz[1], nz[2], K.ptr(w), K.ptr(bias),
                                          K.current_stream()))
    u = philox_uniform((o_, i_), SEED, eff(STREAM))
    ew, eb = philox_normal((o_, i_), SEED, eff(STREAM + 1)), philox_normal(o_, SEED, eff(STREAM + 2))
    mask = u < 1.0 / (1.0 + torch.exp(-lam))          # fp32 alpha, fp32 uniform: the comparison the kernel makes
    assert torch.equal(w != 0, mask)
    d = lambda t: t.double()      # noqa: E731
    assert C.rel_err(w, mask.double() * (d(mu) + torch.log1p(torch.exp(d(rho))) * d(ew))) < TOL
    assert C.rel_err(bias, d(bmu) + torch.log1p(torch.exp(d(brho))) * d(eb)) < TOL
    # the log-probability sampler with native eps, forward and backward
    x = _inputs(n, seed=n + 1)
    eps = _native_eps(n, step or 0)
    flags = _flags(K)[3]
    _check_fwd(K, _fwd(K, x, K.MF_SAMPLE, flags, native=True, step_dev=step_dev), x, K.MF_SAMPLE, flags, eps=eps,
               what="native eps")
    _check_bwd(K, _bwd(K, x, flags, native=True, step_dev=step_dev), x, flags, eps=eps, what="native eps")


# ---- prior kernels -------------------------------------------------------------------------------------------------------
PRIOR_SCALARS = ("s", "a", "b", "tau_w", "pa", "pb")
PRIOR_VECTORS = ("ba", "bb", "tau_b", "bias_mu", "bias_rho")


def _prior_ref(p, sample, eps, n, g, dtype, factors):
    """The comment above PriorArgs in csrc/mf.cu, in torch at `dtype`: (bias, log_prior, log_q) and the derivatives of
    g_lp log_prior + g_lq log_q + sum(g_bias bias); with factors, tau_w and tau_b are functions of (a, b) / (ba, bb) through
    the given partial derivatives."""
    v = {k: p[k].to(dtype).clone().requires_grad_(True) for k in PRIOR_SCALARS + PRIOR_VECTORS}
    l2pi = 0.5 * math.log(2 * math.pi)
    s, a, b, tw, pa, pb = (v[k] for k in PRIOR_SCALARS)
    ba, bb, tb, mu, rho = (v[k] for k in PRIOR_VECTORS)
    sb = torch.log1p(torch.exp(rho))
    bias = mu + sb * eps.to(dtype) if sample else mu
    cw = a * torch.log(b) + (a - 0.5) * tw - b * tw - torch.lgamma(a) - l2pi
    lp = (s[0] * cw - tw * s[1] + (n - s[0]) + n * 1e-8
          + (ba * torch.log(bb) + (ba - 0.5) * tb - bb * tb - torch.lgamma(ba) - l2pi - tb * bias ** 2 + 1e-8).sum()
          + s[2] + n * (torch.lgamma(pa + pb) - torch.lgamma(1 + pa + pb) - torch.lgamma(pa) - torch.lgamma(pb)))
    lq = s[3] + s[4] + (-l2pi - torch.log(sb) - (bias - mu) ** 2 / (2 * sb ** 2)).sum()
    loss = (g["lp"].to(dtype) * lp).sum() + (g["lq"].to(dtype) * lq).sum() + (g["bias"].to(dtype) * bias).sum()
    gr = dict(zip(PRIOR_SCALARS + PRIOR_VECTORS, torch.autograd.grad(loss, [v[k] for k in PRIOR_SCALARS + PRIOR_VECTORS])))
    if factors is not None:
        gr["a"] = gr["a"] + gr["tau_w"] * factors["tw_da"].to(dtype)
        gr["b"] = gr["b"] + gr["tau_w"] * factors["tw_db"].to(dtype)
        gr["ba"] = gr["ba"] + gr["tau_b"] * factors["tb_da"].to(dtype)
        gr["bb"] = gr["bb"] + gr["tau_b"] * factors["tb_db"].to(dtype)
    d10 = torch.cat([gr["s"], gr["a"], gr["b"], gr["tau_w"], gr["pa"], gr["pb"]])
    return bias.detach(), torch.stack([lp.sum(), lq.sum()]).detach(), d10.detach(), {k: gr[k] for k in PRIOR_VECTORS}


@pytest.mark.parametrize("out", [1, 257, 1000])
@pytest.mark.parametrize("with_factors", [False, True])
def test_mf_prior_kernels_match_fp64(out, with_factors):
    """lbbnn_mf_prior_fwd / lbbnn_mf_prior_bwd_tau (one block of 256 threads; out > 256 loops) for the posterior-mean bias,
    an injected and a native bias draw."""
    K = _capi()
    rng = np.random.default_rng(out + 7 * with_factors)
    f32 = lambda a: C.t(np.asarray(a, dtype=np.float64).reshape(-1)).cuda()     # noqa: E731
    n = 7.0 * out * 113
    p = {"s": f32([0.6 * n, 0.02 * n, -0.03 * n, 1.5 * n, -0.7 * n]), "a": f32(rng.uniform(1, 1.1, 1)),
         "b": f32(rng.uniform(1, 1.1, 1)), "tau_w": f32(rng.gamma(1.05, size=1)), "pa": f32(rng.uniform(1, 1.1, 1)),
         "pb": f32([0.05]), "ba": f32(rng.uniform(1, 1.1, out)), "bb": f32(rng.uniform(1, 1.1, out)),
         "tau_b": f32(rng.gamma(1.05, size=out)), "bias_mu": f32(rng.uniform(-0.2, 0.2, out)),
         "bias_rho": f32(rng.uniform(-5, -2, out))}
    g = {"lp": f32(rng.standard_normal(1)), "lq": f32(rng.standard_normal(1)), "bias": f32(rng.standard_normal(out))}
    factors = ({"tw_da": f32(rng.standard_normal(1)), "tw_db": f32(rng.standard_normal(1)),
                "tb_da": f32(rng.standard_normal(out)), "tb_db": f32(rng.standard_normal(out))} if with_factors else None)
    eps_inj = f32(rng.standard_normal(out))
    for sample, native in ((0, False), (1, False), (1, True)):
        what = f"out={out} sample={sample} native={native} factors={with_factors}"
        noise = K.make_noise(None, SEED, STREAM) if native else K.make_noise(eps_inj)
        eps = (_native_eps(out) if native else eps_inj) if sample else torch.zeros(out, device="cuda")
        bias, eps_out, lp = (torch.full((k,), float("nan"), device="cuda") for k in (out, out, 2))
        ts = [p[k] for k in ("s", "a", "b", "tau_w", "pa", "pb", "ba", "bb", "tau_b", "bias_mu", "bias_rho")]
        K.check(K.lib.lbbnn_mf_prior_fwd(*[K.ptr(t) for t in ts], noise, sample, out, n, K.ptr(bias), K.ptr(eps_out), K.ptr(lp),
                                         K.current_stream()))
        d10 = torch.full((10,), float("nan"), device="cuda")
        dv = {k: torch.full((out,), float("nan"), device="cuda") for k in PRIOR_VECTORS}
        fp = [K.ptr(factors[k]) if factors else None for k in ("tw_da", "tw_db", "tb_da", "tb_db")]
        K.check(K.lib.lbbnn_mf_prior_bwd_tau(*[K.ptr(t) for t in ts], K.ptr(bias), K.ptr(eps_out), sample, out, n,
                                             K.ptr(g["lp"]), K.ptr(g["lq"]), K.ptr(g["bias"]), *fp, K.ptr(d10),
                                             *[K.ptr(dv[k]) for k in PRIOR_VECTORS], K.current_stream()))
        assert torch.equal(eps_out, eps), what          # the draw the backward uses; zero for the posterior-mean bias
        b64, lp64, d64, v64 = _prior_ref(p, sample, eps, n, g, torch.float64, factors)
        b32, lp32, d32, v32 = _prior_ref(p, sample, eps, n, g, torch.float32, factors)
        assert C.rel_err(bias, b64) < TOL, what
        bad = _scalar_ok(lp, lp64, lp32)
        assert bad is None, f"{what}: log_prior / log_q {bad}"
        bad = _scalar_ok(d10, d64, d32)
        assert bad is None, f"{what}: d_scalars {bad}"
        for k in PRIOR_VECTORS:
            assert C.rel_err(dv[k], v64[k]) < max(TOL, 4 * C.rel_err(v32[k], v64[k])), f"{what}: d_{k}"


if __name__ == "__main__":
    np.savez(sys.argv[1], **_width_results())
