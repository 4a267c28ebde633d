"""The fp32 LRT layer kernels (csrc/lrt_f32.cu) and the MNF auxiliary kernels (csrc/mnf_aux.cu) through the C-ABI, each
against a float64 restatement of what it computes, on the GPU, from the same fp32 inputs and the same noise:
  lrt_f32_fwd / _fwd_ex   prologue + split-K dual GEMM + epilogue: act, ds_factor (or e_b, var_b), KL, the M / V cache
  lrt_f32_prologue        M = alpha mu z, V, and the KL (lrt_kl_finalize) of the weights with mu z_kl and of the biases
  lrt_kl_finalize         fixed-order sum of KL partials + the bias term
  lrt_f32_bwd_params      dW GEMM + finalize: the five parameter gradients and the MNF z gradients (dz, dz_kl)
  lrt_f32_bwd_input       split-N dx GEMM + epilogue (relu mask, accumulate)
  lrt_f32_finalize        the chain rule from (dM, dV, colsum) alone: the ZRED and the elementwise launch
  lrt_f32_finalize_adam / _finalize_adam_bias   the same gradients consumed by torch.optim.Adam's update
  mnf_aux_kl_fwd / _bwd   log q0 - log r_b and all its gradients; mnf_draw / _draw_bwd; mnf_bwd_rows; mnf_kl_combine
The float64 references are lbbnn_oracle's pieces (lrt_weight_moments, lrt_kl, mnf_forward) and float64 torch autograd.
Bounds (cases.rel_err = max|a-b| / max|b|): 1e-5 on activations, dx, KL and every gradient; 2e-6 on the Adam results
(parameters and both moments; the reference runs on the fp32 values of lr, betas and eps).  Bit-exact: native noise
against the exported Philox stream, and repeated launches -- except the four outputs reduced with atomics (dz, dz_kl,
d_r0_c, d_z2), whose summation order changes from launch to launch: those are held to the float64 bound instead.

The launch rules and configuration tables above the tests are plain Python: tests/test_layer_kernels_cpu.py checks, without
a GPU, that the tables still reach every launch path at 148 SMs."""
import ctypes
import math
import zlib

import numpy as np
import pytest
import torch

import cases as C
import lbbnn_oracle as O

pytestmark = pytest.mark.gpu
TOL, TOL_ADAM = 1e-5, 2e-6
# The Adam step itself (p after the updates minus p before), relative to its largest element: a parameter check relative to
# max|p| (about 8 for lambdal) lets through an error of 1% of a 2e-3 step.  What the step cannot be held below is the fp32
# rounding of the stored parameter, half an ulp of |p| <= 8 per update: 2.4e-4 of the two steps' 4e-3.
TOL_ADAM_STEP = 1e-3
SEED, STREAM = 9876, 21
SMS = 148


def cdiv(a, b):
    return -(-a // b)


# ---- launch rules, restated from the host code ---------------------------------------------------------------------------
F_BM, F_BN, F_BK = 128, 64, 16          # forward tiles, K chunk
X_BM, X_BK, X_BN = 128, 64, 16          # dx tiles, N chunk
W_BN, W_BK, W_BB = 32, 64, 16           # dW tiles, batch step
Z_ROWS, Z_QUADS = 16, 32                # ZRED block: 16 weight rows x 32 column quads
EPI_BATCH = 8                           # forward epilogue: splits read per pass


def pick_split(tiles, chunks, sms=SMS):
    """(chunks per split, splits): enough splits for about one CTA per SM, at least two chunks per split."""
    want = 1 if tiles >= sms else cdiv(sms, tiles)
    want = max(1, min(want, chunks // 2))
    cps = cdiv(chunks, want)
    return cps, max(1, cdiv(chunks, cps))


def fwd_split(B, K, N, sms=SMS):
    return pick_split(cdiv(B, F_BM) * cdiv(N, F_BN), cdiv(K, F_BK), sms)


def dx_split(B, K, N, sms=SMS):
    return pick_split(cdiv(B, X_BM) * cdiv(K, X_BK), cdiv(N, X_BN), sms)


def elementwise_blocks(n, sms=SMS):
    """Blocks of 256 threads, one quad each, capped at 16 per SM (a grid-stride loop beyond)."""
    return max(1, min(cdiv(cdiv(n, 4), 256), 16 * sms))


def finalize_launch(K, N, dz_requested):
    """("zred", blocks) for the patch-shaped launch that reduces the z gradients per block, else ("elem", blocks)."""
    if dz_requested and K % 4 == 0:
        return "zred", cdiv(K // 4, Z_QUADS) * cdiv(N, Z_ROWS)
    return "elem", elementwise_blocks(N * K)


def aux_slices(D, O_, sms=SMS, forced=None):
    """Row slices of mnf_aux_kl_bwd: about two blocks per SM, at least one 64-row pass per slice; LBBNN_AUX_SLICES wins."""
    if forced is not None:
        return max(1, forced)
    s = 2 * sms // cdiv(D, 32)
    return max(1, min(s, cdiv(O_, 64)))


PRIORS = {"default": (0.0, 1.0, 0.05, 0.0, 1.0), "sim": (0.1, 1.3, 0.3, 0.0, 1.3)}     # MNFsim:157-174
NAMES = ("weight_mu", "weight_rho", "lambdal", "bias_mu", "bias_rho")


# ---- configuration tables ------------------------------------------------------------------------------------------------
def _f(B, K, N, **kw):
    c = dict(B=B, K=K, N=N, sample=True, relu=False, kl=False, moments=False, mv=False, noise="inj", off=0, rpg=0,
             rowscale=False, rs_off=0, gstride=0, z="none", var="reference", pri="default")
    c.update(kw)
    return c


FWD_CASES = [
    _f(1024, 100, 1216, relu=True),                            # 152 tiles fill the GPU: 1 split
    _f(8, 47, 10, kl=True),                                    # 3 chunks (ragged last): the chunk cap gives 1 split
    _f(8, 20, 10, relu=True, mv=True),                         # 2 chunks: 1 split
    *[_f(9, 32 * s, 10, kl=s % 2 == 0) for s in range(2, 9)],  # 2 .. 8 splits of 2 chunks
    _f(100, 784, 400, kl=True, mv=True),                       # 17 splits: the epilogue's third pass reads one
    _f(100, 400, 10, relu=True),                               # 9 splits
    _f(100, 400, 10, noise="nat", off=1),                      # 9 splits, scalar loads and stores
    _f(7, 4096, 3, kl=True),                                   # 128 splits
    _f(5, 80, 7),                                              # 5 chunks: 2 splits of 3 and 2
    _f(130, 100, 70, kl=True, noise="nat"),                    # 7 chunks (ragged chunk), splits of 3 / 3 / 1; B, N ragged
    _f(200, 64, 130, off=1, mv=True),                          # K % 4 == 0 at +1 float: scalar loads, scalar epilogue
    _f(200, 64, 130, off=0, mv=True, relu=True),               # the same aligned: vector loads
    _f(33, 50, 9, sample=False, relu=True),                    # mean branch, K % 4 != 0
    _f(33, 64, 12, sample=False, mv=True, kl=True, off=1),     # mean branch: only M cached
    _f(8, 2048, 1216, kl=True),                                # 2.49 M weights: the KL partial count is capped
    _f(40, 100, 24, moments=True, kl=True),                    # e_b and var_b
    _f(40, 100, 24, moments=True, mv=True, off=1),
    _f(64, 200, 36, noise="nat", mv=True),
    _f(10, 64, 6, noise="nat", rpg=4, gstride=1000003),        # 3 noise groups of 4 rows, the last ragged (2 rows)
    _f(12, 64, 6, noise="nat", rpg=4, gstride=77, rowscale=True),
    _f(10, 64, 6, rpg=4, rowscale=True),                       # row scale: groups of 4, last ragged, aligned
    _f(10, 64, 6, rpg=4, rowscale=True, rs_off=1),             # misaligned row scale
    _f(131, 100, 17, rpg=50, rowscale=True, rs_off=1, relu=True),
    _f(300, 784, 20, rpg=100, rowscale=True, noise="nat", gstride=5, z="z"),
    _f(37, 100, 17, z="z", kl=True, mv=True),                  # MNF: M = alpha mu z, KL with mu z
    _f(37, 100, 17, z="zkl", kl=True, var="exact", pri="sim"), # MNF: KL with its own z_kl, exact variance, MNFsim priors
    _f(16, 33, 7, z="zkl", kl=True, pri="sim", off=1),
    _f(16, 784, 400, z="z", kl=True, var="exact", pri="sim", noise="nat"),
]

PRO_CASES = [   # (K, N, z, var, pri, sample) through lbbnn_lrt_f32_prologue with kl_out
    (50, 13, "none", "reference", "default", True),
    (33, 7, "z", "exact", "sim", True),
    (784, 400, "klonly", "reference", "sim", True),       # the KL branch's call: M0 without z, KL with mu z_kl
    (100, 17, "zkl", "exact", "default", False),          # mean branch: no V
    (2048, 1216, "none", "exact", "sim", True),           # partial count capped at 16 x 148
]


def _bw(B, K, N, **kw):
    c = dict(B=B, K=K, N=N, sample=True, z="none", req="none", klg="host", acc=False, off=0, var="reference", pri="default")
    c.update(kw)
    return c


BWDW_CASES = [   # lbbnn_lrt_f32_bwd_params: dW GEMM (32 x 64 tiles, 16-row batch steps) + finalize
    _bw(37, 100, 45),                                          # B % 16, N % 32, K % 64 all ragged; vector loads
    _bw(37, 100, 45, off=1),                                   # the same at +1 float: scalar loads
    _bw(32, 128, 64, klg="dev", var="exact"),                  # whole tiles
    _bw(1, 33, 7, z="z", req="dz"),                            # elementwise z gradients (K % 4 != 0)
    _bw(130, 72, 17, z="zkl", req="both", klg="dev", pri="sim"),   # ZRED, ragged column and row blocks
    _bw(64, 784, 400, z="z", req="dz", var="exact", pri="sim"),
    _bw(50, 64, 20, z="zkl", req="dzkl", acc=True),
    _bw(50, 64, 20, z="zkl", req="dz", klg="0"),
    _bw(20, 50, 30, sample=False, acc=True),                   # sample off: no dV
    _bw(20, 64, 36, sample=False, z="z", req="dz", off=1),
    _bw(300, 200, 70, acc=True, klg="0"),
]


def _dx(B, K, N, **kw):
    c = dict(B=B, K=K, N=N, sample=True, mv=False, mask=False, acc=False, off=0, z="none", var="reference")
    c.update(kw)
    return c


DX_CASES = [   # lbbnn_lrt_f32_bwd_input: split-N dx GEMM (128 x 64 tiles, 16-wide N chunks) + epilogue
    _dx(1024, 1216, 40, mask=True),                            # 152 tiles fill the GPU: 1 split
    _dx(100, 200, 31, mv=True),                                # 2 chunks: 1 split
    _dx(100, 64, 288, mask=True, acc=True),                    # 9 splits of 2
    _dx(100, 50, 544, var="exact"),                            # 17 splits: the epilogue's second pass reads one
    _dx(70, 100, 300, mv=True, z="z"),                         # 19 chunks: 7 splits, the last of 1
    _dx(70, 100, 300, off=1, mask=True),                       # scalar loads and stores
    _dx(45, 33, 17, sample=False, acc=True, mv=True),
    _dx(45, 36, 17, sample=False, mask=True, off=1, z="zkl"),
]


def _fin(K, N, z, req, klg="host", **kw):
    c = dict(K=K, N=N, z=z, req=req, klg=klg, acc=False, sample=True, var="reference", pri="default", off=0)
    c.update(kw)
    return c


FIN_CASES = [   # lbbnn_lrt_f32_finalize from random (dM, dV, colsum)
    _fin(100, 17, "z", "dz"),                                  # ZRED: 25 quads (ragged column block), 17 rows (ragged row block)
    _fin(784, 40, "zkl", "both", "dev", var="exact", pri="sim"),   # 7 column blocks, the last of 4 quads
    _fin(128, 32, "zkl", "dzkl"),                              # whole blocks
    _fin(128, 33, "zkl", "dz", acc=True),                      # z_kl present, only dz requested: both shares into dz
    _fin(100, 17, "klonly", "dzkl", "dev"),                    # the KL branch's layer (z_kl only)
    _fin(100, 17, "z", "dz", off=1, acc=True),                 # ZRED with scalar loads / stores
    _fin(33, 7, "z", "dz"),                                    # elementwise: quads straddle weight rows
    _fin(50, 13, "zkl", "both", "dev", var="exact"),
    _fin(50, 13, "zkl", "dzkl", pri="sim"),
    _fin(50, 13, "zkl", "dz", "0"),
    _fin(100, 17, "z", "none"),                                # the layer has z, nothing requested: elementwise
    _fin(64, 10, "none", "none", "0", acc=True),
    _fin(64, 10, "none", "none", "dev", acc=True, sample=False),
    _fin(37, 9, "none", "none", sample=False, off=1, var="exact"),
    _fin(2048, 1300, "none", "none", pri="sim"),               # 665600 quads: the grid-stride loop
]

ADAM_CASES = [   # (K, N, var, sample, klg)
    (100, 64, "reference", True, "dev"),
    (50, 13, "exact", True, "host"),
    (33, 7, "reference", False, "0"),
]

AUX_FWD_CASES = [(20, 5), (33, 13), (256, 8), (300, 700), (784, 400), (1000, 3)]     # (D, O)
AUX_BWD_CASES = [   # (D, O, LBBNN_AUX_SLICES or None)
    (784, 400, None), (300, 700, None), (33, 13, None), (20, 5, None), (256, 200, None),
    (784, 400, 1), (300, 700, 3), (33, 13, 3), (20, 5, 16), (100, 70, 128),
]
DRAW_CASES = [(1, 50, 13, "inj", True), (3, 50, 13, "nat", True), (3, 37, 0, "nat", False), (1, 784, 400, "nat", True),
              (3, 33, 7, "inj", False)]                                              # (R, D, O, noise, eps_r)
DRAW_BWD_CASES = [(1, 50, -1, False), (1, 50, 0, True), (3, 37, 0, True), (3, 37, 2, True), (3, 37, 2, False),
                  (2, 784, 1, True), (3, 300, -1, True)]                             # (R, D, kl_row, aux terms)
ROWS_CASES = [("dld",), ("rows",), ("dld", "rows"), ("rows", "no_a"), ("rows", "no_b"), ("rows", "no_dzk"),
              ("dld", "rows", "no_a", "no_b", "no_dzk")]
ROWS_D = (1, 37, 300)
MNF_SWEEP = [(1, 33, 7, "default"), (130, 72, 17, "default"), (16, 784, 400, "sim")]


def _id(c):
    return "-".join(f"{k}{v}" for k, v in c.items()
                    if v not in (False, 0, "none", "inj", "reference", "default") and (k, v) != ("sample", True))


# ---- helpers --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def K():
    from lbbnn import _capi
    _capi.require_device()
    return _capi


def _report(name, **kv):
    print(f"[layer-kernels] {name}: " + ", ".join(f"{k} {v:.3e}" for k, v in kv.items()), flush=True)


def _rng(c):
    return np.random.default_rng(zlib.crc32(repr(c).encode()))


def _u(rng, lo, hi, *shape):
    return torch.from_numpy(rng.uniform(lo, hi, size=shape)).float().cuda()


def _n(rng, *shape, scale=1.0):
    return torch.from_numpy(scale * rng.standard_normal(size=shape)).float().cuda()


def _at(t, off=0, fill=float("nan")):
    """A copy of t (or a buffer of t's shape if t is a tuple) starting `off` floats into its storage."""
    shape = t if isinstance(t, tuple) else tuple(t.shape)
    b = torch.full((math.prod(shape) + off,), fill, device="cuda")[off:].view(shape)
    if not isinstance(t, tuple):
        b.copy_(t)
    return b


def _params(rng, K, N):
    return {"weight_mu": _u(rng, -0.3, 0.3, N, K), "weight_rho": _u(rng, -4.0, -1.0, N, K), "lambdal": _n(rng, N, K, scale=2.0),
            "bias_mu": _u(rng, -0.2, 0.2, N), "bias_rho": _u(rng, -4.0, -1.0, N)}


def _zs(rng, kind, K):
    """(z, z_kl) of a layer: none, z only (its KL uses z), z and a separate z_kl, or z_kl only (the KL branch)."""
    z = _u(rng, 0.5, 1.5, K) if kind in ("z", "zkl") else None
    zkl = _u(rng, 0.5, 1.5, K) if kind in ("zkl", "klonly") else None
    return z, zkl


def _layer(K, p, z=None, zkl=None):
    return K.make_layer(*[p[k] for k in NAMES], z=z, z_kl=zkl)


def _ws(K, B, Kf, N):
    return torch.full((K.lrt_workspace_bytes(B, Kf, N),), 0xFF, dtype=torch.uint8, device="cuda")   # NaN everywhere


def _d(t):
    return None if t is None else t.double()


def _moments(p, var, z=None):
    M, V = O.lrt_weight_moments(p["weight_mu"], p["weight_rho"], p["lambdal"], var)
    return (M if z is None else M * z), V


def _priors(K, name):
    return K.Priors(*PRIORS[name]), O.Priors(*PRIORS[name])


def _klg(K, kind):
    """(device tensor or None, host scalar, the fp32 product the kernel applies)."""
    if kind == "0":
        return None, 0.0, 0.0
    if kind == "host":
        return None, 0.37, float(np.float32(0.37))
    return torch.tensor([0.25], device="cuda"), 3.0, float(np.float32(0.25) * np.float32(3.0))


def ref_param_grads(p32, z32, zkl32, dM, dV, cs, klg, var, pri, sample):
    """float64 gradients of  <dM, alpha mu z> + <dV, V> + <colsum, (b_mu, sigma_b^2)> + klg KL(mu z_kl)  -- the chain rule
    lbbnn_lrt_f32_finalize applies to (dM, dV, colsum).  z_kl absent: the KL uses z, so z's gradient holds both shares."""
    p = {k: v.double().requires_grad_(True) for k, v in p32.items()}
    z = None if z32 is None else z32.double().requires_grad_(True)
    zkl = None if zkl32 is None else zkl32.double().requires_grad_(True)
    N = p["bias_mu"].numel()
    M, V = _moments(p, var, z)
    L = (dM.double() * M).sum() + (cs[:N].double() * p["bias_mu"]).sum()
    if sample:
        L = L + (dV.double() * V).sum() + (cs[N:].double() * O.sigma_of(p["bias_rho"]) ** 2).sum()
    if klg != 0.0:
        L = L + klg * O.lrt_kl(p, pri, z=zkl if zkl is not None else z)
    ins = [*p.values()] + [t for t in (z, zkl) if t is not None]
    gs = torch.autograd.grad(L, ins, allow_unused=True)
    gs = [torch.zeros_like(t) if g is None else g for g, t in zip(gs, ins)]
    out = dict(zip(NAMES, gs[:5]))
    rest = gs[5:]
    out["z"] = rest.pop(0) if z is not None else None
    out["z_kl"] = rest.pop(0) if zkl is not None else None
    return out


def _expected_dz(req, ref):
    """What the z-gradient buffers receive: dz_kl the KL share; dz the activation share, plus the KL share when dz_kl is not
    requested."""
    dz = dzkl = None
    if req in ("dz", "both"):
        dz = ref["z"] + (ref["z_kl"] if req == "dz" and ref["z_kl"] is not None else 0.0)
    if req in ("dzkl", "both"):
        dzkl = ref["z_kl"]
    return dz, dzkl


def _grad_bufs(rng, p, off, acc):
    """Gradient outputs: NaN, or random values to accumulate onto."""
    return {k: _at(_n(rng, *v.shape) if acc else tuple(v.shape), off) for k, v in p.items()}


def _check(name, got, ref, tol=TOL):
    e = C.rel_err(got, ref)
    assert e < tol, f"{name}: rel err {e:.3e}"
    return e


# ---- 1) forward ----------------------------------------------------------------------------------------------------------
def _philox_rows(K, B, N, rpg, gstride):
    if not gstride:
        return K.philox_normal((B, N), SEED, STREAM)
    g = cdiv(B, rpg)
    return torch.cat([K.philox_normal((rpg, N), SEED, STREAM + i * gstride) for i in range(g)])[:B].contiguous()


def _fwd_call(K, c, L, x, nz, pk, flags, act, dsf, klo, mvp, rs, ws, plain=False):
    var = K.VAR_EXACT if c["var"] == "exact" else K.VAR_REFERENCE
    if plain:
        return K.lib.lbbnn_lrt_f32_fwd(L, K.ptr(x), c["B"], nz, pk, var, flags, K.ptr(act), K.ptr(dsf, True), K.ptr(klo, True),
                                       mvp, ws.data_ptr(), ws.numel(), K.current_stream())
    return K.lib.lbbnn_lrt_f32_fwd_ex(L, K.ptr(x), c["B"], nz, pk, var, flags, K.ptr(act), K.ptr(dsf, True), K.ptr(klo, True),
                                      mvp, K.ptr(rs, True), c["rpg"], c["gstride"], ws.data_ptr(), ws.numel(), K.current_stream())


@pytest.mark.parametrize("c", FWD_CASES, ids=_id)
def test_forward(K, c):
    rng = _rng(c)
    B, Kf, N, off = c["B"], c["K"], c["N"], c["off"]
    p = _params(rng, Kf, N)
    z, zkl = _zs(rng, c["z"], Kf)
    L = _layer(K, p, z, zkl)
    pk, po = _priors(K, c["pri"])
    x = _at(_u(rng, -0.5, 1.0, B, Kf), off)
    rs = _at(_u(rng, 0.5, 1.5, cdiv(B, c["rpg"]), Kf), c["rs_off"]) if c["rowscale"] else None
    sample, moments = c["sample"], c["moments"]
    flags = ((K.FLAG_SAMPLE if sample else 0) | (K.FLAG_RELU if c["relu"] else 0) | (K.FLAG_KL if c["kl"] else 0)
             | (K.FLAG_MOMENTS if moments else 0))
    if c["noise"] == "inj":
        eps = _n(rng, B, N)
        eps_dev = _at(eps, off)                     # the noise struct holds only its address: keep it alive
        nz = K.make_noise(eps_dev)
    else:
        eps = _philox_rows(K, B, N, c["rpg"], c["gstride"])
        nz = K.make_noise(None, SEED, STREAM)
    mv_floats = K.lrt_mv_bytes(Kf, N) // 4
    mvb = torch.full((mv_floats + 1,), float("nan"), device="cuda") if c["mv"] else None
    mvp = mvb.data_ptr() + 4 * off if c["mv"] else None
    ws = _ws(K, B, Kf, N)

    def run(plain=False, noise=nz):
        act = _at((B, N), off)
        dsf = _at((B, N), off) if sample else None
        klo = torch.full((1,), float("nan"), device="cuda") if c["kl"] else None
        K.check(_fwd_call(K, c, L, x, noise, pk, flags, act, dsf, klo, mvp, rs, ws, plain))
        return act, dsf, klo

    act, dsf, klo = run()
    # float64 reference from the same fp32 inputs and noise
    p64 = {k: v.double() for k, v in p.items()}
    M, V = _moments(p64, c["var"], _d(z))
    x64 = x.double()
    xin = x64 * rs.double().repeat_interleave(c["rpg"], 0)[:B] if c["rowscale"] else x64
    e_b = xin @ M.T + p64["bias_mu"]
    var_b = (x64 * x64) @ V.T + O.sigma_of(p64["bias_rho"]) ** 2
    errs = {}
    if not sample:
        errs["act"] = _check("act", act, e_b.clamp_min(0) if c["relu"] else e_b)
    elif moments:
        errs["e_b"] = _check("e_b", act, e_b)
        errs["var_b"] = _check("var_b", dsf, var_b)
    else:
        a = e_b + var_b.sqrt() * eps.double()
        errs["act"] = _check("act", act, a.clamp_min(0) if c["relu"] else a)
        errs["dsf"] = _check("ds_factor", dsf, eps.double() / (2.0 * var_b.sqrt()))
    if c["kl"]:
        errs["kl"] = _check("kl", klo, O.lrt_kl(p64, po, z=_d(zkl if zkl is not None else z)).reshape(1))
    if c["mv"]:
        nk, vo = N * Kf, off + cdiv(N * Kf * 4, 256) * 64
        errs["M"] = _check("M cache", mvb[off:off + nk].view(N, Kf), M)
        if sample:
            errs["V"] = _check("V cache", mvb[vo:vo + nk].view(N, Kf), V)
    _report(f"fwd {_id(c)}", **errs)
    # native noise is the exported Philox stream, bit for bit
    if c["noise"] == "nat":
        eps_dev = _at(eps, off)
        a2, d2, _ = run(noise=K.make_noise(eps_dev))
        assert torch.equal(a2, act) and (dsf is None or torch.equal(d2, dsf))
    # a repeated launch is bit-identical (through lbbnn_lrt_f32_fwd where the call needs nothing of the _ex form)
    plain = not (moments or c["rowscale"] or c["gstride"])
    a3, d3, k3 = run(plain=plain)
    assert torch.equal(a3, act) and (dsf is None or torch.equal(d3, dsf)) and (klo is None or torch.equal(k3, klo))


@pytest.mark.parametrize("Kf,N,zk,var,pri,sample", PRO_CASES)
def test_prologue_moments_and_kl(K, Kf, N, zk, var, pri, sample):
    rng = _rng((Kf, N, zk, var, pri, sample))
    p = _params(rng, Kf, N)
    z, zkl = _zs(rng, zk, Kf)
    pk, po = _priors(K, pri)
    M, V = torch.full((N, Kf), float("nan"), device="cuda"), torch.full((N, Kf), float("nan"), device="cuda")
    klo = torch.full((1,), float("nan"), device="cuda")
    ws = torch.full((1 << 20,), 0xFF, dtype=torch.uint8, device="cuda")
    L = _layer(K, p, z, zkl)
    vm = K.VAR_EXACT if var == "exact" else K.VAR_REFERENCE
    K.check(K.lib.lbbnn_lrt_f32_prologue(L, pk, vm, K.FLAG_SAMPLE if sample else 0, K.ptr(M), K.ptr(V) if sample else None,
                                         K.ptr(klo), ws.data_ptr(), ws.numel(), K.current_stream()))
    p64 = {k: v.double() for k, v in p.items()}
    M64, V64 = _moments(p64, var, _d(z))
    e = {"M": _check("M", M, M64)}
    if sample:
        e["V"] = _check("V", V, V64)
    else:
        assert torch.isnan(V).all()
    e["kl"] = _check("kl", klo, O.lrt_kl(p64, po, z=_d(zkl if zkl is not None else z)).reshape(1))
    _report(f"prologue {Kf}x{N} {zk} {var} {pri}", **e)


@pytest.mark.parametrize("n_part", [1, 5, 3000])
def test_kl_finalize_sums_partials_and_bias_term(K, n_part):
    rng = _rng(("klfin", n_part))
    p = _params(rng, 8, 300)
    pk, po = _priors(K, "sim")
    part = torch.from_numpy(rng.uniform(-1, 3, size=n_part)).cuda()
    klo = torch.full((1,), float("nan"), device="cuda")
    K.check(K.lib.lbbnn_lrt_kl_finalize(part.data_ptr(), n_part, _layer(K, p), pk, K.ptr(klo), K.current_stream()))
    sb = O.sigma_of(p["bias_rho"].double())
    bias = (math.log(po.bias_sigma) - torch.log(sb) - 0.5 + (sb ** 2 + (p["bias_mu"].double() - po.bias_mu) ** 2)
            / (2.0 * po.bias_sigma ** 2)).sum()
    _check("kl", klo, (part.sum() + bias).reshape(1))


# ---- 2) backward: dW GEMM + finalize, dx, finalize alone, fused Adam --------------------------------------------------
def _lgrads(K, g, dz, dzkl):
    return K.LayerGrads(*[K.ptr(g[k]) for k in NAMES], K.ptr(dz, True), K.ptr(dzkl, True))


def _z_outs(Kf, req):
    dz = torch.zeros(Kf, device="cuda") if req in ("dz", "both") else None        # accumulated with atomics: zeroed first
    dzkl = torch.zeros(Kf, device="cuda") if req in ("dzkl", "both") else None
    return dz, dzkl


def _check_grads(tag, c, g, dz, dzkl, ref, prefill):
    e = {}
    for k in NAMES:
        want = ref[k] + (prefill[k].double() if prefill is not None else 0.0)
        e[k] = _check(f"{tag} {k}", g[k], want)
    edz, edzkl = _expected_dz(c["req"], ref)
    if edz is not None:
        e["dz"] = _check(f"{tag} dz", dz, edz)
    if edzkl is not None:
        e["dz_kl"] = _check(f"{tag} dz_kl", dzkl, edzkl)
    return e


@pytest.mark.parametrize("c", BWDW_CASES, ids=_id)
def test_bwd_params(K, c):
    rng = _rng(c)
    B, Kf, N, off, sample = c["B"], c["K"], c["N"], c["off"], c["sample"]
    p = _params(rng, Kf, N)
    z, zkl = _zs(rng, c["z"], Kf)
    L = _layer(K, p, z, zkl)
    pk, po = _priors(K, c["pri"])
    x, ga = _at(_u(rng, -0.5, 1.0, B, Kf), off), _at(_n(rng, B, N), off)
    dsf = _at(_u(rng, -2.0, 2.0, B, N), off) if sample else None
    kd, kh, klg = _klg(K, c["klg"])
    flags = (K.FLAG_SAMPLE if sample else 0) | (K.FLAG_ACCUMULATE if c["acc"] else 0)
    vm = K.VAR_EXACT if c["var"] == "exact" else K.VAR_REFERENCE
    ws = _ws(K, B, Kf, N)

    def run():
        g = _grad_bufs(_rng(c), p, off, c["acc"])
        pre = {k: v.clone() for k, v in g.items()} if c["acc"] else None
        dz, dzkl = _z_outs(Kf, c["req"])
        K.check(K.lib.lbbnn_lrt_f32_bwd_params(L, K.ptr(x), B, K.ptr(ga), K.ptr(dsf, True), pk, vm, flags, K.ptr(kd, True), kh,
                                               _lgrads(K, g, dz, dzkl), ws.data_ptr(), ws.numel(), K.current_stream()))
        return g, dz, dzkl, pre

    g, dz, dzkl, pre = run()
    x64, g64 = x.double(), ga.double()
    dM = g64.T @ x64
    gs = g64 * dsf.double() if sample else torch.zeros_like(g64)
    dV = gs.T @ (x64 * x64)
    cs = torch.cat([g64.sum(0), gs.sum(0)])
    ref = ref_param_grads(p, z, zkl, dM, dV, cs, klg, c["var"], po, sample)
    _report(f"bwd_params {_id(c)}", **_check_grads("bwd_params", c, g, dz, dzkl, ref, pre))
    # repeated launch: bit-identical, except dz / dz_kl (atomics: the summation order varies), held to the bound above
    g2, dz2, dzkl2, _ = run()
    for k in NAMES:
        assert torch.equal(g2[k], g[k]), k
    _check_grads("bwd_params (repeat)", c, g2, dz2, dzkl2, ref, pre)


@pytest.mark.parametrize("c", DX_CASES, ids=_id)
def test_bwd_input(K, c):
    rng = _rng(c)
    B, Kf, N, off, sample = c["B"], c["K"], c["N"], c["off"], c["sample"]
    p = _params(rng, Kf, N)
    z, zkl = _zs(rng, c["z"], Kf)
    L = _layer(K, p, z, zkl)
    pk, _ = _priors(K, "default")
    vm = K.VAR_EXACT if c["var"] == "exact" else K.VAR_REFERENCE
    x = _at(_u(rng, -0.5, 1.0, B, Kf), off)
    ga = _at(_n(rng, B, N), off)
    dsf = _at(_u(rng, -2.0, 2.0, B, N), off) if sample else None
    mvp = None
    if c["mv"]:    # the cache the forward leaves: [M | V] with V at the next 256-byte boundary
        mvb = torch.full((K.lrt_mv_bytes(Kf, N) // 4,), float("nan"), device="cuda")
        vo = cdiv(N * Kf * 4, 256) * 64
        K.check(K.lib.lbbnn_lrt_f32_prologue(L, pk, vm, K.FLAG_SAMPLE, mvb.data_ptr(), mvb.data_ptr() + 4 * vo, None, None, 0,
                                             K.current_stream()))
        mvp = mvb.data_ptr()
    flags = ((K.FLAG_SAMPLE if sample else 0) | (K.FLAG_MASK_DX if c["mask"] else 0) | (K.FLAG_ACCUMULATE if c["acc"] else 0))
    ws = _ws(K, B, Kf, N)
    pre = _n(rng, B, Kf)

    def run():
        dx = _at(pre if c["acc"] else (B, Kf), off)
        K.check(K.lib.lbbnn_lrt_f32_bwd_input(L, K.ptr(x), B, K.ptr(ga), K.ptr(dsf, True), pk, vm, flags, mvp, K.ptr(dx),
                                              ws.data_ptr(), ws.numel(), K.current_stream()))
        return dx

    dx = run()
    p64 = {k: v.double() for k, v in p.items()}
    M, V = _moments(p64, c["var"], _d(z))
    x64 = x.double()
    ref = ga.double() @ M
    if sample:
        ref = ref + 2.0 * x64 * ((ga.double() * dsf.double()) @ V)
    if c["mask"]:
        ref = ref * (x64 > 0)
    if c["acc"]:
        ref = ref + pre.double()
    _report(f"bwd_input {_id(c)}", dx=_check("dx", dx, ref))
    assert torch.equal(run(), dx)


@pytest.mark.parametrize("c", FIN_CASES, ids=_id)
def test_finalize(K, c):
    rng = _rng(c)
    Kf, N, off, sample = c["K"], c["N"], c["off"], c["sample"]
    p = {k: _at(v, off) for k, v in _params(rng, Kf, N).items()}
    z, zkl = _zs(rng, c["z"], Kf)
    L = _layer(K, p, z, zkl)
    pk, po = _priors(K, c["pri"])
    dM, dV, cs = _at(_n(rng, N, Kf), off), _at(_n(rng, N, Kf), off), _n(rng, 2 * N)
    kd, kh, klg = _klg(K, c["klg"])
    flags = (K.FLAG_SAMPLE if sample else 0) | (K.FLAG_ACCUMULATE if c["acc"] else 0)
    vm = K.VAR_EXACT if c["var"] == "exact" else K.VAR_REFERENCE
    g = _grad_bufs(rng, p, off, c["acc"])
    pre = {k: v.clone() for k, v in g.items()} if c["acc"] else None
    dz, dzkl = _z_outs(Kf, c["req"])
    K.check(K.lib.lbbnn_lrt_f32_finalize(L, K.ptr(dM), K.ptr(dV) if sample else None, K.ptr(cs), pk, vm, flags, K.ptr(kd, True),
                                         kh, _lgrads(K, g, dz, dzkl), K.current_stream()))
    ref = ref_param_grads(p, z, zkl, dM, dV, cs, klg, c["var"], po, sample)
    _report(f"finalize {_id(c)}", **_check_grads("finalize", c, g, dz, dzkl, ref, pre))


def _adam_state(K, shapes):
    m = [torch.zeros(s, device="cuda") for s in shapes]
    v = [torch.zeros(s, device="cuda") for s in shapes]
    coef = torch.empty(2, device="cuda")
    st = K.AdamLayerState((ctypes.c_void_p * 5)(*[t.data_ptr() for t in m]), (ctypes.c_void_p * 5)(*[t.data_ptr() for t in v]),
                          coef.data_ptr(), 0.9, 0.999, 1e-8)
    return m, v, coef, st


def _adam_ref(p, m, v, g, t, lr, b1, b2, eps):
    m.mul_(b1).add_((1 - b1) * g)
    v.mul_(b2).add_((1 - b2) * g * g)
    p.sub_(lr / (1 - b1 ** t) * m / (v.sqrt() / math.sqrt(1 - b2 ** t) + eps))


@pytest.mark.parametrize("bias_only", [False, True])
@pytest.mark.parametrize("Kf,N,var,sample,klgk", ADAM_CASES)
def test_finalize_adam_two_steps(K, Kf, N, var, sample, klgk, bias_only):
    rng = _rng(("adam", Kf, N, var, sample, klgk, bias_only))
    p = _params(rng, Kf, N)
    L = _layer(K, p)
    pk, po = _priors(K, "default")
    vm = K.VAR_EXACT if var == "exact" else K.VAR_REFERENCE
    kd, kh, klg = _klg(K, klgk)
    if bias_only:                       # lbbnn_lrt_f32_finalize_adam_bias takes the KL weight as a host scalar only
        kd, klg = None, float(np.float32(kh))
    m, v, coef, st = _adam_state(K, [t.shape for t in p.values()])
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    lr, b1, b2, eps = (float(np.float32(a)) for a in (2e-3, 0.9, 0.999, 1e-8))
    p64 = {k: t.double() for k, t in p.items()}
    m64 = {k: torch.zeros_like(t) for k, t in p64.items()}
    v64 = {k: torch.zeros_like(t) for k, t in p64.items()}
    w0 = {k: p[k].clone() for k in NAMES[:3]}
    p_start = {k: t.clone().double() for k, t in p.items()}
    for t in (1, 2):
        dM, dV, cs = _n(rng, N, Kf), _n(rng, N, Kf), _n(rng, 2 * N)
        step.fill_(t)
        K.check(K.lib.lbbnn_adam_prepare(step.data_ptr(), lr, b1, b2, coef.data_ptr(), K.current_stream()))
        if bias_only:
            K.check(K.lib.lbbnn_lrt_f32_finalize_adam_bias(L, K.ptr(cs), pk, K.FLAG_SAMPLE if sample else 0, kh, st,
                                                           K.current_stream()))
        else:
            K.check(K.lib.lbbnn_lrt_f32_finalize_adam(L, K.ptr(dM), K.ptr(dV) if sample else None, K.ptr(cs), pk, vm,
                                                      K.FLAG_SAMPLE if sample else 0, K.ptr(kd, True), kh, st, K.current_stream()))
        ref = ref_param_grads({k: x.float() for k, x in p64.items()}, None, None, dM, dV, cs, klg, var, po, sample)
        for k in (NAMES[3:] if bias_only else NAMES):
            _adam_ref(p64[k], m64[k], v64[k], ref[k].double(), t, lr, b1, b2, eps)
    e = {}
    for i, k in enumerate(NAMES):
        if bias_only and i < 3:
            assert torch.equal(p[k], w0[k]) and not m[i].any() and not v[i].any(), k
            continue
        e[k] = _check(f"adam {k}", p[k], p64[k], TOL_ADAM)
        e[f"step {k}"] = _check(f"adam step {k}", p[k].double() - p_start[k], p64[k] - p_start[k], TOL_ADAM_STEP)
        _check(f"adam exp_avg {k}", m[i], m64[k], TOL_ADAM)
        _check(f"adam exp_avg_sq {k}", v[i], v64[k], TOL_ADAM)
    _report(f"adam {Kf}x{N} {var} sample={sample} klg={klgk} bias_only={bias_only}", **e)


# ---- 3) MNF auxiliary kernels --------------------------------------------------------------------------------------------
AUX_NAMES = ("q0_mean", "q0_log_var", "z0", "r0_c", "r0_b1", "r0_b2", "z2", "M0", "V", "eps_r", "z_b")
AUX_GRADS = ("q0_mean", "q0_log_var", "z0", "r0_c", "r0_b1", "r0_b2", "z2", "z_b", "M0", "V")
AUX_ATOMIC = ("r0_c", "z2")                                   # d_r0_c, d_z2: one atomic per column and row slice


def _aux_inputs(D, O_):
    rng = np.random.default_rng(D * 1000 + O_)
    t = lambda *s, scale=1.0, off=0.0: torch.from_numpy(off + scale * rng.standard_normal(size=s)).float().cuda()  # noqa: E731
    return {"q0_mean": t(D, scale=0.1), "q0_log_var": t(D, scale=0.1, off=-3.0), "z0": t(D, scale=0.3), "r0_c": t(D, scale=0.1),
            "r0_b1": t(D, scale=0.1), "r0_b2": t(D, scale=0.1), "z2": t(D, scale=0.5, off=1.0),
            "M0": t(O_, D, scale=0.05), "V": torch.from_numpy(rng.random(size=(O_, D)) * 1e-3 + 1e-5).float().cuda(),
            "eps_r": t(O_), "z_b": t(D)}


def _aux_struct(K, a):
    D, O_ = a["M0"].shape[1], a["M0"].shape[0]
    return K.MnfAux(D, O_, *[K.ptr(a[n]) for n in AUX_NAMES])


def _aux_ref(a, gscale):
    """log_q0 - log_rb (MNF:212-227) in float64 torch ops, its parts and every gradient times gscale."""
    d = {k: v.double().requires_grad_(k != "eps_r") for k, v in a.items()}
    log_q0 = (-0.5 * math.log(math.pi) - 0.5 * d["q0_log_var"] - 0.5 * ((d["z0"] - d["q0_mean"]) ** 2 / d["q0_log_var"].exp())).sum()
    act_var = (d["r0_c"] ** 2) @ d["V"].T
    a_r = torch.tanh((d["r0_c"] * d["z2"]) @ d["M0"].T + act_var.sqrt() * d["eps_r"])
    mean_r, lvr = d["r0_b1"] * a_r.mean(), d["r0_b2"] * a_r.mean()
    log_rb = (-0.5 * math.log(math.pi) - 0.5 * lvr - 0.5 * ((d["z_b"][-1] - mean_r) ** 2 / lvr.exp())).sum()
    out = log_q0 - log_rb
    grads = torch.autograd.grad(gscale * out, [d[n] for n in AUX_GRADS])
    return (torch.stack([out, log_q0, log_rb]).detach(), torch.cat([a_r, act_var, a_r.mean().reshape(1)]).detach(),
            dict(zip(AUX_GRADS, grads)))


def _aux_fwd(K, a, ticket):
    O_ = a["M0"].shape[0]
    out = torch.full((3,), float("nan"), device="cuda")
    save = torch.full((int(K.lib.lbbnn_mnf_aux_save_floats(O_)),), float("nan"), device="cuda")
    K.check(K.lib.lbbnn_mnf_aux_kl_fwd(_aux_struct(K, a), K.ptr(out), K.ptr(save), ticket.data_ptr(), K.current_stream()))
    return out, save


@pytest.mark.parametrize("D,O_", AUX_FWD_CASES)
def test_aux_kl_fwd(K, D, O_):
    a = _aux_inputs(D, O_)
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    out, save = _aux_fwd(K, a, ticket)
    ref, ref_save, _ = _aux_ref(a, 1.0)
    e = {n: _check(n, out[i:i + 1], ref[i:i + 1]) for i, n in enumerate(("q0-rb", "log_q0", "log_rb"))}
    e["a_r"] = _check("a_r", save[:O_], ref_save[:O_])
    e["act_var"] = _check("act_var", save[O_:2 * O_], ref_save[O_:2 * O_])
    e["amean"] = _check("mean a_r", save[2 * O_:], ref_save[2 * O_:])
    _report(f"aux_fwd {D}x{O_}", **e)
    assert int(ticket) == 0                                   # the last block resets the ticket
    out2, save2 = _aux_fwd(K, a, ticket)                      # ... so the same ticket serves the next launch
    assert torch.equal(out2, out) and torch.equal(save2, save) and int(ticket) == 0


@pytest.mark.parametrize("D,O_,forced", AUX_BWD_CASES)
def test_aux_kl_bwd(K, D, O_, forced, monkeypatch):
    if forced is None:
        monkeypatch.delenv("LBBNN_AUX_SLICES", raising=False)
    else:
        monkeypatch.setenv("LBBNN_AUX_SLICES", str(forced))
    a = _aux_inputs(D, O_)
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    _, save = _aux_fwd(K, a, ticket)
    gout = torch.tensor([0.7], device="cuda")
    ref = _aux_ref(a, float(np.float32(0.7)))[2]

    # The per-column gradients (d q0_*, d z0, d r0_b*, d z_b) start as NaN, so a column that no row slice writes fails.  Which
    # slice writes them cannot be seen: every slice computes the same values from the column alone, so more writers than
    # slice 0 would store identical bits.  The guard that keeps it to slice 0 saves stores; this test does not check it.
    def run():
        vec = torch.full((8, D), float("nan"), device="cuda")    # per-column outputs: NaN unless written
        dM0, dV = torch.full((O_, D), float("nan"), device="cuda"), torch.full((O_, D), float("nan"), device="cuda")
        g = {n: vec[i] for i, n in enumerate(AUX_GRADS[:8])}
        g["M0"], g["V"] = dM0, dV
        grads = K.MnfAuxGrads(*[K.ptr(g[n]) for n in AUX_GRADS])
        K.check(K.lib.lbbnn_mnf_aux_kl_bwd(_aux_struct(K, a), K.ptr(save), K.ptr(gout), grads, K.current_stream()))
        return g

    g = run()
    e = {n: _check(f"d {n}", g[n], ref[n]) for n in AUX_GRADS}
    _report(f"aux_bwd {D}x{O_} slices={aux_slices(D, O_, forced=forced)}", **e)
    g2 = run()
    for n in AUX_GRADS:
        if n in AUX_ATOMIC:
            _check(f"d {n} (repeat)", g2[n], ref[n])
        else:
            assert torch.equal(g2[n], g[n]), n


@pytest.mark.parametrize("R,D,O_,noise,with_r", DRAW_CASES)
def test_mnf_draw(K, R, D, O_, noise, with_r):
    rng = np.random.default_rng(R * 7 + D)
    q0m, q0lv = _n(rng, D, scale=0.1), _n(rng, D, scale=0.3) - 2.0
    if noise == "inj":
        eps_in, epsr_in = _n(rng, R, D), _n(rng, O_)
        nz, nzr = K.make_noise(eps_in), K.make_noise(epsr_in)
    else:
        nz, nzr = K.make_noise(None, SEED, STREAM), K.make_noise(None, SEED, STREAM + 1)
        eps_in, epsr_in = K.philox_normal((R, D), SEED, STREAM), (K.philox_normal(O_, SEED, STREAM + 1) if O_ else None)
    eps, z0 = torch.full((R, D), float("nan"), device="cuda"), torch.full((R, D), float("nan"), device="cuda")
    eps_r = torch.full((max(O_, 1),), float("nan"), device="cuda") if with_r else None
    K.check(K.lib.lbbnn_mnf_draw(K.ptr(q0m), K.ptr(q0lv), nz, R, D, K.ptr(eps), K.ptr(z0), nzr if with_r else None, O_,
                                 K.ptr(eps_r, True), K.current_stream()))
    assert torch.equal(eps, eps_in)                            # injected copied / native = the exported stream
    if with_r:
        assert torch.equal(eps_r[:O_], epsr_in)
    ref = q0m.double() + q0lv.double().exp().sqrt() * eps.double()
    _report(f"draw R{R} D{D} {noise}", z0=_check("z0", z0, ref))


@pytest.mark.parametrize("R,D,kl_row,aux", DRAW_BWD_CASES)
def test_mnf_draw_bwd(K, R, D, kl_row, aux):
    rng = np.random.default_rng(R * 11 + D + kl_row)
    q0m, q0lv, eps, dz0 = _n(rng, D, scale=0.1), _n(rng, D, scale=0.3) - 2.0, _n(rng, R, D), _n(rng, R, D)
    am, alv, az0 = (_n(rng, D) for _ in range(3)) if aux else (None, None, None)
    dm, dlv = torch.full((D,), float("nan"), device="cuda"), torch.full((D,), float("nan"), device="cuda")
    K.check(K.lib.lbbnn_mnf_draw_bwd(K.ptr(q0lv), K.ptr(eps), K.ptr(dz0), R, D, kl_row, K.ptr(am, True), K.ptr(alv, True),
                                     K.ptr(az0, True), K.ptr(dm), K.ptr(dlv), K.current_stream()))
    m64, lv64 = q0m.double().requires_grad_(True), q0lv.double().requires_grad_(True)
    z0 = m64 + lv64.exp().sqrt() * eps.double()
    L = (dz0.double() * z0).sum()
    if aux:
        L = L + (am.double() * m64).sum() + (alv.double() * lv64).sum()
        if kl_row >= 0:
            L = L + (az0.double() * z0[kl_row]).sum()
    gm, glv = torch.autograd.grad(L, [m64, lv64])
    _report(f"draw_bwd R{R} D{D} kl_row{kl_row} aux={aux}", d_mean=_check("d q0_mean", dm, gm), d_lv=_check("d q0_log_var", dlv, glv))


@pytest.mark.parametrize("D", ROWS_D)
@pytest.mark.parametrize("what", ROWS_CASES, ids="-".join)
def test_mnf_bwd_rows(K, D, what):
    rng = np.random.default_rng(D)
    g = torch.tensor([1.25], device="cuda")
    dzk, a, b = _n(rng, D), _n(rng, D), _n(rng, D)
    dld = torch.full((2,), float("nan"), device="cuda") if "dld" in what else None
    rows = torch.full((2, D), float("nan"), device="cuda") if "rows" in what else None
    pa, pb, pz = (None if f"no_{n}" in what else t for n, t in (("a", a), ("b", b), ("dzk", dzk)))
    K.check(K.lib.lbbnn_mnf_bwd_rows(K.ptr(g) if dld is not None else None, -0.5, K.ptr(dld, True), K.ptr(pz, True), K.ptr(pa, True),
                                     K.ptr(pb, True), D, K.ptr(rows, True), K.current_stream()))
    if dld is not None:
        assert dld.tolist() == [0.0, -0.625]
    if rows is not None:
        zero = torch.zeros(D, device="cuda")
        assert torch.equal(rows[0], pz if pz is not None else zero)
        assert torch.equal(rows[1], (pa if pa is not None else zero) + (pb if pb is not None else zero))


def test_mnf_kl_combine(K):
    v = torch.tensor([123.25, -7.5, 3.125, 0.0625, float("nan")], device="cuda")
    aux = torch.tensor([-7.5, 1.0, 2.0], device="cuda")
    K.check(K.lib.lbbnn_mnf_kl_combine(v[0:1].data_ptr(), K.ptr(aux), v[2:3].data_ptr(), v[3:4].data_ptr(), v[4:5].data_ptr(),
                                       K.current_stream()))
    rng = np.random.default_rng(3)
    kl, a0, lq, lr_ = (np.float32(x) for x in rng.normal(0, 50, size=4))
    t = torch.tensor([kl, a0, 0.0, 0.0, lq, lr_, float("nan")], device="cuda")
    K.check(K.lib.lbbnn_mnf_kl_combine(t[0:1].data_ptr(), t[1:4].data_ptr(), t[4:5].data_ptr(), t[5:6].data_ptr(),
                                       t[6:7].data_ptr(), K.current_stream()))
    assert v[4].item() == (123.25 - 7.5) - 3.125 - 0.0625
    assert t[6].item() == float(np.float32(np.float32(np.float32(kl + a0) - lq) - lr_))


# ---- 4) the MNF layer end to end, at shapes the golden file lacks --------------------------------------------------------
@pytest.mark.parametrize("B,i,o,pri", MNF_SWEEP)
def test_mnf_layer_sweep(B, i, o, pri):
    import lbbnn as lb
    case = C.mnf_layer_case(100 + i + o, B, i, o)
    po = O.Priors(*PRIORS[pri])
    named = C.flat_named(case["p"])
    named64 = {k: v.double().clone().requires_grad_(True) for k, v in named.items()}
    p64 = C.unflatten_like(case["p"], named64)
    x64 = case["x"].double().clone().requires_grad_(True)
    nz64 = {k: ([m.double() for m in v] if isinstance(v, list) else v.double()) for k, v in case["noise"].items()}
    act64, kl64 = O.mnf_forward(x64, p64, nz64, priors=po)
    ((act64 * case["gout"].double()).sum() + kl64 / C.NUM_BATCHES).backward()
    layer = lb.mnf.BayesianLinear(i, o, 2, mu_prior=po.mu, sigma_prior=po.sigma, alpha_prior=po.alpha, bias_mu_prior=po.bias_mu,
                                  bias_sigma_prior=po.bias_sigma)
    layer.load_state_dict(named)
    layer = layer.cuda().train()
    x = case["x"].cuda().requires_grad_(True)
    nz = {k: ([m.cuda() for m in v] if isinstance(v, list) else v.cuda()) for k, v in case["noise"].items()}
    act = layer(x, noise=nz)
    ((act * case["gout"].cuda()).sum() + layer.kl / C.NUM_BATCHES).backward()
    e = {"act": _check("act", act.detach(), act64.detach()),
         "kl": _check("kl", layer.kl.detach().reshape(1), kl64.detach().reshape(1)),
         "dx": _check("dx", x.grad, x64.grad)}
    got = dict(layer.named_parameters())
    assert set(got) == set(named64)
    worst = max(((C.rel_err(got[n].grad, v.grad), n) for n, v in named64.items()))
    for n, v in named64.items():
        _check(f"d {n}", got[n].grad, v.grad)
    _report(f"mnf layer B{B} {i}->{o} {pri}", **e, worst_grad=worst[0])


# ---- 5) argument rejections ----------------------------------------------------------------------------------------------
def test_entry_points_reject_bad_arguments(K):
    rng = np.random.default_rng(0)
    B, Kf, N = 4, 8, 6
    p = _params(rng, Kf, N)
    z = _u(rng, 0.5, 1.5, Kf)
    L, Lz = _layer(K, p), _layer(K, p, z)
    pk, _ = _priors(K, "default")
    x, act, dsf = _u(rng, 0, 1, B, Kf), torch.empty(B, N, device="cuda"), torch.empty(B, N, device="cuda")
    ws = _ws(K, B, Kf, N)
    s = K.current_stream()

    def fwd(flags=K.FLAG_SAMPLE, ds=dsf, rs=None, rpg=0, gstride=0, nbytes=None, var=K.VAR_REFERENCE, klo=None):
        K.check(K.lib.lbbnn_lrt_f32_fwd_ex(L, K.ptr(x), B, K.make_noise(None, 1, 2), pk, var, flags, K.ptr(act), K.ptr(ds, True),
                                           K.ptr(klo, True), None, K.ptr(rs, True), rpg, gstride, ws.data_ptr(),
                                           ws.numel() if nbytes is None else nbytes, s))

    cases = [
        (lambda: fwd(K.FLAG_SAMPLE | K.FLAG_MOMENTS, ds=None), "FLAG_MOMENTS writes var_b"),
        (lambda: fwd(K.FLAG_MOMENTS), "FLAG_MOMENTS writes var_b"),
        (lambda: fwd(gstride=3, rpg=3), "rows_per_group \\* out_features"),     # 3 * 6 % 4 != 0
        (lambda: fwd(gstride=3), "rows_per_group \\* out_features"),
        (lambda: fwd(rs=x, rpg=0), "rowscale needs rows_per_group"),
        (lambda: fwd(nbytes=ws.numel() - 1), "workspace too small"),
        (lambda: fwd(var=2), "bad var_mode"),
        (lambda: fwd(K.FLAG_SAMPLE | K.FLAG_KL), "FLAG_KL needs kl_out"),
    ]
    g = {k: torch.empty_like(v) for k, v in p.items()}
    dz = torch.zeros(Kf, device="cuda")

    def bwd(layer, dz=None, dzkl=None, ds=dsf, nbytes=None):
        K.check(K.lib.lbbnn_lrt_f32_bwd_params(layer, K.ptr(x), B, K.ptr(act), K.ptr(ds, True), pk, 0, K.FLAG_SAMPLE, None, 1.0,
                                               _lgrads(K, g, dz, dzkl), ws.data_ptr(), ws.numel() if nbytes is None else nbytes, s))

    cases += [
        (lambda: bwd(L, dz=dz), "dz requested but the layer has no z"),
        (lambda: bwd(Lz, dzkl=dz), "dz_kl requested but the layer has no z_kl"),
        (lambda: bwd(L, ds=None), "needs the saved ds_factor"),
        (lambda: bwd(L, nbytes=ws.numel() - 1), "workspace too small"),
        (lambda: K.check(K.lib.lbbnn_lrt_f32_bwd_input(L, K.ptr(x), B, K.ptr(act), K.ptr(dsf), pk, 0, K.FLAG_SAMPLE, None,
                                                       K.ptr(x), ws.data_ptr(), 16, s)), "workspace too small"),
        (lambda: K.check(K.lib.lbbnn_lrt_f32_finalize(L, K.ptr(act), None, K.ptr(act), pk, 0, K.FLAG_SAMPLE, None, 1.0,
                                                      _lgrads(K, g, None, None), s)), "sample branch needs dV"),
        (lambda: K.check(K.lib.lbbnn_lrt_f32_prologue(L, pk, 0, 0, K.ptr(act), None, K.ptr(act), ws.data_ptr(), 8, s)),
         "workspace too small for the KL partials"),
    ]
    m, v, coef, st = _adam_state(K, [t.shape for t in p.values()])
    cases.append((lambda: K.check(K.lib.lbbnn_lrt_f32_finalize_adam(Lz, K.ptr(act), K.ptr(act), K.ptr(act), pk, 0, K.FLAG_SAMPLE,
                                                                    None, 1.0, st, s)), "no multiplicative z"))
    q, e1 = _u(rng, 0, 1, 2, Kf), torch.empty(2, Kf, device="cuda")
    cases += [
        (lambda: K.check(K.lib.lbbnn_mnf_draw_bwd(K.ptr(q[0]), K.ptr(q), K.ptr(q), 2, Kf, 2, None, None, None, K.ptr(e1[0]),
                                                  K.ptr(e1[1]), s)), "kl_row out of range"),
        (lambda: K.check(K.lib.lbbnn_mnf_draw(K.ptr(q[0]), K.ptr(q[0]), K.make_noise(None, 1, 2), 2, Kf, K.ptr(e1), K.ptr(e1), None,
                                              3, K.ptr(e1), s)), "eps_r needs its noise source"),
        (lambda: K.check(K.lib.lbbnn_mnf_bwd_rows(None, 1.0, None, None, None, None, Kf, None, s)), "nothing to do"),
        (lambda: K.check(K.lib.lbbnn_mnf_bwd_rows(None, 1.0, None, None, None, None, 0, K.ptr(e1), s)), "bad shape"),
    ]
    a = _aux_inputs(8, 3)
    bad = _aux_struct(K, a)
    bad.z_b = None
    t = torch.zeros(1, dtype=torch.int32, device="cuda")
    cases.append((lambda: K.check(K.lib.lbbnn_mnf_aux_kl_fwd(bad, K.ptr(e1), K.ptr(e1), t.data_ptr(), s)), "NULL argument"))
    for call, msg in cases:
        with pytest.raises(K.LbbnnError, match=msg):
            call()
    torch.cuda.synchronize()
    assert int(t) == 0
