"""The posterior-predictive kernels through the C-ABI, each against a float64 restatement of what it computes, on the GPU,
from the same inputs and the same noise:
  tc_linear_tf32x3       out = [relu](A W^T + b) on the tensor cores (3xTF32), 1-CTA and CTA-pair kernels (csrc/tc_gemm_tf32.cu)
  lrt_mc_epilogue        act = [relu](E + b_mu + sqrt(S + sigma_b^2) eps), hi / lo of act .* rowscale and of act^2
  tf32_split_rows        hi / lo of x .* rowscale and of x^2                                  (csrc/lrt_predict.cu)
  lrt_sample_expand      act = [relu](e + sqrt(var) eps)                                      (csrc/lrt_f32.cu)
  linear_f32_batched     out[s] = [relu](x[s] W[s]^T + b[s]) on the CUDA cores, 64- and 128-wide column tiles
  mc_head_accumulate     the <= 16-class head fused with the two fp64 accumulators
  mc_accumulate_batched  the two fp64 accumulators
  mc_prepare, mc_sample, mc_sample_split   sigma, alpha and the weight draws of the MF loop  (csrc/mc_predict.cu)
Bounds (cases.rel_err = max|a-b| / max|b|): 1e-5 for the GEMMs and the accumulators, 1e-6 for the elementwise kernels, and
bit-exact wherever a kernel promises it: hi + lo == value, hi representable in TF32 (low 13 bits clear), native noise ==
the exported Philox stream, masks, and repeated launches.

The launch rules and configuration tables above the tests are plain Python: tests/test_predict_kernels_cpu.py checks,
without a GPU, that the tables still reach every launch path at 148 SMs."""
import itertools
import random
import zlib

import pytest
import torch

import cases as C

pytestmark = pytest.mark.gpu
TOL_GEMM, TOL_ELEM, TOL_ACC = 1e-5, 1e-6, 1e-5
SEED, STREAM = 4321, 11


def cdiv(a, b):
    return -(-a // b)


# ---- launch rules, restated from the host code ---------------------------------------------------------------------------
TC_BM, TC_BN, TC_BK = 128, 128, 32
TC_STAGES = {"1cta": 3, "pair": 4}


def tc_kernel(m, n, z, mode, sms):
    """The kernel lbbnn_tc_linear_tf32x3 launches under LBBNN_TC_PAIR=0 ("1cta"), =2 ("pair") or unset ("auto")."""
    if mode == "1cta" or m <= TC_BM:
        return "1cta"
    tiles2 = cdiv(m, 2 * TC_BM) * cdiv(n, TC_BN) * z
    return "pair" if mode == "pair" or tiles2 >= sms // 2 else "1cta"


def tc_tiles_per_cta(m, n, z, kernel, sms):
    """Most output tiles one CTA (or one CTA pair) processes in the persistent loop."""
    if kernel == "pair":
        tiles = cdiv(m, 2 * TC_BM) * cdiv(n, TC_BN) * z
        return cdiv(tiles, min(tiles, sms // 2))
    tiles = cdiv(m, TC_BM) * cdiv(n, TC_BN) * z
    return cdiv(tiles, min(tiles, sms))


def sgemm_tile(out_features):
    """Column tile of sgemm_tn_batched_kernel: 128 unless it would be mostly padding."""
    return 128 if cdiv(out_features, 128) * 128 * 100 <= cdiv(out_features, 64) * 64 * 112 else 64


HEAD_SMEM_MAX = 220 * 1024


def head_fits(c, k):
    return 4 * (c + 8) * k * 4 <= HEAD_SMEM_MAX


def head_kmax(c):
    return HEAD_SMEM_MAX // (16 * (c + 8)) // 4 * 4


def grid_stride(quads, sms):
    """lrt_predict.cu's elementwise kernels cap the grid at 16 blocks of 256 threads per SM."""
    return quads > 16 * sms * 256


def elementwise_vector(total, offset):
    """The float4 path of the elementwise kernels: a whole number of quads and 16-byte aligned operands."""
    return total % 4 == 0 and offset == 0


def noise_path(total, noise):
    return noise if noise in ("inj", "none") else ("nat4" if total % 4 == 0 else "nat1")


# ---- configuration tables ------------------------------------------------------------------------------------------------
def _tc(z, m, n, k, relu=False, outs="both", layout="dense"):
    return dict(z=z, m=m, n=n, k=k, relu=relu, outs=outs, layout=layout)


TC_CASES = [
    _tc(7, 520, 700, 100, relu=True),                        # 210 1-CTA / 126 pair tiles at 148 SMs, crossing z
    _tc(16, 520, 700, 160, outs="out"),                      # 3-4 tiles per CTA: both TMEM buffers twice, 5 K blocks
    *[_tc(2, m, 72, 36, relu=m % 2 == 1) for m in (1, 127, 128, 129, 255, 257)],
    *[_tc(1, 200, n, 28, outs=("both", "out", "hilo")[i % 3]) for i, n in enumerate((1, 15, 16, 17, 65, 129))],
    *[_tc(2, 130, 70, k, relu=k % 8 == 4) for k in (4, 8, 28, 36, 100, 220)],
    _tc(3, 140, 64, 64, relu=True, outs="hilo", layout="pad"),
    _tc(2, 300, 61, 40, outs="both", layout="pad"),
    _tc(3, 140, 48, 64, outs="out", layout="chain"),
    _tc(5, 300, 40, 48, relu=True, outs="both", layout="chain"),
    _tc(4, 257, 45, 36, outs="hilo", layout="chain"),
]
TC_EXACT_SHAPES = [(2, 260, 140, 40), (1, 129, 17, 8), (3, 257, 70, 100)]
TC_LONG_K = [4096, 8192]
# Measured on a B200 with these inputs (rel_err, the same for both kernels): signed 1.07e-5 at K = 4096 and 2.15e-5 at 8192,
# all-positive 3.03e-5 and 6.15e-5.  The 1e-5 fp32 bound does not hold at these K: the truncating accumulation into the
# main TMEM sum grows with K / 8 and is largest when nothing cancels.
_LONG_K_OVER = pytest.mark.xfail(strict=True, reason="3xTF32 truncation error exceeds 1e-5 at K >= 4096 (measured above)")


def _epilogue_configs():
    """Every stride, noise and output combination of lrt_mc_epilogue; relu, group stride, row scale, sample count and a
    one-float offset picked by a fixed-seed generator; plus one launch past the grid cap."""
    rnd = random.Random(7)
    outs_all = [c for r in (1, 2, 3) for c in itertools.combinations(("act", "m", "v"), r)]
    cfgs = []
    for sample in (True, False):
        for es, ss in (itertools.product((0, 1), (0, 1)) if sample else ((0, 0), (1, 0))):
            for noise in (("inj", "nat4", "nat1") if sample else ("none",)):
                for outs in outs_all:
                    b, n = (6, 10) if noise == "nat4" else (5, 13) if noise == "nat1" else rnd.choice(((6, 10), (5, 13)))
                    cfgs.append(dict(sample=sample, es=es, ss=ss if sample else 0, noise=noise, outs=outs, B=b, N=n,
                                     relu=rnd.random() < 0.5, gstride=rnd.choice((0, 1000003)) if noise[:3] == "nat" else 0,
                                     rowscale="m" in outs and rnd.random() < 0.6, n=rnd.choice((1, 3, 17)),
                                     off=int(rnd.random() < 0.3)))
    cfgs.append(dict(sample=True, es=1, ss=1, noise="nat4", outs=("act", "m", "v"), B=1000, N=1000, relu=True,
                     gstride=1000003, rowscale=True, n=3, off=0))
    return cfgs


EPI_CASES = _epilogue_configs()

SPLIT_CASES = [   # tf32_split_rows: x stride 0 / dense / padded by 8 / padded by 5 (odd samples unaligned)
    dict(rows=7, cols=12, n=3, xs="shared", rowscale=True, outs="both", off=0),
    dict(rows=7, cols=12, n=3, xs="dense", rowscale=False, outs="hi", off=0),
    dict(rows=5, cols=13, n=4, xs="dense", rowscale=True, outs="hi", off=0),
    dict(rows=9, cols=8, n=3, xs="pad8", rowscale=False, outs="sq", off=0),
    dict(rows=9, cols=8, n=4, xs="pad5", rowscale=True, outs="both", off=0),
    dict(rows=3, cols=11, n=2, xs="pad8", rowscale=False, outs="both", off=1),
    dict(rows=1, cols=1, n=1, xs="shared", rowscale=True, outs="both", off=0),
    dict(rows=1000, cols=1000, n=3, xs="dense", rowscale=True, outs="both", off=0),
]

EXPAND_CASES = [
    dict(B=6, N=10, n=3, noise="nat4", relu=True, gstride=1000003, off=0),
    dict(B=5, N=13, n=4, noise="nat1", relu=False, gstride=1000003, off=0),
    dict(B=6, N=10, n=2, noise="nat4", relu=False, gstride=0, off=1),
    dict(B=5, N=13, n=3, noise="inj", relu=True, gstride=0, off=0),
    dict(B=6, N=10, n=1, noise="inj", relu=False, gstride=0, off=1),
    dict(B=1000, N=2500, n=2, noise="nat4", relu=True, gstride=1000003, off=0),
]

SGEMM_CASES = [   # (samples, batch M, in K, out N, x stride, relu); "odd": per-sample stride M K + 1
    (3, 130, 20, 64, "per", True),
    (3, 130, 20, 65, "per", False),
    (2, 257, 33, 128, "shared", True),
    (2, 100, 8, 129, "odd", False),
    (4, 1, 3, 192, "per", True),
    (2, 130, 16, 193, "odd", True),
    (2, 64, 36, 448, "shared", False),
    (2, 129, 100, 449, "per", True),
    (1, 300, 7, 1, "shared", False),
    (5, 37, 12, 17, "odd", True),
    (2, 128, 64, 513, "per", False),
]


def _head_cases():
    bs, ks, ns, hss = (1, 7, 8, 9, 1000), (4, 124, 128, 132, "max"), (1, 2, 3, 4, 5, 33), ("shared", "dense", "padded")
    out = [dict(C=c, B=bs[i % 5], K=ks[(3 * i) % 5], n=ns[i % 6], hs=hss[i % 3]) for i, c in enumerate(range(1, 17))]
    out += [dict(C=16, B=1000, K="max", n=5, hs="padded"), dict(C=10, B=1000, K=600, n=33, hs="dense")]
    for c in out:
        if c["K"] == "max":
            c["K"] = head_kmax(c["C"])
    return out


HEAD_CASES = _head_cases()
ACC_CASES = [(1, 37, 3, True), (10, 100, 5, False), (31, 9, 2, True), (32, 64, 7, True), (33, 5, 4, False), (100, 300, 3, True)]

# (out, in, samples, first sample); 600 x 400 at 40 samples: the 8 SMs / samples block cap forces the grid-stride loop
SAMPLE_CASES = [(7, 9, 3, 0), (12, 20, 5, 5), (600, 400, 40, 3)]
SAMPLE_STREAM_BASE, SAMPLE_STREAM_STRIDE = 8, 12


# ---- helpers --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def K():
    from lbbnn import _capi
    _capi.require_device()
    return _capi


@pytest.fixture(params=["1cta", "pair", "auto"])
def tc_mode(request, monkeypatch):
    """LBBNN_TC_PAIR=0 forces the 1-CTA kernel, =2 the CTA-pair kernel; unset, the host picks by tile count."""
    if request.param == "auto":
        monkeypatch.delenv("LBBNN_TC_PAIR", raising=False)
    else:
        monkeypatch.setenv("LBBNN_TC_PAIR", "0" if request.param == "1cta" else "2")
    return request.param


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def bits(t):
    return t.contiguous().view(torch.int32)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(bits(a), bits(b))


def same_value_bits(a, b):
    """Bit-identical once a zero's sign is dropped: a split of -0.0 is (-0.0, +0.0), whose sum is +0.0."""
    return same_bits(a + 0.0, b + 0.0)


def tf32_clean(hi):
    return int((bits(hi) & 0x1FFF).abs().max()) == 0


def _report(name, **kv):
    print(f"[predict-kernels] {name}: " + ", ".join(f"{k} {v:.3e}" for k, v in kv.items()), flush=True)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _buf(numel, off=0, fill=float("nan")):
    """A 1-D CUDA buffer of numel floats starting `off` floats into its storage."""
    return torch.full((numel + off,), fill, device="cuda")[off:]


def _split(K, x):
    hi, lo = torch.empty_like(x), torch.empty_like(x)
    K.check(K.lib.lbbnn_tf32_split(K.ptr(x), x.numel(), K.ptr(hi), K.ptr(lo), K.current_stream()))
    return hi, lo


def _philox_stack(K, n, total, stream, gstride):
    return torch.stack([K.philox_normal(total, SEED, (stream + s * gstride) % 2 ** 64) for s in range(n)])


# ---- a) lbbnn_tc_linear_tf32x3 ----------------------------------------------------------------------------------------------
def _tc_layout(layout, z, m, n, k):
    """(a pitch, a batch stride, a floats, out pitch, out batch stride, out floats)"""
    if layout == "dense":
        return k, m * k, z * m * k, n, m * n, z * m * n
    if layout == "pad":          # padded A rows and batches; an output pitch that is not a multiple of 4
        ap, op = k + 4, n + 3 if (n + 3) % 4 else n + 1
        return ap, m * ap + 4, z * (m * ap + 4), op, m * op, z * m * op
    # the MC chain: sample z of the (M, Z*K) output of the layer before, into an (M, Z*N) buffer
    return z * k, k, m * z * k, z * n, n, m * z * n


def _tc_call(K, ah, al, ap, ab, wh, wl, bias, z, m, n, k, relu, out, oh, ol, op, ob):
    K.check(K.lib.lbbnn_tc_linear_tf32x3(K.ptr(ah), K.ptr(al), ap, ab, K.ptr(wh), K.ptr(wl), K.ptr(bias), z, m, n, k,
                                         K.FLAG_RELU if relu else 0, K.ptr(out, True), K.ptr(oh, True), K.ptr(ol, True),
                                         op, ob, K.current_stream()))


def _tc_run(K, c, a, ah, al, wh, wl, bias):
    z, m, n, k = c["z"], c["m"], c["n"], c["k"]
    ap, ab, _, op, ob, on = _tc_layout(c["layout"], z, m, n, k)
    out = _buf(on) if c["outs"] in ("out", "both") else None
    oh, ol = (_buf(on), _buf(on)) if c["outs"] in ("hilo", "both") else (None, None)
    _tc_call(K, ah, al, ap, ab, wh, wl, bias, z, m, n, k, c["relu"], out, oh, ol, op, ob)
    return out, oh, ol


@pytest.mark.parametrize("c", TC_CASES, ids=lambda c: "z{z}-m{m}-n{n}-k{k}-{outs}-{layout}{r}".format(**c, r="-relu" * c["relu"]))
def test_tc_linear_tf32x3_matches_fp64(K, tc_mode, c):
    z, m, n, k = c["z"], c["m"], c["n"], c["k"]
    g = _gen(z * 7919 + m * 31 + n * 7 + k)
    ap, ab, an, op, ob, on = _tc_layout(c["layout"], z, m, n, k)
    a = _buf(an)                                              # NaN outside the view: a stray read poisons the result
    av = a.as_strided((z, m, k), (ab, ap, 1))
    av.copy_(torch.randn(z, m, k, device="cuda", generator=g))
    w = torch.randn(z, n, k, device="cuda", generator=g) * 0.1
    w = w * (torch.rand(z, n, k, device="cuda", generator=g) < 0.6)
    bias = torch.rand(z, n, device="cuda", generator=g) * 0.4 - 0.2
    ah, al = _split(K, a)
    wh, wl = _split(K, w)
    out, oh, ol = _tc_run(K, c, a, ah, al, wh, wl, bias)
    out2, oh2, ol2 = _tc_run(K, c, a, ah, al, wh, wl, bias)
    torch.cuda.synchronize()
    ref = torch.einsum("zmk,znk->zmn", av.double(), w.double()) + bias.double()[:, None, :]
    ref = torch.relu(ref) if c["relu"] else ref
    view = lambda t: t.as_strided((z, m, n), (ob, op, 1))   # noqa: E731
    written = torch.zeros(on, dtype=torch.bool, device="cuda")
    view(written).fill_(True)
    for t, t2 in ((out, out2), (oh, oh2), (ol, ol2)):
        if t is not None:
            assert same_bits(t, t2), "two launches differ"
            assert bool(torch.isnan(t[~written]).all()), "wrote outside the output view"
    if out is not None:
        assert C.rel_err(view(out), ref) < TOL_GEMM
    if oh is not None:
        assert tf32_clean(view(oh))
        assert C.rel_err(view(oh) + view(ol), ref) < TOL_GEMM
        if out is not None:
            assert same_value_bits(view(oh) + view(ol), view(out))


def test_tc_rule_reaches_both_kernels_unforced():
    picks = {tc_kernel(c["m"], c["n"], c["z"], "auto", sms()) for c in TC_CASES}
    assert picks == {"1cta", "pair"}, picks


@pytest.mark.parametrize("z,m,n,k", TC_EXACT_SHAPES)
def test_tc_linear_tf32x3_each_product_alone(K, tc_mode, z, m, n, k):
    """Small integers make every product and sum exact: hi*hi, lo*hi and hi*lo each give X Y^T alone; lo*lo is dropped."""
    g = _gen(m + n + k)
    x = torch.randint(-8, 9, (z, m, k), device="cuda", generator=g).float()
    y = torch.randint(-8, 9, (z, n, k), device="cuda", generator=g).float()
    zx, zy, bias = torch.zeros_like(x), torch.zeros_like(y), torch.zeros(z, n, device="cuda")
    prod = torch.einsum("zmk,znk->zmn", x.double(), y.double()).float()
    for name, (ah, al, wh, wl), want in (("hi.hi", (x, zx, y, zy), prod), ("lo.hi", (zx, x, y, zy), prod),
                                         ("hi.lo", (x, zx, zy, y), prod), ("lo.lo", (zx, x, zy, y), torch.zeros_like(prod))):
        out = torch.full((z, m, n), float("nan"), device="cuda")
        _tc_call(K, ah, al, k, m * k, wh, wl, bias, z, m, n, k, False, out, None, None, n, m * n)
        torch.cuda.synchronize()
        assert torch.equal(out, want), name


@pytest.mark.parametrize("signed", [True, False], ids=["signed", "positive"])
@pytest.mark.parametrize("k", [pytest.param(k, marks=_LONG_K_OVER) for k in TC_LONG_K])
def test_tc_linear_tf32x3_long_contraction(K, tc_mode, k, signed):
    """The tensor core truncates as it accumulates; that error grows with K and is largest when nothing cancels."""
    g = _gen(k + signed)
    m = n = 256
    if signed:
        a = torch.randn(1, m, k, device="cuda", generator=g)
        w = torch.randn(1, n, k, device="cuda", generator=g) * 0.05
    else:
        a = torch.rand(1, m, k, device="cuda", generator=g)
        w = torch.rand(1, n, k, device="cuda", generator=g) * 0.05
    bias = torch.zeros(1, n, device="cuda")
    ah, al = _split(K, a)
    wh, wl = _split(K, w)
    out = torch.full((1, m, n), float("nan"), device="cuda")
    _tc_call(K, ah, al, k, m * k, wh, wl, bias, 1, m, n, k, False, out, None, None, n, m * n)
    torch.cuda.synchronize()
    err = C.rel_err(out, torch.einsum("zmk,znk->zmn", a.double(), w.double()))
    _report(f"tf32x3 {m}x{n}x{k} {'signed' if signed else 'positive'} {tc_kernel(m, n, 1, tc_mode, sms())}", rel_err=err)
    assert err < TOL_GEMM


# ---- b) lbbnn_lrt_mc_epilogue, lbbnn_tf32_split_rows, lbbnn_lrt_sample_expand ----------------------------------------------
def _epi_inputs(c, seed):
    g = _gen(seed)
    n, total, off = c["n"], c["B"] * c["N"], c["off"]
    x = {"E": _buf(n * total, off), "S": _buf(n * total, off), "eps": _buf(n * total, off)}
    # every sample's slot holds its own values even when a stride of 0 says only the first may be read
    x["E"].copy_(torch.randn(n * total, device="cuda", generator=g))
    x["S"].copy_(torch.rand(n * total, device="cuda", generator=g) * 0.5)
    x["eps"].copy_(torch.randn(n * total, device="cuda", generator=g))
    x["bias_mu"] = torch.randn(c["N"], device="cuda", generator=g) * 0.1
    x["bias_rho"] = torch.rand(c["N"], device="cuda", generator=g) * 5 - 6
    x["rowscale"] = 1 + 0.3 * torch.randn(n, c["N"], device="cuda", generator=g)
    return x


def _epi_run(K, c, x, outs, eps=None):
    """One launch; eps overrides the configured noise with an injected tensor."""
    n, total, off = c["n"], c["B"] * c["N"], c["off"]
    o = {k: _buf(n * total, off) for k in ("act", "m_hi", "m_lo", "v_hi", "v_lo")}
    if eps is not None:
        noise = K.make_noise(eps)
    elif c["noise"] == "inj":
        noise = K.make_noise(x["eps"])
    elif c["noise"] == "none":
        noise = None
    else:
        noise = K.make_noise(None, SEED, STREAM)
    sample = c["sample"]
    K.check(K.lib.lbbnn_lrt_mc_epilogue(
        K.ptr(x["E"]), total * c["es"], K.ptr(x["S"]) if sample else None, total * c["ss"], K.ptr(x["bias_mu"]),
        K.ptr(x["bias_rho"]) if sample else None, c["B"], c["N"], n, noise, c["gstride"],
        (K.FLAG_SAMPLE if sample else 0) | (K.FLAG_RELU if c["relu"] else 0),
        K.ptr(o["act"]) if "act" in outs else None, K.ptr(x["rowscale"]) if c["rowscale"] else None,
        *((K.ptr(o["m_hi"]), K.ptr(o["m_lo"])) if "m" in outs else (None, None)),
        *((K.ptr(o["v_hi"]), K.ptr(o["v_lo"])) if "v" in outs else (None, None)), K.current_stream()))
    return {k: v.view(n, total) for k, v in o.items()}


def _epi_ref(K, c, x):
    n, total, N = c["n"], c["B"] * c["N"], c["N"]
    per = lambda t, s: t.view(n, total) if s else t.view(n, total)[:1].expand(n, total)   # noqa: E731
    o = per(x["E"], c["es"]).double() + x["bias_mu"].double().repeat(c["B"])
    if c["sample"]:
        if c["noise"] == "inj":
            eps = x["eps"].view(n, total)
        else:
            eps = _philox_stack(K, n, total, STREAM, c["gstride"])
        sb = torch.log1p(torch.exp(x["bias_rho"].double())).repeat(c["B"])
        o = o + torch.sqrt(per(x["S"], c["ss"]).double() + sb * sb) * eps.double()
    act = torch.relu(o) if c["relu"] else o
    z = x["rowscale"].double().repeat(1, c["B"]) if c["rowscale"] else 1.0
    return act, act * z, act * act


def _epi_id(c):
    return ("sample-" if c["sample"] else "mean-") + "e{es}s{ss}-{noise}-".format(**c) + "+".join(c["outs"]) + \
        "-b{B}n{N}-x{n}".format(**c) + "-relu" * c["relu"] + "-z" * c["rowscale"] + "-g" * bool(c["gstride"]) + "-off" * c["off"]


@pytest.mark.parametrize("c", EPI_CASES, ids=_epi_id)
def test_lrt_mc_epilogue(K, c):
    x = _epi_inputs(c, zlib.crc32(_epi_id(c).encode()))
    full = _epi_run(K, c, x, ("act", "m", "v"))
    part = _epi_run(K, c, x, c["outs"])
    torch.cuda.synchronize()
    act_ref, m_ref, v_ref = _epi_ref(K, c, x)
    act = full["act"]
    assert C.rel_err(act, act_ref) < TOL_ELEM
    assert C.rel_err(full["m_hi"] + full["m_lo"], m_ref) < TOL_ELEM
    assert C.rel_err(full["v_hi"] + full["v_lo"], v_ref) < TOL_ELEM
    # the splits are of the fp32 products of the kernel's own act, bit for bit
    z = x["rowscale"].repeat(1, c["B"]) if c["rowscale"] else None
    assert same_value_bits(full["m_hi"] + full["m_lo"], act * z if z is not None else act)
    assert same_value_bits(full["v_hi"] + full["v_lo"], act * act)
    assert tf32_clean(full["m_hi"]) and tf32_clean(full["v_hi"])
    # asking for fewer outputs changes none of them
    for k in ("act",) * ("act" in c["outs"]) + ("m_hi", "m_lo") * ("m" in c["outs"]) + ("v_hi", "v_lo") * ("v" in c["outs"]):
        assert same_bits(part[k], full[k]), k
    if c["noise"][:3] == "nat":       # native noise is the exported Philox stream of sample s: stream + s * group stride
        eps = _buf(c["n"] * c["B"] * c["N"], c["off"])
        eps.copy_(_philox_stack(K, c["n"], c["B"] * c["N"], STREAM, c["gstride"]).view(-1))
        inj = _epi_run(K, c, x, ("act", "m", "v"), eps=eps)
        for k in full:
            assert same_bits(inj[k], full[k]), k


def _split_id(c):
    return "r{rows}c{cols}-x{n}-{xs}-{outs}".format(**c) + "-z" * c["rowscale"] + "-off" * c["off"]


def split_rows_stride(c):
    total = c["rows"] * c["cols"]
    return {"shared": 0, "dense": total, "pad8": total + 8, "pad5": total + 5}[c["xs"]]


@pytest.mark.parametrize("c", SPLIT_CASES, ids=_split_id)
def test_tf32_split_rows(K, c):
    g = _gen(c["rows"] * 131 + c["cols"] + c["n"])
    n, total, xs, off = c["n"], c["rows"] * c["cols"], split_rows_stride(c), c["off"]
    x = _buf(max(xs, total) * n + total, off)
    x.copy_(torch.randn(x.numel(), device="cuda", generator=g) * torch.exp(torch.randn(x.numel(), device="cuda", generator=g) * 4))
    rs = torch.randn(n, c["cols"], device="cuda", generator=g) if c["rowscale"] else None
    o = {k: _buf(n * total, off) for k in ("hi", "lo", "sq_hi", "sq_lo")}
    want_hi, want_sq = c["outs"] in ("hi", "both"), c["outs"] in ("sq", "both")
    K.check(K.lib.lbbnn_tf32_split_rows(K.ptr(x), xs, c["rows"], c["cols"], n, K.ptr(rs, True),
                                        *((K.ptr(o["hi"]), K.ptr(o["lo"])) if want_hi else (None, None)),
                                        *((K.ptr(o["sq_hi"]), K.ptr(o["sq_lo"])) if want_sq else (None, None)),
                                        K.current_stream()))
    torch.cuda.synchronize()
    xv = x.as_strided((n, total), (xs, 1))
    if want_hi:
        m = xv * rs.repeat(1, c["rows"]) if rs is not None else xv
        assert same_value_bits(o["hi"].view(n, total) + o["lo"].view(n, total), m) and tf32_clean(o["hi"])
    else:
        assert bool(torch.isnan(o["hi"]).all())
    if want_sq:
        assert same_value_bits(o["sq_hi"].view(n, total) + o["sq_lo"].view(n, total), xv * xv) and tf32_clean(o["sq_hi"])
    else:
        assert bool(torch.isnan(o["sq_hi"]).all())


@pytest.mark.parametrize("c", EXPAND_CASES, ids=lambda c: "b{B}n{N}-x{n}-{noise}".format(**c) + "-relu" * c["relu"] +
                         "-g" * bool(c["gstride"]) + "-off" * c["off"])
def test_lrt_sample_expand(K, c):
    g = _gen(c["B"] * 17 + c["N"] + c["n"])
    n, total, off = c["n"], c["B"] * c["N"], c["off"]
    e, var, eps = _buf(total, off), _buf(total, off), _buf(n * total, off)
    e.copy_(torch.randn(total, device="cuda", generator=g))
    var.copy_(torch.rand(total, device="cuda", generator=g) * 0.5)
    eps.copy_(torch.randn(n * total, device="cuda", generator=g))

    def run(noise):
        act = _buf(n * total, off)
        K.check(K.lib.lbbnn_lrt_sample_expand(K.ptr(e), K.ptr(var), c["B"], c["N"], n, noise, c["gstride"],
                                              K.FLAG_RELU if c["relu"] else 0, K.ptr(act), K.current_stream()))
        return act.view(n, total)

    if c["noise"] == "inj":
        act, ref_eps = run(K.make_noise(eps)), eps.view(n, total)
    else:
        act = run(K.make_noise(None, SEED, STREAM))
        ref_eps = _philox_stack(K, n, total, STREAM, c["gstride"])
        eps.copy_(ref_eps.view(-1))
        assert same_bits(run(K.make_noise(eps)), act)
    torch.cuda.synchronize()
    ref = e.double() + torch.sqrt(var.double()) * ref_eps.double()
    assert C.rel_err(act, torch.relu(ref) if c["relu"] else ref) < TOL_ELEM


# ---- c) CUDA-core MC kernels ------------------------------------------------------------------------------------------------
def sgemm_x_stride(kind, m, k):
    return {"shared": 0, "per": m * k, "odd": m * k + 1}[kind]


@pytest.mark.parametrize("n,m,k,o,xs,relu", SGEMM_CASES)
def test_linear_f32_batched(K, n, m, k, o, xs, relu):
    g = _gen(n * 1000 + m + k + o)
    stride = sgemm_x_stride(xs, m, k)
    x = torch.rand(max(stride, 0) * (n - 1) + m * k, device="cuda", generator=g)
    w = torch.randn(n, o, k, device="cuda", generator=g) * 0.2
    w = w * (torch.rand(n, o, k, device="cuda", generator=g) < 0.6)
    b = torch.randn(n, o, device="cuda", generator=g) * 0.1
    out = torch.full((n, m, o), float("nan"), device="cuda")
    K.check(K.lib.lbbnn_linear_f32_batched(K.ptr(x), stride, K.ptr(w), K.ptr(b), n, m, k, o, K.FLAG_RELU if relu else 0,
                                           K.ptr(out), K.current_stream()))
    torch.cuda.synchronize()
    xv = x.as_strided((n, m, k), (stride, k, 1))
    ref = torch.einsum("smk,sok->smo", xv.double(), w.double()) + b.double()[:, None, :]
    assert C.rel_err(out, torch.relu(ref) if relu else ref) < TOL_GEMM


def test_linear_f32_batched_sample_limit(K):
    n, m, k, o = 65535, 3, 4, 2
    g = _gen(65535)
    x = torch.rand(m, k, device="cuda", generator=g)
    w = torch.randn(n, o, k, device="cuda", generator=g)
    b = torch.randn(n, o, device="cuda", generator=g)
    out = torch.full((n, m, o), float("nan"), device="cuda")
    K.check(K.lib.lbbnn_linear_f32_batched(K.ptr(x), 0, K.ptr(w), K.ptr(b), n, m, k, o, 0, K.ptr(out), K.current_stream()))
    torch.cuda.synchronize()
    ref = torch.einsum("mk,sok->smo", x.double(), w.double()) + b.double()[:, None, :]
    assert C.rel_err(out, ref) < TOL_GEMM
    with pytest.raises(K.LbbnnError):
        K.check(K.lib.lbbnn_linear_f32_batched(K.ptr(x), 0, K.ptr(w), K.ptr(b), n + 1, m, k, o, 0, K.ptr(out),
                                               K.current_stream()))


def _accum_ref(logits):
    """log_softmax and the row-normalised expit of it, summed over samples (dim 0), in float64."""
    lp = logits - torch.logsumexp(logits, -1, keepdim=True)
    e = torch.sigmoid(lp)
    return lp.sum(0), (e / e.sum(-1, keepdim=True)).sum(0)


def _start_sums(g, b, c):
    return (torch.randn(b, c, device="cuda", generator=g, dtype=torch.float64),
            torch.rand(b, c, device="cuda", generator=g, dtype=torch.float64) * 3)


def head_stride(c):
    return {"shared": 0, "dense": c["B"] * c["K"], "padded": c["B"] * c["K"] + 8}[c["hs"]]


@pytest.mark.parametrize("c", HEAD_CASES, ids=lambda c: "C{C}-B{B}-K{K}-x{n}-{hs}".format(**c))
def test_mc_head_accumulate(K, c):
    C_, B, k, n, hs = c["C"], c["B"], c["K"], c["n"], head_stride(c)
    g = _gen(C_ * 100003 + B * 7 + k)
    h = torch.rand(hs * (n - 1) + B * k, device="cuda", generator=g)
    w = torch.randn(n, C_, k, device="cuda", generator=g) * 0.2
    b = torch.randn(n, C_, device="cuda", generator=g) * 0.5
    lp0, pr0 = _start_sums(g, B, C_)
    lp, pr = lp0.clone(), pr0.clone()
    counter = torch.tensor([41], dtype=torch.int64, device="cuda")
    K.check(K.lib.lbbnn_mc_head_accumulate(K.ptr(h), hs, K.ptr(w), K.ptr(b), n, B, k, C_, K.ptr(lp, torch.float64),
                                           K.ptr(pr, torch.float64), K.ptr(counter, torch.int64), K.current_stream()))
    torch.cuda.synchronize()
    hv = h.as_strided((n, B, k), (hs, k, 1))
    dlp, dpr = _accum_ref(torch.einsum("sbk,sck->sbc", hv.double(), w.double()) + b.double()[:, None, :])
    assert C.rel_err(lp - lp0, dlp) < TOL_ACC and C.rel_err(lp, lp0 + dlp) < TOL_ACC
    assert C.rel_err(pr - pr0, dpr) < TOL_ACC and C.rel_err(pr, pr0 + dpr) < TOL_ACC
    assert int(counter) == 41 + n


def test_mc_head_accumulate_refusals(K):
    """Host-side checks: nothing is launched."""
    t = torch.zeros(4096, device="cuda")
    d = torch.zeros(64, dtype=torch.float64, device="cuda")

    def call(k, classes, hs=0):
        K.check(K.lib.lbbnn_mc_head_accumulate(K.ptr(t), hs, K.ptr(t), K.ptr(t), 1, 1, k, classes, K.ptr(d, torch.float64),
                                               K.ptr(d, torch.float64), None, K.current_stream()))
    assert head_fits(16, head_kmax(16)) and not head_fits(16, head_kmax(16) + 4)
    for args in ((8, 17), (6, 10), (head_kmax(16) + 4, 16), (8, 10, 2)):
        with pytest.raises(K.LbbnnError):
            call(*args)


@pytest.mark.parametrize("classes,b,n,counter", ACC_CASES)
def test_mc_accumulate_batched(K, classes, b, n, counter):
    g = _gen(classes * 1000 + b)
    logits = torch.randn(n, b, classes, device="cuda", generator=g) * 3
    lp0, pr0 = _start_sums(g, b, classes)
    lp, pr = lp0.clone(), pr0.clone()
    cnt = torch.tensor([7], dtype=torch.int64, device="cuda")
    K.check(K.lib.lbbnn_mc_accumulate_batched(K.ptr(logits), n, b, classes, K.ptr(lp, torch.float64), K.ptr(pr, torch.float64),
                                              K.ptr(cnt, torch.int64) if counter else None, K.current_stream()))
    torch.cuda.synchronize()
    dlp, dpr = _accum_ref(logits.double())
    assert C.rel_err(lp - lp0, dlp) < TOL_ACC and C.rel_err(lp, lp0 + dlp) < TOL_ACC
    assert C.rel_err(pr - pr0, dpr) < TOL_ACC and C.rel_err(pr, pr0 + dpr) < TOL_ACC
    assert int(cnt) == 7 + n * counter


@pytest.mark.parametrize("out,inp,n,first", SAMPLE_CASES)
def test_mc_sample(K, out, inp, n, first):
    g = _gen(out * inp + n)
    mu = torch.rand(out, inp, device="cuda", generator=g) * 0.4 - 0.2
    rho = torch.rand(out, inp, device="cuda", generator=g) * 3 - 5
    lam = torch.randn(out, inp, device="cuda", generator=g) * 2
    bmu = torch.randn(out, device="cuda", generator=g) * 0.1
    brho = torch.rand(out, device="cuda", generator=g) * 3 - 5
    st = K.current_stream()
    sig, alp, bsig = torch.empty_like(rho), torch.empty_like(lam), torch.empty_like(brho)
    K.check(K.lib.lbbnn_mc_prepare(K.make_layer(mu, rho, lam, bmu, brho), K.ptr(sig), K.ptr(alp), K.ptr(bsig), st))
    first_dev = torch.tensor([first], dtype=torch.int64, device="cuda")
    seed, base, stride = SEED, SAMPLE_STREAM_BASE, SAMPLE_STREAM_STRIDE

    def draw(prepared, split):
        L = K.make_layer(mu, sig, alp, bmu, bsig) if prepared else K.make_layer(mu, rho, lam, bmu, brho)
        w, lo, b = (torch.full((n, out, inp), float("nan"), device="cuda"), torch.full((n, out, inp), float("nan"), device="cuda"),
                    torch.full((n, out), float("nan"), device="cuda"))
        if split is None:
            K.check(K.lib.lbbnn_mc_sample(L, n, K.ptr(first_dev, torch.int64), seed, base, stride, K.ptr(w), K.ptr(b), st))
        else:
            K.check(K.lib.lbbnn_mc_sample_split(L, n, K.ptr(first_dev, torch.int64), seed, base, stride, prepared,
                                                K.ptr(w), K.ptr(lo) if split else None, K.ptr(b), st))
        return w, lo, b

    w0, _, b0 = draw(0, None)
    draws = [draw(p, s) for p in (0, 1) for s in (False, True)]
    torch.cuda.synchronize()
    assert C.rel_err(sig, torch.log1p(torch.exp(rho.double()))) < TOL_ELEM
    assert C.rel_err(alp, torch.sigmoid(lam.double())) < TOL_ELEM
    assert C.rel_err(bsig, torch.log1p(torch.exp(brho.double()))) < TOL_ELEM
    for (w, lo, b), (p, s) in zip(draws, itertools.product((0, 1), (False, True))):
        assert same_bits(b, b0), (p, s)
        assert same_value_bits(w + lo, w0) if s else same_bits(w, w0), (p, s)
        if s:
            assert tf32_clean(w)
    # the reference draws: the exported Philox streams of sample first + s, masks from the kernel's own fp32 alpha
    numel = out * inp
    u, e, eb = [], [], []
    for s in range(n):
        sid = base + (first + s) * stride
        u.append(K.philox_uniform(numel, seed, sid).view(out, inp))
        e.append(K.philox_normal(numel, seed, sid + 1).view(out, inp))
        eb.append(K.philox_normal(out, seed, sid + 2))
    u, e, eb = torch.stack(u), torch.stack(e), torch.stack(eb)
    mask = u < alp
    assert torch.equal(w0 != 0, mask)
    assert C.rel_err(w0, mask * (mu.double() + sig.double() * e.double())) < TOL_ELEM
    assert C.rel_err(b0, bmu.double() + bsig.double() * eb.double()) < TOL_ELEM
