"""Host-only checks for tests/test_predict_kernels_gpu.py and the tf32x3 entry point, no GPU needed:
  * the GPU file's configuration tables still reach every launch path of the posterior-predictive kernels at 148 SMs, by
    the launch rules restated there (an edited table that silently drops a path fails here);
  * lbbnn_tc_linear_tf32x3 refuses outputs its float4 epilogue cannot store to, before it touches the device (integer fake
    pointers: nothing is dereferenced)."""
import itertools

import pytest

import cases as C  # noqa: F401  (sets sys.path)
import test_predict_kernels_gpu as G

SMS = 148


def _tc_launches():
    for c, mode in itertools.product(G.TC_CASES, ("1cta", "pair", "auto")):
        yield c, mode, G.tc_kernel(c["m"], c["n"], c["z"], mode, SMS)


def test_tf32x3_table_reaches_every_path():
    launches = list(_tc_launches())
    assert {k for c, mode, k in launches if mode == "auto"} == {"1cta", "pair"}
    for kernel in ("1cta", "pair"):
        runs = [c for c, _, k in launches if k == kernel]
        per_cta = [G.tc_tiles_per_cta(c["m"], c["n"], c["z"], kernel, SMS) for c in runs]
        assert max(per_cta) >= 3, kernel              # the second use of each TMEM accumulator buffer
        # a CTA whose later tile lies in another batch z than its first
        grid = SMS // 2 if kernel == "pair" else SMS
        rows = 2 * G.TC_BM if kernel == "pair" else G.TC_BM
        crosses = False
        for c in runs:
            per_z = G.cdiv(c["m"], rows) * G.cdiv(c["n"], G.TC_BN)
            tiles = per_z * c["z"]
            crosses |= any(b // per_z != (b + grid) // per_z for b in range(min(grid, tiles)) if b + grid < tiles)
        assert crosses, kernel
        # K blocks: fewer than one stage ring, a ring that wraps inside a tile, and K < 32 / ragged last block
        kbs = {G.cdiv(c["k"], G.TC_BK) for c in runs}
        assert min(kbs) == 1 and any(kb % G.TC_STAGES[kernel] for kb in kbs)
    pair_m = {c["m"] for c, _, k in launches if k == "pair"}
    assert any(0 < m % 256 <= 128 for m in pair_m)     # the last pair tile's second CTA wholly past M
    assert any(m % 256 > 128 for m in pair_m)          # ... partly past M
    ms, ns, ks = ({c[d] for c in G.TC_CASES} for d in "mnk")
    assert {1, 127, 128, 129, 255, 257} <= ms and {1, 15, 16, 17, 65, 129} <= ns and {4, 8, 28, 36, 100} <= ks
    assert any(G.cdiv(k, G.TC_BK) % 3 and G.cdiv(k, G.TC_BK) % 4 for k in ks)
    assert {c["outs"] for c in G.TC_CASES} == {"out", "hilo", "both"} and {c["relu"] for c in G.TC_CASES} == {False, True}
    # epilogue stores: float4, the scalar tail of a ragged 16-column chunk, scalar pitches, warps whose columns are all past N
    layouts = [(c, G._tc_layout(c["layout"], c["z"], c["m"], c["n"], c["k"])) for c in G.TC_CASES]
    vec_pitch = [c for c, (_, _, _, op, ob, _) in layouts if op % 4 == 0 and ob % 4 == 0]
    assert any(c["n"] >= 16 for c in vec_pitch) and any(c["n"] % 16 for c in vec_pitch)
    assert any(op % 4 for c, (_, _, _, op, _, _) in layouts)
    assert any(ob % 4 and op % 4 == 0 and c["z"] > 1 for c, (_, _, _, op, ob, _) in layouts)
    assert any(c["n"] <= 64 for c in G.TC_CASES)
    assert {c["layout"] for c in G.TC_CASES} == {"dense", "pad", "chain"}
    assert any(ab != c["m"] * ap for c, (ap, ab, _, _, _, _) in layouts)
    assert len({shape[1] for shape in G.TC_EXACT_SHAPES} & {129, 257}) == 2


def test_epilogue_table_reaches_every_path():
    cases = G.EPI_CASES
    combos = {(c["sample"], c["es"], c["ss"], G.noise_path(c["B"] * c["N"], c["noise"]), c["outs"]) for c in cases}
    outs = [o for r in (1, 2, 3) for o in itertools.combinations(("act", "m", "v"), r)]
    for sample in (True, False):
        for es, ss in (itertools.product((0, 1), (0, 1)) if sample else ((0, 0), (1, 0))):
            for noise in (("inj", "nat4", "nat1") if sample else ("none",)):
                for o in outs:
                    assert (sample, es, ss, noise, o) in combos
    assert {G.elementwise_vector(c["B"] * c["N"], c["off"]) for c in cases} == {False, True}
    assert any(not G.elementwise_vector(c["B"] * c["N"], c["off"]) and c["B"] * c["N"] % 4 == 0 for c in cases)
    assert any(G.grid_stride(c["n"] * G.cdiv(c["B"] * c["N"], 4), SMS) for c in cases)
    assert {c["relu"] for c in cases} == {False, True} and {c["n"] for c in cases} == {1, 3, 17}
    assert {bool(c["rowscale"]) for c in cases if "m" in c["outs"]} == {False, True}
    assert any(c["rowscale"] and not c["sample"] for c in cases)
    assert {bool(c["gstride"]) for c in cases if c["noise"][:3] == "nat"} == {False, True}


def test_split_rows_and_expand_tables_reach_every_path():
    sc = G.SPLIT_CASES
    assert {c["xs"] for c in sc} == {"shared", "dense", "pad8", "pad5"}
    assert {c["outs"] for c in sc} == {"hi", "sq", "both"} and {c["rowscale"] for c in sc} == {False, True}
    assert any(c["rows"] * c["cols"] % 4 for c in sc)
    assert {G.elementwise_vector(c["rows"] * c["cols"], c["off"]) for c in sc} == {False, True}
    assert any(G.grid_stride(c["n"] * G.cdiv(c["rows"] * c["cols"], 4), SMS) for c in sc)
    ec = G.EXPAND_CASES
    assert {G.noise_path(c["B"] * c["N"], c["noise"]) for c in ec} == {"inj", "nat4", "nat1"}
    assert {c["relu"] for c in ec} == {False, True} and {c["off"] for c in ec} == {0, 1}


def test_cuda_core_tables_reach_every_path():
    tiles = {o: G.sgemm_tile(o) for _, _, _, o, _, _ in G.SGEMM_CASES}
    assert set(tiles.values()) == {64, 128}
    for lo, hi in ((64, 65), (128, 129), (192, 193), (448, 449)):
        assert lo in tiles and hi in tiles and tiles[lo] != tiles[hi]
    ks = {k for _, _, k, _, _, _ in G.SGEMM_CASES}
    assert any(k % 4 for k in ks) and any(k < 16 for k in ks) and any(k % 16 and k % 4 == 0 for k in ks)
    assert any(m % 128 for _, m, _, _, _, _ in G.SGEMM_CASES)
    assert {xs for *_, xs, _ in G.SGEMM_CASES} == {"shared", "per", "odd"}
    assert any(xs == "odd" and k % 4 == 0 and n > 1 for n, _, k, _, xs, _ in G.SGEMM_CASES)   # vector loads off for some samples
    assert {r for *_, r in G.SGEMM_CASES} == {False, True}

    hc = G.HEAD_CASES
    assert {c["C"] for c in hc} == set(range(1, 17))
    assert {1, 7, 8, 9, 1000} <= {c["B"] for c in hc} and {1, 2, 3, 4, 5, 33} <= {c["n"] for c in hc}
    assert {4, 124, 128, 132} <= {c["K"] for c in hc} and G.head_kmax(16) == 584
    assert any(c["C"] == 16 and c["K"] == 584 for c in hc)
    assert all(G.head_fits(c["C"], c["K"]) for c in hc)
    assert {c["hs"] for c in hc} == {"shared", "dense", "padded"}
    assert {c for c, *_ in G.ACC_CASES} >= {1, 10, 31, 32, 33, 100}
    assert {cnt for *_, cnt in G.ACC_CASES} == {False, True}

    caps = [(G.cdiv(G.cdiv(o * i, 4), 256), max(1, 8 * SMS // n)) for o, i, n, _ in G.SAMPLE_CASES]
    assert any(need > cap for need, cap in caps)                                   # grid-stride loop
    assert any(o * i % 4 for o, i, _, _ in G.SAMPLE_CASES) and any(f for *_, f in G.SAMPLE_CASES)


def test_tf32x3_refuses_misaligned_outputs():
    """Both output pitches multiples of 4 mean float4 stores: every requested output must be 16-byte aligned.  The check
    runs before any CUDA call, and the fake A operand is unaligned too, so that no build of the library can launch."""
    from lbbnn import _capi as K
    base = 1 << 32

    def call(out=None, hi=None, lo=None, pitch=16, bstride=16 * 128, a=base + 4):
        K.check(K.lib.lbbnn_tc_linear_tf32x3(a, a, 16, 0, base, base, base, 1, 128, 16, 16, 0, out, hi, lo, pitch, bstride,
                                             None))

    for outs in ((base + 4, None, None), (None, base + 8, base), (None, base, base + 12), (base + 4, base, base)):
        with pytest.raises(K.LbbnnError, match="outputs must be 16-byte aligned"):
            call(*outs)
    with pytest.raises(K.LbbnnError, match="outputs must be 16-byte aligned"):
        call(base + 4, pitch=20, bstride=0)
    # scalar stores (a pitch that is not a multiple of 4) take any address; the unaligned A stops the call later
    for pitch, bstride in ((17, 17 * 128), (16, 18 * 128 + 2)):
        with pytest.raises(K.LbbnnError) as e:
            call(base + 4, base + 4, base + 8, pitch=pitch, bstride=bstride)
        assert "outputs must be" not in str(e.value)
