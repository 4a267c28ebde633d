"""Host-only checks for tests/test_layer_kernels_gpu.py, no GPU needed: by the launch rules restated there (split counts,
ZRED grid, elementwise grid, auxiliary row slices), the GPU file's configuration tables still reach every launch path of the
fp32 LRT layer kernels and the MNF auxiliary kernels at 148 SMs.  An edited table that silently drops a path fails here."""
import cases as C  # noqa: F401  (sets sys.path)
import test_layer_kernels_gpu as G

SMS = 148


def test_launch_rules_match_the_documented_examples():
    assert G.fwd_split(100, 784, 400) == (3, 17)
    assert G.fwd_split(100, 400, 10) == (3, 9)
    assert G.fwd_split(7, 4096, 3) == (2, 128)
    assert G.fwd_split(1024, 100, 1216)[1] == 1
    assert G.elementwise_blocks(8 * 4096) == 32 and G.elementwise_blocks(1) == 1 and G.elementwise_blocks(10 ** 8) == 16 * SMS
    assert G.finalize_launch(784, 400, True) == ("zred", 7 * 25)
    assert G.finalize_launch(33, 7, True)[0] == "elem" and G.finalize_launch(784, 400, False)[0] == "elem"
    assert G.aux_slices(784, 400) == 7 and G.aux_slices(33, 13) == 1 and G.aux_slices(300, 700) == 11
    assert G.aux_slices(20, 5, forced=16) == 16


def _fwd_rows():
    for c in G.FWD_CASES:
        B, K, N = c["B"], c["K"], c["N"]
        cps, s = G.fwd_split(B, K, N, SMS)
        tiles = G.cdiv(B, G.F_BM) * G.cdiv(N, G.F_BN)
        yield c, cps, s, tiles, G.cdiv(K, G.F_BK)


def test_forward_table_reaches_every_split():
    rows = list(_fwd_rows())
    splits = {s for _, _, s, _, _ in rows}
    assert any(s == 1 and tiles >= SMS for _, _, s, tiles, _ in rows)                 # the tiles fill the GPU
    assert any(s == 1 and tiles < SMS and c["K"] <= 47 for c, _, s, tiles, _ in rows)  # the chunk cap
    assert set(range(2, 9)) <= splits
    eight_k1 = {s for s in splits if s > 1 and s % G.EPI_BATCH == 1}
    assert len(eight_k1) >= 2                                                           # 8k+1: the last pass reads one split
    assert max(splits) >= 128
    assert any(s > 1 and chunks % cps for _, cps, s, _, chunks in rows)                 # ragged last split
    assert any(c["K"] % G.F_BK for c in G.FWD_CASES)                                    # ragged last chunk
    assert any(c["B"] % G.F_BM for c in G.FWD_CASES) and any(c["N"] % G.F_BN for c in G.FWD_CASES)
    assert any(c["B"] > G.F_BM and c["B"] % G.F_BM for c in G.FWD_CASES)
    assert any(c["N"] > G.F_BN and c["N"] % G.F_BN for c in G.FWD_CASES)


def test_forward_table_reaches_every_load_flag_and_noise_path():
    fc = G.FWD_CASES
    assert any(c["K"] % 4 == 0 and c["off"] == 0 for c in fc)                           # vector loads
    assert any(c["K"] % 4 == 0 and c["off"] == 1 and c["mv"] for c in fc)               # scalar loads at +1 float (x, M/V, outputs)
    assert any(c["K"] % 4 for c in fc)
    assert any(c["B"] * c["N"] % 4 == 0 and c["off"] == 1 for c in fc)                  # scalar epilogue with whole quads
    assert {c["sample"] for c in fc} == {True, False} and {c["relu"] for c in fc} == {True, False}
    assert any(c["kl"] and not c["sample"] for c in fc) and any(c["kl"] and c["sample"] for c in fc)
    cap = 16 * SMS
    assert any(c["kl"] and G.cdiv(G.cdiv(c["N"] * c["K"], 4), 256) > cap for c in fc)   # KL partial count capped
    assert any(c["moments"] for c in fc) and any(c["moments"] and c["mv"] for c in fc)
    assert {c["mv"] for c in fc} == {True, False} and any(c["mv"] and not c["sample"] for c in fc)
    assert {c["noise"] for c in fc} == {"inj", "nat"}
    nat_groups = [c for c in fc if c["noise"] == "nat" and c["gstride"]]
    assert nat_groups and any(c["B"] % c["rpg"] for c in nat_groups)                   # row groups, ragged last group
    assert any(c["noise"] == "nat" and not c["gstride"] for c in fc)
    assert all(c["rpg"] * c["N"] % 4 == 0 for c in nat_groups)
    rs = [c for c in fc if c["rowscale"]]
    assert {c["rs_off"] for c in rs} == {0, 1} and any(c["B"] % c["rpg"] for c in rs)
    assert any(c["K"] % 4 == 0 and c["rs_off"] == 0 and c["off"] == 0 for c in rs)       # vector row-scale loads
    assert {c["z"] for c in fc} >= {"none", "z", "zkl"}
    assert any(c["z"] != "none" and c["var"] == "exact" for c in fc) and any(c["z"] != "none" and c["var"] == "reference" for c in fc)
    assert any(c["z"] != "none" and c["pri"] != "default" and c["kl"] for c in fc)
    pro = G.PRO_CASES
    assert {z for _, _, z, *_ in pro} == {"none", "z", "zkl", "klonly"} and {s for *_, s in pro} == {True, False}
    assert any(G.cdiv(G.cdiv(n * k, 4), 256) > cap for k, n, *_ in pro)


def test_backward_tables_reach_every_path():
    bw = G.BWDW_CASES
    assert any(c["B"] % G.W_BB and c["N"] % G.W_BN and c["K"] % G.W_BK for c in bw)
    assert any(c["B"] % G.W_BB == 0 and c["N"] % G.W_BN == 0 and c["K"] % G.W_BK == 0 for c in bw)
    assert any(c["K"] % 4 == 0 and c["N"] % 4 == 0 and c["off"] == 0 for c in bw)       # vector loads
    assert any(c["K"] % 4 == 0 and c["N"] % 4 == 0 and c["off"] == 1 for c in bw)       # ... off by alignment
    assert any(c["N"] > G.W_BN and c["K"] > G.W_BK for c in bw)                        # bias sums from k-tile 0 of many
    launches = {G.finalize_launch(c["K"], c["N"], c["req"] != "none")[0] for c in bw if c["z"] != "none"}
    assert launches == {"zred", "elem"}
    assert {c["req"] for c in bw} == {"none", "dz", "dzkl", "both"}
    assert {c["klg"] for c in bw} == {"0", "host", "dev"} and {c["acc"] for c in bw} == {True, False}
    assert {c["sample"] for c in bw} == {True, False} and {c["var"] for c in bw} == {"reference", "exact"}

    dx = G.DX_CASES
    sp = [(c, *G.dx_split(c["B"], c["K"], c["N"], SMS)) for c in dx]
    tiles = lambda c: G.cdiv(c["B"], G.X_BM) * G.cdiv(c["K"], G.X_BK)  # noqa: E731
    assert any(s == 1 and tiles(c) >= SMS for c, _, s in sp)
    assert any(s == 1 and tiles(c) < SMS for c, _, s in sp)
    assert 9 in {s for *_, s in sp}
    assert any(s > 2 * G.EPI_BATCH for *_, s in sp)                                     # the epilogue's second pass
    assert any(s > 1 and G.cdiv(c["N"], G.X_BN) % cps for c, cps, s in sp)              # ragged last split
    assert {c["mv"] for c in dx} == {True, False} and {c["mask"] for c in dx} == {True, False}
    assert {c["acc"] for c in dx} == {True, False} and {c["sample"] for c in dx} == {True, False}
    assert any(c["K"] % 4 == 0 and c["off"] == 1 for c in dx) and any(c["K"] % 4 == 0 and c["off"] == 0 for c in dx)
    assert any(c["K"] % G.X_BK for c in dx) and any(c["B"] % G.X_BM for c in dx)


def test_finalize_table_reaches_every_path():
    fin = G.FIN_CASES
    zred = [c for c in fin if c["z"] != "none" and G.finalize_launch(c["K"], c["N"], c["req"] != "none")[0] == "zred"]
    assert any((c["K"] // 4) % G.Z_QUADS for c in zred)                                # ragged column block
    assert any((c["K"] // 4) % G.Z_QUADS and c["K"] // 4 > G.Z_QUADS for c in zred)    # ... after whole ones
    assert any((c["K"] // 4) % G.Z_QUADS == 0 for c in zred)
    assert any(c["N"] % G.Z_ROWS for c in zred) and any(c["N"] % G.Z_ROWS == 0 for c in zred)
    assert any(c["off"] == 1 for c in zred) and any(c["acc"] for c in zred)
    elem_z = [c for c in fin if c["z"] != "none" and c["K"] % 4]
    assert elem_z and any(c["N"] > 1 for c in elem_z)                                  # quads straddle weight rows
    assert {c["req"] for c in elem_z} >= {"dz", "dzkl", "both"}
    assert {c["req"] for c in zred} >= {"dz", "dzkl", "both"}
    assert any(c["z"] != "none" and c["req"] == "none" for c in fin)
    assert any(c["z"] == "zkl" and c["req"] == "dz" for c in fin)                      # KL share routed into dz
    assert any(c["z"] == "klonly" for c in fin)
    assert {c["klg"] for c in fin} == {"0", "host", "dev"} and {c["sample"] for c in fin} == {True, False}
    assert any(c["acc"] and c["z"] == "none" for c in fin) and {c["var"] for c in fin} == {"reference", "exact"}
    assert any(G.cdiv(c["N"] * c["K"], 4) > 16 * SMS * 256 for c in fin)               # grid-stride loop
    ad = G.ADAM_CASES
    assert {v for _, _, v, _, _ in ad} == {"reference", "exact"} and {s for *_, s, _ in ad} == {True, False}
    assert {k for *_, k in ad} == {"0", "host", "dev"}
    assert any((k * n) % 4 for k, n, *_ in ad) and any((k * n) % 4 == 0 and k % 4 == 0 for k, n, *_ in ad)


def test_aux_tables_reach_every_path():
    fw = G.AUX_FWD_CASES
    assert any(o < 8 for _, o in fw) and any(o % 8 for _, o in fw) and any(o >= 100 for _, o in fw)
    assert any(d < 32 for d, _ in fw) and any(d % 256 and d > 256 for d, _ in fw) and any(d % 256 == 0 for d, _ in fw)
    bw = G.AUX_BWD_CASES
    default = [G.aux_slices(d, o, SMS) for d, o, f in bw if f is None]
    assert 1 in default and any(s > 1 for s in default)
    forced = [(d, o, f) for d, o, f in bw if f is not None]
    assert {1, 3} <= {f for *_, f in forced}
    assert any(f > o for _, o, f in forced)                                             # empty row slices
    assert any(f > 1 and G.cdiv(o, f) * (f - 1) >= o for _, o, f in forced)            # ... including the last
    assert any(d % 32 for d, _, _ in bw) and any(d > 256 for d, _, _ in bw)
    dr = G.DRAW_CASES
    assert {n for *_, n, _ in dr} == {"inj", "nat"} and {r for *_, r in dr} == {True, False}
    assert {r for r, *_ in dr} == {1, 3} and any(n == "nat" and r for *_, n, r in dr)
    db = G.DRAW_BWD_CASES
    assert {-1, 0} <= {k for _, _, k, _ in db} and any(k == r - 1 and r > 1 for r, _, k, _ in db)
    assert {a for *_, a in db} == {True, False} and any(k >= 0 and not a for _, _, k, a in db)
    rows = G.ROWS_CASES
    assert {("dld",), ("rows",), ("dld", "rows")} <= set(rows)
    assert all(any(f"no_{n}" in r for r in rows) for n in ("a", "b", "dzk")) and 1 in G.ROWS_D


def test_mnf_sweep_shapes_are_not_in_the_golden_file():
    import numpy as np
    import os
    g = np.load(os.path.join(C.GOLDEN, "mnf_layer.npz"))
    golden = {tuple(int(v) for v in g[k][1:4]) for k in g.files if k.endswith("_meta")}
    sweep = {(b, i, o) for b, i, o, _ in G.MNF_SWEEP}
    assert not sweep & golden
    assert (1, 33, 7) in sweep and any(b > 128 for b, *_ in sweep) and any(i == 784 and p != "default" for _, i, _, p in G.MNF_SWEEP)
