"""Pins the CPU oracle (oracle/cn_oracle.c and the numpy restatement) to the reference.

Two anchors:
  1. the committed golden fixtures in tests/golden/ -- outputs of the reference's own object code
     (src/cn.c + src/raster.c compiled unmodified, see tests/golden/make_golden.py);
  2. that same object code run live (oracle/_ref/libgcn10_ref.so travels with the repo), on
     seeded random geometries.
Everything is integer/byte work: comparisons are exact.
"""
import os

import numpy as np
import pytest

from gcn10_b200 import synth
from tests import lookups
from oracle import oracle as O
from tests import golden_io
from tests.cases import SMALL_CASES, make_block, PX, PX_VRT, HSG_PX

BLOCKS = golden_io.block_cases()


@pytest.mark.parametrize("name", sorted(BLOCKS))
def test_restatement_matches_golden_blocks(name, port, tables, lookup_dir):
    c = BLOCKS[name]
    esa, gt, hsg, sgt = golden_io.window_inputs(port, c)
    assert np.array_equal(np.array(gt), c["gt"]), "clipped geotransform differs from the reference's"
    got = port.block_rows(esa, gt, hsg, sgt, tables)
    assert got.shape == c["planes"].shape
    assert np.array_equal(got, c["planes"])
    # Port.run_block, the stand-in for process_block() where oracle/_ref is not built: the same block from the whole
    # rasters, and a bbox west of the land cover skipped
    r = port.run_block(c["esa"], c["esa_t"], c["hsg"], c["hsg_t"], c["bbox"], lookup_dir)
    assert (r["nplanes"], r["gt"]) == (18, gt) and np.array_equal(r["planes"], c["planes"])
    t0, t3 = float(c["esa_t"][0]), float(c["esa_t"][3])
    assert port.run_block(c["esa"], c["esa_t"], c["hsg"], c["hsg_t"], (t0 - 2, t3 - 1, t0 - 1, t3), lookup_dir)["nplanes"] == 0


@pytest.mark.parametrize("name", sorted(BLOCKS))
def test_numpy_restatement_matches_golden_blocks(name, port, tables):
    c = BLOCKS[name]
    esa, gt, hsg, sgt = golden_io.window_inputs(port, c)
    assert np.array_equal(O.numpy_block(esa, gt, hsg, sgt, tables), c["planes"])


def test_window_arithmetic_matches_golden(port):
    for c in golden_io.window_cases():
        got = port.window(c["rw"], c["rh"], c["t"], c["bbox"])
        if c["expect"] is None:
            assert got is None, c
        else:
            e = c["expect"]
            assert got == (e["xoff"], e["yoff"], e["xsize"], e["ysize"], tuple(e["gt"])), c


def test_real_vrt_blocks_are_36001(port):
    """SURVEY 8: with the shipped VRT pixel size ceil() yields 36001-pixel windows."""
    t = (-180.0, PX_VRT, 0.0, 84.0, 0.0, -PX_VRT)
    w = port.window(4320000, 1728000, t, (-114.0, 39.0, -111.0, 42.0))
    assert (w[2], w[3]) == (36001, 36001)
    t = (-114.0, PX, 0.0, 42.0, 0.0, -PX)
    w = port.window(36000, 36000, t, (-114.0, 39.0, -111.0, 42.0))
    assert (w[2], w[3]) == (36000, 36000)


def test_default_lookup_tables_match_golden(port, lookup_dir):
    tabs = port.load_tables(lookup_dir)
    assert np.array_equal(golden_io.effective_lut(tabs), golden_io.luts()["default"])
    # known answers straight from the shipped CSVs (SURVEY 8c)
    g_ii = tabs[7]
    assert (g_ii[10, 1], g_ii[10, 4], g_ii[50, 2], g_ii[100, 4]) == (15, 59, 81, 62)
    assert list(g_ii[70, 1:5]) == [0, 0, 0, 0] and list(g_ii[80, 1:5]) == [100] * 4
    assert [int(tabs[t][10, 1]) for t in range(9)] == [45, 26, 65, 19, 36, 56, 30, 15, 50]
    assert (tabs[:, :, 0] == 255).all(), "column 0 is never written (cn.c:66)"


def test_hostile_lookup_tables_match_golden(port, tmp_path):
    from tests.golden.make_golden import write_hostile
    d = write_hostile(str(tmp_path / "hostile"))
    tabs = port.load_tables(d)
    assert np.array_equal(golden_io.effective_lut(tabs), golden_io.luts()["hostile"])
    assert tabs[0][20, 4] == 11 and tabs[0][7, 4] == 51 and tabs[0][0, 1] == 61 and tabs[0][200, 2] == 1


def test_lookup_errors(port, tmp_path):
    with pytest.raises(OSError):
        port.parse_lookup(str(tmp_path / "missing.csv"))
    (tmp_path / "empty.csv").write_bytes(b"")
    with pytest.raises(OSError):
        port.parse_lookup(str(tmp_path / "empty.csv"))
    (tmp_path / "header_only.csv").write_bytes(b"grid_code,cn\n")
    assert (port.parse_lookup(str(tmp_path / "header_only.csv")) == 255).all()


# ---- live runs of the reference object code ------------------------------------------------------


@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_restatement_matches_reference_live(name, kw, port, ref, tables, lookup_dir):
    b = make_block(**kw)
    h, w = b["esa"].shape
    gt = b["gt"]
    # a bbox exactly on the window edges can gain a pixel through ceil(); pull the far edges in
    # by 1/4 pixel so the reference reads exactly w x h
    bbox = (gt[0], gt[3] + (h - 0.25) * gt[5], gt[0] + (w - 0.25) * gt[1], gt[3])
    r = ref.run_block(b["esa"], gt, b["hsg"], b["soil_gt"], bbox, lookup_dir)
    if (r["w"], r["h"]) != (w, h):
        pytest.skip(f"reference window {r['w']}x{r['h']} differs from the synthetic {w}x{h}")
    assert r["nplanes"] == 18, r["log"]
    # the HSG window the reference cut from the same bbox
    hh, hw = b["hsg"].shape
    hxo, hyo, hxc, hyc, sgt = port.window(hw, hh, b["soil_gt"], bbox)
    got = port.block_rows(b["esa"], r["gt"], b["hsg"][hyo:hyo + hyc, hxo:hxo + hxc], sgt, tables)
    assert np.array_equal(got, r["planes"])


def test_random_geometries_against_reference_live(port, ref, tables, lookup_dir):
    rng = np.random.default_rng(1234)
    checked = 0
    for i in range(40):
        rw, rh = int(rng.integers(40, 400)), int(rng.integers(30, 300))
        px = float(rng.choice([PX, PX_VRT, 0.001, 1.0 / 3600]))
        ratio = float(rng.choice([25.0, 10.0, 3.0, 7.3, 1.0, 40.0]))
        lon0, lat0 = float(rng.integers(-180, 177)), float(rng.integers(-57, 84))
        esa_t = (lon0, px, 0.0, lat0, 0.0, -px)
        hpx = px * ratio
        hw, hh = int(rw / ratio) + 4, int(rh / ratio) + 4
        hsg_t = (lon0 - float(rng.uniform(0, 2)) * hpx, hpx, 0.0, lat0 + float(rng.uniform(0, 2)) * hpx, 0.0, -hpx)
        esa = synth.esa_tile(rw, rh, 100 + i, "random" if i % 3 == 0 else "worldcover", patch=16)
        hsg = synth.hsg_tile(hw, hh, 200 + i, "coastal" if i % 2 else "random", patch=2)
        x0, x1 = sorted(rng.uniform(-0.1 * rw, 1.1 * rw, 2))
        y0, y1 = sorted(rng.uniform(-0.1 * rh, 1.1 * rh, 2))
        bbox = (lon0 + x0 * px, lat0 - y1 * px, lon0 + x1 * px, lat0 - y0 * px)
        r = ref.run_block(esa, esa_t, hsg, hsg_t, bbox, lookup_dir)
        we = port.window(rw, rh, esa_t, bbox)
        wh = port.window(hw, hh, hsg_t, bbox)
        if r["nplanes"] == 0:
            assert we is None or wh is None, r["log"]
            continue
        assert r["nplanes"] == 18
        xo, yo, xc, yc, gt = we
        hxo, hyo, hxc, hyc, sgt = wh
        assert (xc, yc) == (r["w"], r["h"]) and gt == r["gt"]
        got = port.block_rows(esa[yo:yo + yc, xo:xo + xc], gt, hsg[hyo:hyo + hyc, hxo:hxo + hxc], sgt, tables)
        assert np.array_equal(got, r["planes"]), i
        checked += 1
    assert checked >= 20


def test_reference_save_order_and_options(ref, lookup_dir):
    b = make_block(w=64, h=48)
    gt = b["gt"]
    bbox = (gt[0], gt[3] + 47.75 * gt[5], gt[0] + 63.75 * gt[1], gt[3])
    r = ref.run_block(b["esa"], gt, b["hsg"], b["soil_gt"], bbox, lookup_dir, block_id=77)
    want = [f"cn_rasters_{c}/cn_{h}_{a}_77.tif" for c in O.CONDS for h in O.HCS for a in O.ARCS]
    assert r["paths"] == want                                   # cn.c:236,258-259,308
    assert r["options"] == ["COMPRESS=DEFLATE", "TILED=YES"]    # raster.c:206-207
    assert "completed condition for 77: drained/p/i" in r["log"]    # cn.c:366-369


def test_index_maps_tie_columns_differ_from_fma(port):
    """SURVEY appendix B: at lon -3 an FMA-contracted evaluation flips tie columns; the
    restatement must follow the unfused sequence."""
    w = 36000
    gt = (-3.0, PX, 0.0, 3.0, 0.0, -PX)
    sgt = (-3.0, HSG_PX, 0.0, 3.0, 0.0, -HSG_PX)
    ci = port.col_index(w, gt, sgt, 1440)
    ci_np, _ = O.numpy_index_maps(w, 1, gt, sgt, 1440, 1)
    assert np.array_equal(ci, ci_np)
    ties = np.arange(12, w, 25)
    up = int((ci[ties] == ties // 25 + 1).sum())
    assert up == 1132, up                                       # SURVEY appendix B, row "lon -3"
    assert ci[0] == 0 and ci[-1] == 1439
