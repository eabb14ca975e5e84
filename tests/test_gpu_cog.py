"""GPU tests of option "cog": the whole-block compressed-tile calls deliver the overview levels first, smallest first,
then the full resolution, then the mean rasters, and with "ordered" every tile leaves the device framed for a Cloud
Optimized GeoTIFF.  The tile streams must be byte-identical to the same call without the option; the framing is
checked on every tile; the program's outputs must pass tests/cog_rule.py and equal the reference."""
import ctypes as C

import numpy as np
import pytest

from gcn10_b200 import capi, synth
from tests import cog_rule, fixtures
from tests import overview_rule as R
from tests.cases import SMALL_CASES, make_block
from tests.test_gpu_overviews import _assemble, _frames, _parts, world  # noqa: F401  (world: module fixture)

pytestmark = pytest.mark.gpu

T = 256
CALLS = ["deflate", "tiles", "parts"]
# (mask, fused, ordered, ship), dealt out over the cases x calls below: every (fused, ordered) pair several times
CONFIGS = [(m, f, o, s) for m in (capi.MASK_ALL, capi.MASK_DRAINED, 1 << 13) for o in (1, 0) for f in (1, 0)
           for s in (0, 1)]
AGG = 25


@pytest.fixture(scope="module")
def ctx(tables):
    with capi.Context(0) as c:
        c.set_luts(tables)
        yield c


def _set(ctx, cog=0, overviews=0, aggregate=0, fused=1, ordered=0, ship=0, strip_rows=2048):
    for k, v in dict(cog=cog, overviews=overviews, aggregate=aggregate, fused=fused, ordered=ordered, ship=ship,
                     strip_rows=strip_rows).items():
        ctx.set_option(k, v)


def _collector(strips, tiles, fail_at=None):
    """A sink that records every strip (aggregate, level, tile_row0, n_tile_rows, framed), checks the framing of framed
    strips tile by tile, and files the streams under (kind, plane, tile_row, tile_x), kind = level or "agg"."""

    def on_strip(st):
        blob = C.string_at(st.blob, st.blob_bytes)
        strips.append((st.aggregate, st.level, st.tile_row0, st.n_tile_rows, st.framed))
        kind = "agg" if st.aggregate else st.level
        for k in range(st.n_planes):
            for tr in range(st.n_tile_rows):
                for tx in range(st.tiles_x):
                    i = (k * st.n_tile_rows + tr) * st.tiles_x + tx
                    o, n = st.offsets[i], st.sizes[i]
                    if st.framed:
                        assert blob[o - 4:o] == n.to_bytes(4, "little"), "leader"
                        assert blob[o + n:o + n + 4] == blob[o + n - 4:o + n], "trailer"
                    tiles[(kind, st.plane_ids[k], st.tile_row0 + tr, tx)] = blob[o:o + n]
        return 7 if fail_at is not None and fail_at(st) else 0

    return on_strip


def _run(ctx, call, b, mask, on_strip):
    esa = b["esa"]
    h, w = esa.shape
    if call == "deflate":
        return ctx.block_deflate(esa, b["gt"], b["hsg"], b["soil_gt"], mask, on_strip=on_strip)
    if call == "tiles":
        src = capi.TileSource.from_raster(esa, 256, 256)
        return ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"], mask, on_strip=on_strip)
    return ctx.block_parts_deflate(_parts(esa), 0, w, h, b["gt"], b["hsg"], b["soil_gt"], mask, on_strip=on_strip)


def _check_order(strips, nlev, agg=True):
    """Levels nlev .. 1, then level 0, then the mean rasters; tile rows in order within each."""
    kinds = [("agg", 0) if a else ("lv", lv) for a, lv, *_ in strips]
    want_kinds = [("lv", k) for k in range(nlev, -1, -1)] + ([("agg", 0)] if agg else [])
    seen = [k for i, k in enumerate(kinds) if i == 0 or kinds[i - 1] != k]
    assert seen == want_kinds, seen
    for kind in want_kinds:
        rows = [(r0, n) for (a, lv, r0, n, _), k in zip(strips, kinds) if k == kind]
        at = 0
        for r0, n in rows:
            assert r0 == at, (kind, rows)
            at += n


@pytest.mark.parametrize("call", CALLS)
@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_cog_order_same_streams_framed(name, kw, call, ctx, port, tables):
    i = [c[0] for c in SMALL_CASES].index(name) * len(CALLS) + CALLS.index(call)
    mask, fused, ordered, ship = CONFIGS[i % len(CONFIGS)]
    b = make_block(**kw)
    h, w = b["esa"].shape
    nlev = R.levels(w, h)
    got = {}
    for cog in (0, 1):
        strips, tiles = [], {}
        _set(ctx, cog, 16, AGG, fused, ordered, ship)
        try:
            _run(ctx, call, b, mask, _collector(strips, tiles))
        finally:
            _set(ctx)
        got[cog] = (strips, tiles)
    strips, tiles = got[1]
    assert tiles == got[0][1]                       # every stream byte-identical to the call without the option
    _check_order(strips, nlev)
    assert all(f == (ordered == 1) for *_, f in strips)
    assert not any(f for *_, f in got[0][0])
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    for p in [p for p in range(18) if mask >> p & 1][:2]:
        full = _assemble({(r, c): z for (k, q, r, c), z in tiles.items() if k == 0 and q == p}, w, h)
        assert np.array_equal(full, want[p])
        for k in range(1, nlev + 1):
            lv = _assemble({(r, c): z for (kk, q, r, c), z in tiles.items() if kk == k and q == p}, R.dim(w, k), R.dim(h, k))
            assert np.array_equal(lv, R.decimate(want[p], k)), (p, k)


def test_rows_refuses_cog(ctx):
    b = make_block(w=700, h=600, seed=40)
    _set(ctx, cog=1, overviews=16)
    try:
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_deflate_rows(b["esa"], 600, 0, b["gt"], b["hsg"], b["soil_gt"])
        assert e.value.code == -1
    finally:
        _set(ctx)


def test_option_off_launches_nothing_new(ctx, tables):
    b = make_block(w=1300, h=1100, seed=41)
    counts = []
    with capi.Context(0) as fresh:
        fresh.set_luts(tables)
        fresh.set_option("overviews", 16)
        fresh.set_option("ordered", 1)
        n0 = fresh.launch_count()
        fresh.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        counts.append(fresh.launch_count() - n0)
    for cog in (1, 0):                                  # set, then back off: exactly the launches of a fresh context
        _set(ctx, cog, 16, ordered=1)
        n0 = ctx.launch_count()
        ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        counts.append(ctx.launch_count() - n0)
    _set(ctx)
    assert counts[2] == counts[0]
    # the levels in one decimation instead of one per full-resolution strip (a single strip here): same count
    assert counts[1] == counts[0]


def test_prefetch_next_block_and_host_raster_between(ctx, port, tables):
    """A prefetched block survives a host-raster call in between, whose whole upload takes the other slot."""
    blocks = [make_block(w=2100, h=1900, seed=42 + i) for i in range(3)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    other = make_block(w=1700, h=1500, seed=49)
    results, res_other = [], None
    _set(ctx, 1, 16, ordered=1)
    try:
        ctx.tiles_prefetch(srcs[0], 2100, 1900)
        for i, b in enumerate(blocks):
            if i + 1 < len(blocks):
                ctx.tiles_prefetch(srcs[i + 1], 2100, 1900)
            results.append(ctx.block_tiles_deflate(srcs[i], 2100, 1900, b["gt"], b["hsg"], b["soil_gt"]))
            if i == 0:
                res_other = ctx.block_deflate(other["esa"], other["gt"], other["hsg"], other["soil_gt"])
    finally:
        _set(ctx)
    for b, res, (w, h) in list(zip(blocks, results, [(2100, 1900)] * 3)) + [(other, res_other, (1700, 1500))]:
        want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
        for p in (0, 17):
            assert np.array_equal(_assemble(res["tiles"][p], w, h), want[p])
            for k in range(1, R.levels(w, h) + 1):
                assert np.array_equal(_assemble(res["overviews"][k][p], R.dim(w, k), R.dim(h, k)), R.decimate(want[p], k))


def test_sink_failure_in_a_level_and_damaged_tile(ctx, port, tables):
    b = make_block(w=1500, h=1300, seed=50)
    h, w = b["esa"].shape
    _set(ctx, 1, 16, AGG, ordered=1)
    try:
        strips = []
        with pytest.raises(capi.Gcn10Error):
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"],
                              on_strip=_collector(strips, {}, fail_at=lambda st: st.level == 1))
        assert [lv for _, lv, *_ in strips] == list(range(R.levels(w, h), 0, -1))     # stopped at level 1
        src = capi.TileSource.from_raster(b["esa"], 256, 256)
        blob = src.blob.copy()
        o = int(src.offsets[5])
        blob[o + 2:o + 40] ^= 0x5A
        bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
        strips.clear()
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_tiles_deflate(bad, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=_collector(strips, {}))
        assert e.value.code == -6 and strips == []
        strips, tiles = [], {}
        ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=_collector(strips, tiles))
    finally:
        _set(ctx)
    _check_order(strips, R.levels(w, h))
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    full = _assemble({(r, c): z for (k, q, r, c), z in tiles.items() if k == 0 and q == 3}, w, h)
    assert np.array_equal(full, want[3])


@pytest.mark.parametrize("shape", ["worldcover_36000", "vrt_36001_four_parts"])
def test_full_size_block(shape, ctx, port, tables):
    if shape == "worldcover_36000":
        n, px, lon0, lat0 = 36000, 1.0 / 12000.0, -114.0, 42.0
    else:
        n, px, lon0, lat0 = 36001, 8.3333333333330430e-05, 33.0, -3.0
    gt, sgt, hsx, hsy = synth.block_geometry(lon0, lat0, n, n, px, 1.0 / 480.0, (0.0011, 0.0004), 2)
    esa = synth.esa_tile(n, n, 77, patch=64)
    hsg = synth.hsg_tile(hsx, hsy, 78, patch=3)
    if shape == "worldcover_36000":
        parts = [(capi.TileSource.from_raster(esa, 1024, 1024), 0, 0, n, n)]
    else:
        c = 35000
        parts = [(capi.TileSource.from_raster(np.ascontiguousarray(esa[y:y + hh, x:x + ww]), 1024, 1024), x, y, ww, hh)
                 for (y, hh) in ((0, c), (c, n - c)) for (x, ww) in ((0, c), (c, n - c))]
    strips, tiles = [], {}
    _set(ctx, 1, 16, ordered=1)
    try:
        ctx.block_parts_deflate(parts, 0, n, n, gt, hsg, sgt, on_strip=_collector(strips, tiles))
    finally:
        _set(ctx)
    _check_order(strips, 8, agg=False)
    assert all(f for *_, f in strips)
    for p in (0, 17):
        full = _assemble({(r, cc): z for (k, q, r, cc), z in tiles.items() if k == 0 and q == p}, n, n)
        for k in range(1, 9):
            lv = _assemble({(r, cc): z for (kk, q, r, cc), z in tiles.items() if kk == k and q == p}, R.dim(n, k), R.dim(n, k))
            assert np.array_equal(lv, R.decimate(full, k)), (p, k)
        for y in list(range(0, n, 997)) + [n - 1]:
            want = port.block_rows(esa[y:y + 1], gt, hsg, sgt, tables, y0=y, y1=y + 1, h=n)[p][0]
            assert np.array_equal(full[y], want), f"plane {p} row {y}"


# ---- the program, file to file ---------------------------------------------------------------------------------

@pytest.mark.parametrize("config,host_inflate", [("config.txt", False), ("config_vrt.txt", False), ("config.txt", True)],
                         ids=["geotiff", "vrt_mosaic", "host_inflate"])
def test_program_cog(world, reference, config, host_inflate, tmp_path):  # noqa: F811
    root = world["root"]
    r = fixtures.run_program(root, config, "-o", "--outdir", str(tmp_path), "--cog", "--stats", "--aggregate", str(AGG),
                             host_inflate=host_inflate)
    assert r.returncode == 0, r.stderr
    for bid, x0, y0, x1, y1 in world["blocks"]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                                   str(root / "lookups"), block_id=bid)
        for k, rel in enumerate(want["paths"]):
            path = str(tmp_path / rel)
            ifds = cog_rule.check(path)
            f = _frames(path)
            assert len(f) == len(ifds) == R.levels(want["w"], want["h"]) + 1, rel
            assert np.array_equal(f[0], want["planes"][k]), rel
            for lv in range(1, len(f)):
                assert np.array_equal(f[lv], R.decimate(f[0], lv)), (rel, lv)
            cond, name = rel.split("/")[-2:]
            agg = str(tmp_path / f"{cond}_agg{AGG}" / name)
            assert len(cog_rule.check(agg)) == 1, agg               # the mean raster: a COG without levels
            assert len(_frames(agg)) == 1
