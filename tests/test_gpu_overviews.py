"""GPU tests of option "overviews": the compressed-tile calls deliver nearest-neighbour overview levels of every
selected plane behind the block's full-resolution strips.  Every level tile is inflated with CPython's zlib and must
equal the rule of include/gcn10_cuda.h (tests/overview_rule.py) applied to the oracle's planes; the full-resolution
strips must be byte-identical to the same call without the option."""
import zlib

import numpy as np
import pytest

from gcn10_b200 import capi, hostlib, synth
from tests import fixtures, lookups
from tests import overview_rule as R
from tests.cases import SMALL_CASES, make_block

pytestmark = pytest.mark.gpu

T = 256
MASKS = [capi.MASK_ALL, capi.MASK_DRAINED, 1 << 13]
# (mask, fused, ordered, ship): all 24 combinations, dealt out over the cases x calls below
CONFIGS = [(m, f, o, s) for m in MASKS for f in (1, 0) for o in (0, 1) for s in (0, 1)]
CALLS = ["deflate", "rows", "tiles", "parts"]


@pytest.fixture(scope="module")
def ctx(tables):
    with capi.Context(0) as c:
        c.set_luts(tables)
        yield c


def _set(ctx, overviews=0, fused=1, ordered=0, ship=0, strip_rows=2048):
    for k, v in dict(overviews=overviews, fused=fused, ordered=ordered, ship=ship, strip_rows=strip_rows).items():
        ctx.set_option(k, v)


def _assemble(tiles, w, h):
    tx_n, ty_n = (w + T - 1) // T, (h + T - 1) // T
    assert sorted(tiles) == [(r, c) for r in range(ty_n) for c in range(tx_n)], "tile grid incomplete"
    full = np.zeros((ty_n * T, tx_n * T), dtype=np.uint8)
    for (r, c), z in tiles.items():
        raw = zlib.decompress(z)
        assert len(raw) == T * T
        full[r * T:(r + 1) * T, c * T:(c + 1) * T] = np.frombuffer(raw, dtype=np.uint8).reshape(T, T)
    return full[:h, :w]


def _parts(esa):
    h, w = esa.shape
    cut = max(1, w // 2)
    parts = [(capi.TileSource.from_raster(esa[:, :cut], 256, 256), 0, 0, cut, h)]
    if cut < w:
        parts.append((capi.TileSource.from_raster(esa[:, cut:], 256, 256), cut, 0, w - cut, h))
    return parts


def _run(ctx, call, b, mask, band=768):
    esa = b["esa"]
    h, w = esa.shape
    if call == "deflate":
        return ctx.block_deflate(esa, b["gt"], b["hsg"], b["soil_gt"], mask)
    if call == "rows":
        res = dict(tiles={}, overviews={}, bytes=0)
        for y0 in range(0, h, band):
            r = ctx.block_deflate_rows(esa[y0:y0 + band], h, y0, b["gt"], b["hsg"], b["soil_gt"], mask)
            for k, d in r["tiles"].items():
                res["tiles"].setdefault(k, {}).update(d)
            assert not r["overviews"] or y0 + band >= h, "levels before the band that ends the block"
            res["overviews"].update(r["overviews"])
        return res
    if call == "tiles":
        src = capi.TileSource.from_raster(esa, 256, 256)
        return ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"], mask)
    return ctx.block_parts_deflate(_parts(esa), 0, w, h, b["gt"], b["hsg"], b["soil_gt"], mask)


def _check_levels(res, want, mask, w, h):
    nlev = R.levels(w, h)
    assert sorted(res["overviews"]) == list(range(1, nlev + 1))
    for k in range(1, nlev + 1):
        lw, lh = R.dim(w, k), R.dim(h, k)
        planes = res["overviews"][k]
        assert sorted(planes) == [p for p in range(18) if mask >> p & 1]
        for p, tiles in planes.items():
            got = _assemble(tiles, lw, lh)
            assert np.array_equal(got, R.decimate(want[p], k)), f"level {k} plane {p}"


@pytest.mark.parametrize("call", CALLS)
@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_levels_equal_decimated_oracle(name, kw, call, ctx, port, tables):
    i = [c[0] for c in SMALL_CASES].index(name) * len(CALLS) + CALLS.index(call)
    mask, fused, ordered, ship = CONFIGS[i % len(CONFIGS)]
    b = make_block(**kw)
    h, w = b["esa"].shape
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    _set(ctx, 0, fused, ordered, ship)
    base = _run(ctx, call, b, mask)
    assert base["overviews"] == {}
    _set(ctx, 16, fused, ordered, ship)
    try:
        res = _run(ctx, call, b, mask)
    finally:
        _set(ctx)
    assert res["tiles"] == base["tiles"]            # level 0: byte-identical to the call without overviews
    _check_levels(res, want, mask, w, h)


def test_strip_fields_and_order(ctx, port, tables):
    b = make_block(w=3001, h=2600, seed=21)
    h, w = b["esa"].shape
    seen = []

    def on_strip(st):
        seen.append((st.level, st.tile_row0, st.n_tile_rows, st.tiles_x, st.level_w, st.level_h))

    _set(ctx, 16, strip_rows=512)
    try:
        ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], capi.MASK_DRAINED, on_strip=on_strip)
    finally:
        _set(ctx)
    nlev = R.levels(w, h)
    expect = []
    for k in range(nlev + 1):
        lw, lh = R.dim(w, k), R.dim(h, k)
        for y0 in range(0, lh, 512):
            rows = min(512, lh - y0)
            expect.append((k, y0 // T, (rows + T - 1) // T, (lw + T - 1) // T, lw, lh))
    assert seen == expect


def test_option_off_launches_nothing_new(ctx, tables):
    b = make_block(w=1300, h=1100, seed=22)
    counts = []
    with capi.Context(0) as fresh:
        fresh.set_luts(tables)
        n0 = fresh.launch_count()
        fresh.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        counts.append(fresh.launch_count() - n0)
    for ov in (3, 0):                                   # set, then back off: exactly the launches of a fresh context
        _set(ctx, ov)
        n0 = ctx.launch_count()
        levels = []
        ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=lambda st: levels.append(st.level))
        counts.append(ctx.launch_count() - n0)
        assert (max(levels) > 0) == (ov > 0)
    assert counts[2] == counts[0]
    assert counts[1] > counts[0]
    _set(ctx)


def test_bands_out_of_order_are_refused(ctx):
    b = make_block(w=700, h=1100, seed=23)
    esa, h = b["esa"], 1100
    _set(ctx, 16)
    try:
        with pytest.raises(capi.Gcn10Error) as e:       # no block open
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        assert e.value.code == -1
        ctx.block_deflate_rows(esa[:256], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        with pytest.raises(capi.Gcn10Error):            # a gap
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        r = ctx.block_deflate_rows(esa, h, 0, b["gt"], b["hsg"], b["soil_gt"])      # a new block starts at row 0
        assert sorted(r["overviews"]) == list(range(1, R.levels(700, h) + 1))
    finally:
        _set(ctx)
    # without the option the band calls are as free as before
    ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])


def test_prefetch_next_block_while_levels_run(ctx, port, tables):
    blocks = [make_block(w=2100, h=1900, seed=24 + i) for i in range(3)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    _set(ctx, 16)
    try:
        ctx.tiles_prefetch(srcs[0], 2100, 1900)
        results = []
        for i, b in enumerate(blocks):
            if i + 1 < len(blocks):
                ctx.tiles_prefetch(srcs[i + 1], 2100, 1900)
            results.append(ctx.block_tiles_deflate(srcs[i], 2100, 1900, b["gt"], b["hsg"], b["soil_gt"]))
    finally:
        _set(ctx)
    for b, res in zip(blocks, results):
        want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
        for p in (0, 17):
            assert np.array_equal(_assemble(res["tiles"][p], 2100, 1900), want[p])
        _check_levels(res, want, capi.MASK_ALL, 2100, 1900)


def test_sink_failure_in_a_level_aborts_and_damaged_tile_gives_no_strip(ctx, port, tables):
    b = make_block(w=1500, h=1300, seed=30)
    h, w = b["esa"].shape
    _set(ctx, 16)
    try:
        seen = []

        def fail_in_level_2(st):
            seen.append(st.level)
            return 7 if st.level == 2 else 0

        with pytest.raises(capi.Gcn10Error):
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=fail_in_level_2)
        assert seen[-1] == 2 and 3 not in seen
        src = capi.TileSource.from_raster(b["esa"], 256, 256)
        blob = src.blob.copy()
        o = int(src.offsets[5])
        blob[o + 2:o + 40] ^= 0x5A
        bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
        seen.clear()
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_tiles_deflate(bad, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=lambda st: seen.append(st.level))
        assert e.value.code == -6 and seen == []
        # the context is usable afterwards, levels included
        res = ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"])
    finally:
        _set(ctx)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    _check_levels(res, want, capi.MASK_ALL, w, h)


def _levels_of_decoded(res, planes, w, h):
    """Every level tile of the given planes equals the rule applied to the decoded level-0 tiles."""
    for p in planes:
        full = _assemble(res["tiles"][p], w, h)
        for k in range(1, R.levels(w, h) + 1):
            got = _assemble(res["overviews"][k][p], R.dim(w, k), R.dim(h, k))
            assert np.array_equal(got, R.decimate(full, k)), f"level {k} plane {p}"
        yield p, full


@pytest.mark.parametrize("shape", ["worldcover_36000", "vrt_36001_four_parts"])
def test_full_size_block_all_levels(shape, ctx, port, tables):
    if shape == "worldcover_36000":
        n, px, lon0, lat0 = 36000, 1.0 / 12000.0, -114.0, 42.0
    else:
        n, px, lon0, lat0 = 36001, 8.3333333333330430e-05, 33.0, -3.0
    gt, sgt, hsx, hsy = synth.block_geometry(lon0, lat0, n, n, px, 1.0 / 480.0, (0.0011, 0.0004), 2)
    esa = synth.esa_tile(n, n, 77, patch=64)
    hsg = synth.hsg_tile(hsx, hsy, 78, patch=3)
    if shape == "worldcover_36000":
        parts = [(capi.TileSource.from_raster(esa, 1024, 1024), 0, 0, n, n)]
    else:                                               # the real VRT's four files around a block corner
        c = 35000
        parts = [(capi.TileSource.from_raster(np.ascontiguousarray(esa[y:y + hh, x:x + ww]), 1024, 1024), x, y, ww, hh)
                 for (y, hh) in ((0, c), (c, n - c)) for (x, ww) in ((0, c), (c, n - c))]
    _set(ctx, 16)
    try:
        res = ctx.block_parts_deflate(parts, 0, n, n, gt, hsg, sgt)
    finally:
        _set(ctx)
    assert sorted(res["overviews"]) == list(range(1, 9))
    assert all(len(res["overviews"][k]) == 18 for k in res["overviews"])
    assert sum(len(res["overviews"][k][0]) for k in res["overviews"]) == 6781        # level tiles of one plane
    cols = R.src(np.arange(R.dim(n, 1)), 1, n)
    for p, _ in _levels_of_decoded(res, (0, 17), n, n):
        # level 1 against the oracle on the sampled pixels of every 997th level row
        lv1 = _assemble(res["overviews"][1][p], R.dim(n, 1), R.dim(n, 1))
        for r in range(0, R.dim(n, 1), 997):
            y = int(R.src(r, 1, n))
            want = port.block_rows(esa[y:y + 1], gt, hsg, sgt, tables, y0=y, y1=y + 1, h=n)[p][0]
            assert np.array_equal(lv1[r], want[cols]), f"plane {p} level 1 row {r}"


# ---- the program, file to file ---------------------------------------------------------------------------------

PX = 1.0 / 12000.0
HSG_PX = 1.0 / 480.0


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    root = tmp_path_factory.mktemp("gcn10_ov")
    W, H = 3000, 2200
    esa_t = (-114.0, PX, 0.0, 42.0, 0.0, -PX)
    esa = synth.esa_tile(W, H, 51, patch=96)
    hsg_t = (-114.0 - 1.3 * HSG_PX, HSG_PX, 0.0, 42.0 + 2.6 * HSG_PX, 0.0, -HSG_PX)
    hsg = synth.hsg_tile(130, 100, 52, "coastal", patch=3)
    hostlib.tiff_write(str(root / "esa.tif"), esa, esa_t)
    hostlib.tiff_write(str(root / "hsg.tif"), hsg, hsg_t)
    blocks = [(21, -114.0 + 100 * PX, 42.0 - 1500 * PX, -114.0 + 1400 * PX, 42.0 - 200 * PX),
              (22, -114.0 + 1700 * PX, 42.0 - 2500 * PX, -114.0 + 3300 * PX, 42.0 - 900 * PX)]
    fixtures.write_block_shapefile(str(root / "blocks.shp"), blocks)
    lookups.write_default_lookups(str(root / "lookups"))
    (root / "blocks.txt").write_text("21\n22\n")
    # the same land cover as a VRT mosaic of four GeoTIFFs
    from tests.fixtures import write_vrt
    srcs = []
    for (y, hh) in ((0, 1100), (1100, 1100)):
        for (x, ww) in ((0, 1600), (1600, 1400)):
            name = f"esa_{x}_{y}.tif"
            hostlib.tiff_write(str(root / name), np.ascontiguousarray(esa[y:y + hh, x:x + ww]),
                               (esa_t[0] + x * PX, PX, 0.0, esa_t[3] - y * PX, 0.0, -PX))
            srcs.append((name, 0, 0, x, y, ww, hh))
    write_vrt(str(root / "mosaic.vrt"), W, H, esa_t, srcs)
    for cfg, land in (("config.txt", "esa.tif"), ("config_vrt.txt", "mosaic.vrt")):
        fixtures.write_config(str(root / cfg), str(root / land), str(root / "hsg.tif"), str(root / "blocks.shp"),
                              str(root / "lookups"), str(root / "logs"))
    return dict(root=root, esa=esa, esa_t=esa_t, hsg=hsg, hsg_t=hsg_t, blocks=blocks)


def _frames(path):
    from PIL import Image
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append(np.array(im))
    return out


@pytest.mark.parametrize("config", ["config.txt", "config_vrt.txt"], ids=["geotiff", "vrt_mosaic"])
def test_program_overviews(world, reference, config, tmp_path):
    root = world["root"]
    modes = dict(gpu=False, host_inflate=True)
    for mode, hi in modes.items():
        r = fixtures.run_program(root, config, "-o", "--overviews", "--outdir", str(tmp_path / mode), host_inflate=hi)
        assert r.returncode == 0, r.stderr
    for bid, x0, y0, x1, y1 in world["blocks"]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                                   str(root / "lookups"), block_id=bid)
        for k, rel in enumerate(want["paths"]):
            frames = {m: _frames(str(tmp_path / m / rel)) for m in modes}
            f = frames["gpu"]
            assert len(f) == R.levels(want["w"], want["h"]) + 1, rel
            assert np.array_equal(f[0], want["planes"][k]), rel
            for lv in range(1, len(f)):
                assert np.array_equal(f[lv], R.decimate(f[0], lv)), (rel, lv)
            for m in modes:
                assert len(frames[m]) == len(f) and all(np.array_equal(a, c) for a, c in zip(frames[m], f)), (rel, m)
            t = hostlib.Tiff(str(tmp_path / "gpu" / rel))       # the project's reader: IFD0
            assert np.array_equal(t.read(), want["planes"][k])
            t.close()
