"""What the GPU tests of the block options (overviews, stats, aggregate, cog) share: a context of the test module's
own with an option setter that puts every option back, the (mask, fused, ordered, ship) configurations dealt out over
the small cases, the compressed-tile calls, the one decoder of a grid of 256 x 256 zlib tiles, a strip sink that checks
framing, and the program's input world.  Test modules import the fixtures ``ctx`` and ``world`` by name."""
import contextlib
import ctypes as C
import zlib

import numpy as np
import pytest

from gcn10_b200 import capi, hostlib, synth
from tests import fixtures, lookups
from tests.cases import HSG_PX, PX, PX_VRT, SMALL_CASES

T = 256
# every option the tests set, at the library's defaults
DEFAULTS = dict(overviews=0, stats=0, aggregate=0, cog=0, fused=1, ordered=0, ship=0, strip_rows=2048)
MASKS = [capi.MASK_ALL, capi.MASK_DRAINED, 1 << 13]
# (mask, fused, ordered, ship): all 24 combinations, dealt out over the cases x calls
CONFIGS = [(m, f, o, s) for m in MASKS for f in (1, 0) for o in (0, 1) for s in (0, 1)]
CALLS = ["deflate", "rows", "tiles", "parts"]


@pytest.fixture(scope="module")
def ctx(tables):
    """A context of the importing test module's own: options set there never reach the session's gpu_ctx."""
    with capi.Context(0) as c:
        c.set_luts(tables)
        yield c


@contextlib.contextmanager
def options(ctx, **kw):
    """Sets the given options; on exit puts every option of DEFAULTS back, whatever was set."""
    try:
        for k, v in kw.items():
            ctx.set_option(k, v)
        yield ctx
    finally:
        for k, v in DEFAULTS.items():
            ctx.set_option(k, v)


def config_for(case_name, call, configs=CONFIGS, calls=CALLS):
    """The entry of ``configs`` dealt to (case, call): round robin over the SMALL_CASES x calls grid in order."""
    i = [c[0] for c in SMALL_CASES].index(case_name) * len(calls) + calls.index(call)
    return configs[i % len(configs)]


def parts(esa):
    """The land cover as a mosaic of two tile sources, split at half its width."""
    h, w = esa.shape
    cut = max(1, w // 2)
    out = [(capi.TileSource.from_raster(esa[:, :cut], 256, 256), 0, 0, cut, h)]
    if cut < w:
        out.append((capi.TileSource.from_raster(esa[:, cut:], 256, 256), cut, 0, w - cut, h))
    return out


def run_call(ctx, call, b, mask, band=768, on_strip=None):
    """Block b through one of CALLS.  "rows" runs it in bands of ``band`` rows and merges their results: the overview
    levels, mean rasters and histograms must come with the band that ends the block, not before."""
    esa = b["esa"]
    h, w = esa.shape
    args = (b["gt"], b["hsg"], b["soil_gt"], mask)
    if call == "deflate":
        return ctx.block_deflate(esa, *args, on_strip=on_strip)
    if call == "tiles":
        return ctx.block_tiles_deflate(capi.TileSource.from_raster(esa, 256, 256), w, h, *args, on_strip=on_strip)
    if call == "parts":
        return ctx.block_parts_deflate(parts(esa), 0, w, h, *args, on_strip=on_strip)
    res = dict(tiles={}, overviews={}, aggregate={}, histograms=None)
    for y0 in range(0, h, band):
        r = ctx.block_deflate_rows(esa[y0:y0 + band], h, y0, *args, on_strip=on_strip)
        if y0 + band < h:
            assert not r["overviews"], "levels before the band that ends the block"
            assert not r["aggregate"], "mean rasters before the band that ends the block"
            assert r["histograms"] is None, "histograms before the band that ends the block"
        for k, d in r["tiles"].items():
            res["tiles"].setdefault(k, {}).update(d)
        res["overviews"].update(r["overviews"])
        res["aggregate"].update(r["aggregate"])
        res["histograms"] = r["histograms"]
    return res


def assemble(tiles, w, h, exact=None):
    """The w x h plane that tiles = {(tile_row, tile_x): zlib stream} decode to.  The grid must be complete, every tile
    256 x 256 bytes with zeros past the plane's right and bottom edges; with ``exact`` ({(tile_row, tile_x): bytes},
    the reference's) every stream must equal the reference's, byte for byte."""
    tx_n, ty_n = (w + T - 1) // T, (h + T - 1) // T
    assert sorted(tiles) == [(r, c) for r in range(ty_n) for c in range(tx_n)], "tile grid incomplete"
    full = np.zeros((ty_n * T, tx_n * T), dtype=np.uint8)
    for (r, c), z in tiles.items():
        if exact is not None:
            assert z == exact[(r, c)], f"tile {(r, c)}: {len(z)} bytes, reference {len(exact[(r, c)])}"
        raw = zlib.decompress(z)
        assert len(raw) == T * T
        full[r * T:(r + 1) * T, c * T:(c + 1) * T] = np.frombuffer(raw, dtype=np.uint8).reshape(T, T)
    assert not full[h:, :].any() and not full[:, w:].any(), "edge padding must be zero"
    return full[:h, :w]


def strip_collector(strips, tiles, fail_at=None):
    """A sink that records every strip as (aggregate, level, tile_row0, n_tile_rows, framed), checks the leader and
    trailer of every tile of a framed strip, and files the streams as tiles[kind][plane][(tile_row, tile_x)], kind =
    the level or "agg"; it fails the strips for which ``fail_at(strip)`` holds."""

    def on_strip(st):
        blob = C.string_at(st.blob, st.blob_bytes)
        strips.append((st.aggregate, st.level, st.tile_row0, st.n_tile_rows, st.framed))
        kind = "agg" if st.aggregate else st.level
        for k in range(st.n_planes):
            d = tiles.setdefault(kind, {}).setdefault(st.plane_ids[k], {})
            for tr in range(st.n_tile_rows):
                for tx in range(st.tiles_x):
                    i = (k * st.n_tile_rows + tr) * st.tiles_x + tx
                    o, n = st.offsets[i], st.sizes[i]
                    if st.framed:
                        assert blob[o - 4:o] == n.to_bytes(4, "little"), "leader"
                        assert blob[o + n:o + n + 4] == blob[o + n - 4:o + n], "trailer"
                    d[(st.tile_row0 + tr, tx)] = blob[o:o + n]
        return 7 if fail_at is not None and fail_at(st) else 0

    return on_strip


FULL_SIZE = ["worldcover_36000", "vrt_36001_four_parts"]


def full_size_block(shape):
    """(n, gt, soil_gt, esa, hsg) of an n x n block: 36000 at WorldCover's pixel size, or 36001 at the real VRT's."""
    if shape == "worldcover_36000":
        n, px, lon0, lat0 = 36000, PX, -114.0, 42.0
    else:
        n, px, lon0, lat0 = 36001, PX_VRT, 33.0, -3.0
    gt, sgt, hsx, hsy = synth.block_geometry(lon0, lat0, n, n, px, HSG_PX, (0.0011, 0.0004), 2)
    return n, gt, sgt, synth.esa_tile(n, n, 77, patch=64), synth.hsg_tile(hsx, hsy, 78, patch=3)


def full_size_parts(shape, esa):
    """The land cover of full_size_block in 1024 x 1024 tiles: one file, or the real VRT's four files around a block
    corner."""
    n = esa.shape[0]
    if shape == "worldcover_36000":
        return [(capi.TileSource.from_raster(esa, 1024, 1024), 0, 0, n, n)]
    c = 35000
    return [(capi.TileSource.from_raster(np.ascontiguousarray(esa[y:y + hh, x:x + ww]), 1024, 1024), x, y, ww, hh)
            for (y, hh) in ((0, c), (c, n - c)) for (x, ww) in ((0, c), (c, n - c))]


# ---- the program, file to file ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def world(tmp_path_factory):
    """The program's inputs: land cover as one GeoTIFF (config.txt) and as a VRT mosaic of four (config_vrt.txt), soil
    groups, two blocks and the default lookup tables."""
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
    srcs = []
    for (y, hh) in ((0, 1100), (1100, 1100)):
        for (x, ww) in ((0, 1600), (1600, 1400)):
            name = f"esa_{x}_{y}.tif"
            hostlib.tiff_write(str(root / name), np.ascontiguousarray(esa[y:y + hh, x:x + ww]),
                               (esa_t[0] + x * PX, PX, 0.0, esa_t[3] - y * PX, 0.0, -PX))
            srcs.append((name, 0, 0, x, y, ww, hh))
    fixtures.write_vrt(str(root / "mosaic.vrt"), W, H, esa_t, srcs)
    for cfg, land in (("config.txt", "esa.tif"), ("config_vrt.txt", "mosaic.vrt")):
        fixtures.write_config(str(root / cfg), str(root / land), str(root / "hsg.tif"), str(root / "blocks.shp"),
                              str(root / "lookups"), str(root / "logs"))
    return dict(root=root, esa=esa, esa_t=esa_t, hsg=hsg, hsg_t=hsg_t, blocks=blocks)


def frames(path):
    """Every image of a TIFF file (IFD0, then the overview levels), read with PIL."""
    from PIL import Image
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append(np.array(im))
    return out
