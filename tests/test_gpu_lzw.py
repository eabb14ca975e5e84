"""GPU decode of LZW land-cover tiles (TIFF Compression 5) against libtiff, and the chained calls against DEFLATE input.

GDAL reads an LZW GeoTIFF through libtiff, so libtiff is the judge: the tiles are made by libtiff's encoder
(gcn10_b200/tiff_lzw.py) from a known raster, the decoded window must equal that raster, and a damaged tile must get
an error exactly where libtiff gives one.  A block computed from LZW land cover must give the same output tile streams,
byte for byte, as the same block from DEFLATE land cover of the same pixels, which the other GPU tests pin to the
oracle."""
import numpy as np
import pytest

from gcn10_b200 import capi, synth, tiff_lzw
from tests.cases import make_block

pytestmark = pytest.mark.gpu


GEOMS = [
    # name, grid w, grid h, tile w, tile h, window (x_off, y_off, w, h) or None
    ("tiles256", 1300, 777, 256, 256, None),
    ("tiles512", 1500, 1100, 512, 512, None),
    ("tiles1024", 2500, 2100, 1024, 1024, None),
    ("tiles1000x700", 2100, 1500, 1000, 700, None),
    ("window_inside", 3000, 2200, 1024, 1024, (700, 300, 1500, 1300)),
    ("window_small_tiles", 1200, 900, 256, 256, (255, 257, 600, 500)),
    ("one_pixel_window", 600, 600, 256, 256, (300, 299, 1, 1)),
]


@pytest.mark.parametrize("name,gw,gh,tw,th,win", GEOMS, ids=[g[0] for g in GEOMS])
@pytest.mark.parametrize("profile", ["worldcover", "random"])
def test_decode_equals_libtiff_source(name, gw, gh, tw, th, win, profile, gpu_ctx):
    grid = synth.esa_tile(gw, gh, seed=len(name) * 7 + gw, profile=profile, patch=48)
    x_off, y_off, w, h = win if win else (0, 0, gw, gh)
    src = capi.TileSource.from_raster(grid, tw, th, x_off=x_off, y_off=y_off, gap=3, codec="lzw")
    assert src.compression == 5
    out = np.full((h + 2, w + 37), 0xEE, dtype=np.uint8)
    view = out[1:h + 1, :w]
    rc, _, status = gpu_ctx.inflate_tiles(src, w, h, out=view, want_status=True)
    assert rc == 0, gpu_ctx.lib.gcn10_cuda_last_error().decode()
    assert not status.any()
    assert np.array_equal(view, grid[y_off:y_off + h, x_off:x_off + w])
    assert (out[0] == 0xEE).all() and (out[-1] == 0xEE).all() and (out[:, w:] == 0xEE).all()
    assert gpu_ctx.last_inflate_ms() > 0


def test_flat_noise_and_sparse_tiles(gpu_ctx):
    """Long strings (flat tiles), table refills (noise), and sparse tiles read as zeros."""
    rng = np.random.default_rng(4)
    grid = np.full((1024, 2048), 70, dtype=np.uint8)
    grid[:, 1024:] = rng.integers(0, 256, (1024, 1024), dtype=np.uint8)
    grid[:300, :300] = 10
    src = capi.TileSource.from_raster(grid, 512, 512, codec="lzw", sparse={(1, 3)})
    want = grid.copy()
    want[512:, 1536:] = 0
    assert np.array_equal(gpu_ctx.inflate_tiles(src, 2048, 1024), want)


def _damage(src, k, fn):
    blob = src.blob.copy()
    o, n = int(src.offsets[k]), int(src.sizes[k])
    stream = fn(blob[o:o + n].tobytes())
    blob[o:o + len(stream)] = np.frombuffer(stream, dtype=np.uint8)
    sizes = src.sizes.copy()
    sizes[k] = len(stream)
    return capi.TileSource(src.tile_w, src.tile_h, src.tiles_x, src.tiles_y, src.x_off, src.y_off, blob, src.offsets,
                           sizes, 5)


def test_damaged_tiles_get_libtiff_verdicts(gpu_ctx):
    b = make_block(w=768, h=512, seed=3)
    src = capi.TileSource.from_raster(b["esa"], 256, 256, codec="lzw")
    cases = [
        (lambda s: s[:len(s) // 2], 8),                       # input ends before the tile is full
        (lambda s: bytes([0x00, 0x01]) + s[2:], 11),          # old-style (LSB-first) signature
        (lambda s: bytes([0xFF, 0xFF]) + s[2:], 12),          # no Clear first: code 511 before any table
    ]
    for k, (fn, want) in enumerate(cases):
        bad = _damage(src, k, fn)
        o = int(bad.offsets[k])
        if want != 11:                                        # (libtiff would try its old-style decoder)
            assert tiff_lzw.decode(bad.blob[o:o + int(bad.sizes[k])].tobytes(), 256, 256) is None
        rc, _, status = gpu_ctx.inflate_tiles(bad, 768, 512, want_status=True)
        assert rc == -6
        assert status[k] == want and not np.delete(status, k).any(), status
    calls = []
    with pytest.raises(capi.Gcn10Error) as ei:
        gpu_ctx.block_tiles_deflate(_damage(src, 4, cases[0][0]), 768, 512, b["gt"], b["hsg"], b["soil_gt"],
                                    on_strip=lambda s: calls.append(1))
    assert ei.value.code == -6 and not calls


def test_unknown_compression_is_refused(gpu_ctx):
    b = make_block(w=300, h=200, seed=2)
    src = capi.TileSource.from_raster(b["esa"], 256, 256)
    for c in (1, 7, 34887):
        src.compression = c
        rc, _, _ = gpu_ctx.inflate_tiles(src, 300, 200, want_status=True)
        assert rc == -1
    for c in (0, 8, 32946):
        src.compression = c
        assert np.array_equal(gpu_ctx.inflate_tiles(src, 300, 200), b["esa"])


@pytest.mark.parametrize("options", [{}, {"overviews": 3}, {"stats": 1}, {"aggregate": 25},
                                     {"cog": 1, "ordered": 1, "overviews": 3}],
                         ids=["plain", "overviews", "stats", "aggregate", "cog_ordered"])
def test_block_streams_equal_deflate_input(options, tables):
    b = make_block(w=1500, h=1100, seed=12)
    with capi.Context(0) as ctx:
        ctx.set_luts(tables)
        for k, v in options.items():
            ctx.set_option(k, v)
        results = []
        for codec in ("deflate", "lzw"):
            src = capi.TileSource.from_raster(b["esa"], 512, 512, codec=codec)
            before = ctx.launch_count()
            results.append(ctx.block_tiles_deflate(src, 1500, 1100, b["gt"], b["hsg"], b["soil_gt"]))
            results[-1]["launches"] = ctx.launch_count() - before
    d, z = results
    assert d["tiles"] == z["tiles"] and d["overviews"] == z["overviews"] and d["aggregate"] == z["aggregate"]
    assert d["launches"] == z["launches"]
    if options.get("stats"):
        assert np.array_equal(d["histograms"], z["histograms"])


def test_mosaic_mixes_codecs(gpu_ctx):
    """Nine parts, DEFLATE and LZW alternating, with tile grids that do not line up: one call, both kernels."""
    w, h = 1900, 1500
    b = make_block(w=w, h=h, seed=31)
    esa = b["esa"]
    xs, ys = [0, 700, 1300, w], [0, 500, 1100, h]
    parts = []
    for j in range(3):
        for i in range(3):
            x, y, pw, ph = xs[i], ys[j], xs[i + 1] - xs[i], ys[j + 1] - ys[j]
            ox, oy = 11 * i, 7 * j
            grid = synth.esa_tile(ox + pw + 5, oy + ph + 9, seed=200 + 3 * j + i, patch=40)
            grid[oy:oy + ph, ox:ox + pw] = esa[y:y + ph, x:x + pw]
            src = capi.TileSource.from_raster(grid, (256, 240, 512)[i], (256, 112, 512)[j], x_off=ox, y_off=oy,
                                              codec=("deflate", "lzw")[(3 * j + i) % 2])
            parts.append((src, x, y, pw, ph))
    assert np.array_equal(gpu_ctx.inflate_parts(parts, 0, w, h), esa)
    plain = [(capi.TileSource.from_raster(esa, 512, 512), 0, 0, w, h)]
    got = gpu_ctx.block_parts_deflate(parts, 0, w, h, b["gt"], b["hsg"], b["soil_gt"])
    want = gpu_ctx.block_parts_deflate(plain, 0, w, h, b["gt"], b["hsg"], b["soil_gt"])
    assert got["tiles"] == want["tiles"]


def test_prefetch_with_alternating_codecs(gpu_ctx):
    blocks = [make_block(w=900, h=700, seed=80 + i, esa_patch=30) for i in range(4)]
    codecs = ["lzw", "deflate", "lzw", "lzw"]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256, codec=c) for b, c in zip(blocks, codecs)]
    refs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    wants = [gpu_ctx.block_tiles_deflate(r, 900, 700, b["gt"], b["hsg"], b["soil_gt"])["tiles"]
             for r, b in zip(refs, blocks)]
    gpu_ctx.tiles_prefetch(srcs[0], 900, 700)
    for i in range(4):
        if i + 1 < 4:
            gpu_ctx.tiles_prefetch(srcs[i + 1], 900, 700)
        b = blocks[i]
        assert gpu_ctx.block_tiles_deflate(srcs[i], 900, 700, b["gt"], b["hsg"], b["soil_gt"])["tiles"] == wants[i]


@pytest.mark.parametrize("shape", ["worldcover_36000", "vrt_36001_four_parts"])
def test_full_size_block_equals_deflate_input(shape, gpu_ctx):
    """Full-size blocks in 1024 x 1024 tiles: a 36000 x 36000 WorldCover-like block in LZW tiles, and the four-part
    36001 x 36001 window of the shipped VRT's geometry (parts 35000 and 1001 pixels wide, so every part has clipped edge
    tiles that decode through scratch copies) with three LZW parts and one zlib part.  The 18 rasters' tile streams equal
    those of the same call on zlib tiles of the same pixels."""
    if shape == "worldcover_36000":
        n, px, lon0, lat0 = 36000, 1.0 / 12000.0, -114.0, 42.0
        rects = [(0, 0, n, n)]
        codecs = ["lzw"]
    else:
        n, px, lon0, lat0 = 36001, 8.3333333333330430e-05, 33.0, -3.0
        c = 35000
        rects = [(x, y, ww, hh) for (y, hh) in ((0, c), (c, n - c)) for (x, ww) in ((0, c), (c, n - c))]
        codecs = ["lzw", "lzw", "deflate", "lzw"]
    gt, sgt, hsx, hsy = synth.block_geometry(lon0, lat0, n, n, px, 1.0 / 480.0, (0.0011, 0.0004), 2)
    esa = synth.esa_tile(n, n, 77, patch=64)
    hsg = synth.hsg_tile(hsx, hsy, 78, patch=3)

    def parts(codec_of):
        return [(capi.TileSource.from_raster(np.ascontiguousarray(esa[y:y + hh, x:x + ww]), 1024, 1024,
                                             codec=codec_of(k)), x, y, ww, hh)
                for k, (x, y, ww, hh) in enumerate(rects)]
    want = gpu_ctx.block_parts_deflate(parts(lambda k: "deflate"), 0, n, n, gt, hsg, sgt)["tiles"]
    got = gpu_ctx.block_parts_deflate(parts(lambda k: codecs[k]), 0, n, n, gt, hsg, sgt)["tiles"]
    assert sorted(got) == list(range(18))
    assert got == want


@pytest.mark.parametrize("mosaic", [False, True], ids=["geotiff", "vrt_mosaic"])
def test_program_on_lzw_land_cover(mosaic, reference, tmp_path):
    """gcn10 on an LZW GeoTIFF, and on a VRT whose sources are LZW and DEFLATE files: the land cover is decoded on the
    GPU, the 18 rasters equal the reference's process_block() and the GCN10_HOST_INFLATE=1 run."""
    import os
    import subprocess
    from gcn10_b200 import hostlib
    from tests import fixtures, lookups
    from tests.lzw_files import recode_to_lzw
    px, hpx = 1.0 / 12000.0, 1.0 / 480.0
    W, H = 2000, 1500
    esa_t = (-114.0, px, 0.0, 42.0, 0.0, -px)
    esa = synth.esa_tile(W, H, 43, patch=96)
    hsg_t = (-114.0 - 1.3 * hpx, hpx, 0.0, 42.0 + 2.6 * hpx, 0.0, -hpx)
    hsg = synth.hsg_tile(90, 70, 44, "coastal", patch=3)
    hostlib.tiff_write(str(tmp_path / "hsg.tif"), hsg, hsg_t)
    if mosaic:
        half = W // 2
        hostlib.tiff_write(str(tmp_path / "a_deflate.tif"), esa[:, :half], esa_t)
        hostlib.tiff_write(str(tmp_path / "b.tif"), esa[:, half:], (esa_t[0] + half * px,) + esa_t[1:])
        recode_to_lzw(str(tmp_path / "b.tif"), str(tmp_path / "b_lzw.tif"))
        land = fixtures.write_vrt(str(tmp_path / "esa.vrt"), W, H, esa_t,
                                  [("a_deflate.tif", 0, 0, 0, 0, half, H), ("b_lzw.tif", 0, 0, half, 0, W - half, H)])
        tag = "mosaic parts (LZW) decoded on the gpu"
    else:
        hostlib.tiff_write(str(tmp_path / "esa_deflate.tif"), esa, esa_t)
        recode_to_lzw(str(tmp_path / "esa_deflate.tif"), str(tmp_path / "esa.tif"))
        land = str(tmp_path / "esa.tif")
        tag = "LZW tiles decoded on the gpu"
    blocks = [(21, -114.0 + 100 * px, 42.0 - 1300 * px, -114.0 + 1400 * px, 42.0 - 100 * px)]
    fixtures.write_block_shapefile(str(tmp_path / "blocks.shp"), blocks)
    lookups.write_default_lookups(str(tmp_path / "lookups"))
    planes = {}
    for host_inflate in (False, True):
        run = tmp_path / ("host" if host_inflate else "gpu")
        run.mkdir()
        fixtures.write_config(str(run / "config.txt"), land, str(tmp_path / "hsg.tif"), str(tmp_path / "blocks.shp"),
                              str(tmp_path / "lookups"), str(run / "logs"))
        (run / "blocks.txt").write_text("21\n")
        env = dict(os.environ, GCN10_HOST_INFLATE="1" if host_inflate else "0", GCN10_HOST_DEFLATE="0")
        r = subprocess.run([hostlib.EXE_PATH, "-c", str(run / "config.txt"), "-l", str(run / "blocks.txt"), "--gpus",
                            "1", "-o"], cwd=str(run), capture_output=True, text=True, timeout=300, env=env)
        assert r.returncode == 0, r.stderr
        log = (run / "logs" / "rank_0.log").read_text()
        assert (tag in log) == (not host_inflate), log[-2000:]
        assert "inflated on the gpu" not in log
        want = reference.run_block(esa, esa_t, hsg, hsg_t, blocks[0][1:], str(tmp_path / "lookups"), block_id=21)
        got = []
        for k, rel in enumerate(want["paths"]):
            t = hostlib.Tiff(str(run / rel))
            got.append(t.read())
            t.close()
            assert np.array_equal(got[-1], want["planes"][k]), rel
        planes[host_inflate] = got
    assert all(np.array_equal(a, b) for a, b in zip(planes[False], planes[True]))
