"""CPU tests of the C host program's CUDA-free parts (gcn10_b200/host/libgcn10host.so): the lookup CSV
reader, window arithmetic, config file, block list, shapefile extents, GeoTIFF writer/reader and log
format.  Expected values come from the golden fixtures (reference object code) and the oracle."""
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from gcn10_b200 import hostlib
from tests import lookups
from tests import fixtures, golden_io

PX = 1.0 / 12000.0


def test_lookup_reader_matches_oracle_and_golden(port, lookup_dir, tmp_path):
    from tests.golden.make_golden import write_hostile
    g = golden_io.luts()
    for label, d in (("default", lookup_dir), ("hostile", write_hostile(str(tmp_path / "hostile")))):
        t = hostlib.load_lookup_tables(d)
        assert np.array_equal(t, port.load_tables(d)), label
        assert np.array_equal(golden_io.effective_lut(t), g[label]), label


def test_lookup_reader_errors(tmp_path):
    with pytest.raises(hostlib.HostError) as e:
        hostlib.load_lookup_tables(str(tmp_path))
    assert e.value.code == -2 and "cannot open lookup table" in e.value.msg       # cn.c:30
    lookups.write_default_lookups(str(tmp_path))
    open(tmp_path / "default_lookup_f_ii.csv", "wb").close()
    with pytest.raises(hostlib.HostError) as e:
        hostlib.load_lookup_tables(str(tmp_path))
    assert e.value.code == -3 and "empty lookup table" in e.value.msg             # cn.c:44


def test_window_arithmetic_matches_golden():
    for c in golden_io.window_cases():
        got = hostlib.raster_window(c["rw"], c["rh"], c["t"], c["bbox"])
        if c["expect"] is None:
            assert got is None, c
        else:
            e = c["expect"]
            assert got == (e["xoff"], e["yoff"], e["xsize"], e["ysize"], tuple(e["gt"])), c


def test_window_matches_reference_live(reference):
    rng = np.random.default_rng(7)
    for _ in range(300):
        rw, rh = int(rng.integers(1, 5000)), int(rng.integers(1, 5000))
        px = float(rng.choice([PX, 8.3333333333330430e-05, 0.01, 1 / 480]))
        t = (float(rng.uniform(-180, 180)), px, 0.0, float(rng.uniform(-60, 84)), 0.0, -px)
        x0, x1 = sorted(rng.uniform(-0.2 * rw, 1.2 * rw, 2))
        y0, y1 = sorted(rng.uniform(-0.2 * rh, 1.2 * rh, 2))
        bbox = (t[0] + x0 * px, t[3] - y1 * px, t[0] + x1 * px, t[3] - y0 * px)
        assert hostlib.raster_window(rw, rh, t, bbox) == reference.window(rw, rh, t, bbox)


def test_config_parser(tmp_path):
    p = fixtures.write_config(str(tmp_path / "config.txt"), "/data/esa.tif", "/data/hsg.tif", "/data/b.shp",
                              "/data/lookups", "logs/")
    cfg = hostlib.parse_config(p)
    assert cfg == {"hysogs_data_path": "/data/hsg.tif", "esa_data_path": "/data/esa.tif",
                   "blocks_shp_path": "/data/b.shp", "lookup_table_path": "/data/lookups", "log_dir": "logs/"}
    (tmp_path / "bad.txt").write_text("esa_data_path=x\nnot a pair\n#log_dir=zzz\n")
    with pytest.raises(hostlib.HostError) as e:
        hostlib.parse_config(str(tmp_path / "bad.txt"))
    assert e.value.code == -2 and e.value.msg.startswith("missing one of: hysogs_data_path")   # config.c:108
    with pytest.raises(hostlib.HostError) as e:
        hostlib.parse_config(str(tmp_path / "absent.txt"))
    assert e.value.code == -1 and "cannot open config" in e.value.msg                           # config.c:52


def test_block_list(tmp_path):
    (tmp_path / "blocks.txt").write_text("2234\n2261 2256\n\n 7\nx 9\n")
    assert hostlib.read_block_list(str(tmp_path / "blocks.txt")) == [2234, 2261, 2256, 7]     # fscanf stops at 'x'
    with pytest.raises(hostlib.HostError):
        hostlib.read_block_list(str(tmp_path / "none.txt"))


def test_shapefile_reader(tmp_path):
    blocks = [(3, 168.0, -54.0, 171.0, -51.0), (2234, -114.0, 39.0, -111.0, 42.0), (77, -3.0, 0.0, 0.0, 3.0)]
    shp = fixtures.write_block_shapefile(str(tmp_path / "blocks.shp"), blocks)
    b = hostlib.Blocks(shp)
    assert len(b) == 3 and b.ids() == [3, 2234, 77]
    assert b.bbox(2234) == (-114.0, 39.0, -111.0, 42.0)                     # minx, miny, maxx, maxy (cn.c:179-182)
    assert b.bbox(5) is None
    b.close()
    with pytest.raises(hostlib.HostError) as e:
        hostlib.Blocks(str(tmp_path / "missing.shp"))
    assert "ogr open failed" in e.value.msg                                  # cn.c:157


def test_reference_shapefile_if_present():
    shp = "/root/reference/blocks/esa_extent_blocks.shp"
    if not os.path.exists(shp):
        pytest.skip("reference tree not present")
    b = hostlib.Blocks(shp)
    ids = b.ids()
    assert len(ids) == 2651 and min(ids) == 3 and max(ids) == 2653
    for bid in (2234, 2261, 2256):                                          # src/test/blocks.txt
        x0, y0, x1, y1 = b.bbox(bid)
        assert (x1 - x0, y1 - y0) == (3.0, 3.0) and x0 == int(x0) and y0 == int(y0)
    assert b.bbox(2234) == (-114.0, 39.0, -111.0, 42.0)
    b.close()


@pytest.mark.parametrize("w,h", [(1, 1), (255, 257), (256, 256), (700, 1000), (4097, 300)])
def test_geotiff_roundtrip_and_libtiff_decode(w, h, tmp_path):
    from PIL import Image
    rng = np.random.default_rng(w * 31 + h)
    a = (rng.integers(0, 4, (h, w)) * 25 + (np.arange(w)[None, :] // 37) % 3).astype(np.uint8)
    gt = (-114.0, PX, 0.0, 42.0, 0.0, -PX)
    p = str(tmp_path / "out.tif")
    hostlib.tiff_write(p, a, gt, threads=3)
    t = hostlib.Tiff(p)
    assert (t.width, t.height) == (w, h) and t.georeferenced and t.gt == gt
    assert np.array_equal(t.read(), a)
    if w > 10 and h > 10:
        assert np.array_equal(t.read(3, 5, w - 7, h - 9, threads=1), a[5:h - 4, 3:w - 4])
    t.close()
    im = Image.open(p)                                      # independent decoder (libtiff)
    assert im.size == (w, h) and im.info.get("compression") == "tiff_adobe_deflate"      # raster.c:206
    assert im.tag_v2[322] == 256 and im.tag_v2[323] == 256                                 # raster.c:207, GDAL default tile
    assert np.array_equal(np.array(im), a)
    assert 42113 not in im.tag_v2, "the reference sets no NoData tag"


@pytest.mark.parametrize("compression", ["raw", "tiff_lzw", "tiff_adobe_deflate"])
def test_geotiff_reader_on_libtiff_files(compression, tmp_path):
    from PIL import Image
    rng = np.random.default_rng(5)
    a = (rng.integers(0, 6, (333, 517)) * 20).astype(np.uint8)
    a[100:200, 50:400] = 80
    p = str(tmp_path / f"{compression}.tif")
    Image.fromarray(a).save(p, compression=compression)
    t = hostlib.Tiff(p)
    assert (t.width, t.height) == (517, 333) and not t.georeferenced
    assert np.array_equal(t.read(threads=2), a)
    assert np.array_equal(t.read(17, 99, 200, 101), a[99:200, 17:217])
    t.close()


def test_geotiff_reader_rejects_garbage(tmp_path):
    (tmp_path / "x.tif").write_bytes(b"not a tiff at all")
    with pytest.raises(hostlib.HostError) as e:
        hostlib.Tiff(str(tmp_path / "x.tif"))
    assert "gdal open failed" in e.value.msg                 # raster.c:121


def test_log_format(tmp_path):
    L = hostlib.load()
    lg = L.gh_log_open(os.fsencode(str(tmp_path / "logs")), 3)
    L.gh_log_message(lg, b"INFO", b"completed condition for 2234: drained/p/i", 0)
    L.gh_log_message(lg, b"ERROR", b"block 9 not found", 0)
    L.gh_log_close(lg)
    lines = (tmp_path / "logs" / "rank_3.log").read_text().splitlines()                  # log.c:76
    ts = r"\[\d{4}-\d\d-\d\dT\d\d:\d\d:\d\d\]"
    assert re.fullmatch(ts + r" \[rank 3\] logging started", lines[0])                   # log.c:112
    assert re.fullmatch(ts + r" \[INFO\] \[rank 3\] completed condition for 2234: drained/p/i", lines[1])   # log.c:158
    assert re.fullmatch(ts + r" \[ERROR\] \[rank 3\] block 9 not found", lines[2])
    assert re.fullmatch(ts + r" \[rank 3\] logging finished", lines[3])                  # log.c:263


def test_cli_meta_flags_and_errors(tmp_path):
    exe = hostlib.EXE_PATH
    if not os.path.exists(exe):
        pytest.skip("gcn10 executable not built")
    r = subprocess.run([exe, "--version"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == "gcn10 0.1.0\n"                             # main.c:51
    r = subprocess.run([exe, "-h"], capture_output=True, text=True)
    assert r.returncode == 0 and "--config, -c <file>" in r.stdout and "--overwrite, -o" in r.stdout
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 1 and "missing -c/--config <file>" in r.stderr               # main.c:103-108
    r = subprocess.run([exe, "-c", str(tmp_path / "nope.txt")], capture_output=True, text=True)
    assert r.returncode == 1 and "cannot open config" in r.stderr                        # config.c:52


def test_geotiff_writer_accepts_precompressed_tile_rows(tmp_path):
    """The path the GPU encoder feeds: complete zlib streams per 256 x 256 tile, appended tile row by tile row
    (here produced with CPython's zlib at two different levels, to show any valid stream is accepted)."""
    import zlib
    from PIL import Image
    rng = np.random.default_rng(11)
    w, h = 700, 600
    a = (rng.integers(0, 5, (h, w)) * 20).astype(np.uint8)
    a[:, 300:] = 77
    p = str(tmp_path / "tiles.tif")
    gt = (10.0, PX, 0.0, 5.0, 0.0, -PX)
    tw = hostlib.TiffWriter(p, w, h, gt)
    pad = np.zeros((768, 768), dtype=np.uint8)
    pad[:h, :w] = a
    for tr in range(3):
        streams = [zlib.compress(pad[tr * 256:(tr + 1) * 256, tx * 256:(tx + 1) * 256].tobytes(), 1 + 4 * (tx % 2))
                   for tx in range(3)]
        assert tw.put_tile_row(tr, streams) == 0
    assert tw.close() == 0
    t = hostlib.Tiff(p)
    assert (t.width, t.height) == (w, h) and t.gt == gt
    assert np.array_equal(t.read(), a)
    t.close()
    assert np.array_equal(np.array(Image.open(p)), a)


def test_geotiff_writer_rejects_out_of_order_and_incomplete(tmp_path):
    import zlib
    z = zlib.compress(bytes(65536))
    tw = hostlib.TiffWriter(str(tmp_path / "a.tif"), 256, 512, (0, 1, 0, 0, 0, -1))
    assert tw.put_tile_row(1, [z]) != 0                         # must start at tile row 0
    assert tw.close() != 0                                      # nothing valid was written
    tw = hostlib.TiffWriter(str(tmp_path / "b.tif"), 256, 512, (0, 1, 0, 0, 0, -1))
    assert tw.put_tile_row(0, [z]) == 0
    assert tw.close() != 0                                      # second tile row missing


def test_window_tiles_are_the_files_zlib_streams(tmp_path):
    """gh_tiff_window_tiles_plan / _read (the GPU-inflate input path): the tiles of a window come back as the
    zlib streams the file holds, in window order, with the window's position inside the tile grid; inflating
    them with zlib reproduces the raster.  Datasets that are not tiled DEFLATE without predictor are refused."""
    import zlib
    from gcn10_b200 import synth
    w, h = 1100, 700
    esa = synth.esa_tile(w, h, 5, patch=40)
    path = str(tmp_path / "lc.tif")
    hostlib.tiff_write(path, esa, (-114.0, 1 / 12000, 0, 42.0, 0, -1 / 12000))
    t = hostlib.Tiff(path)
    for (xo, yo, xc, yc) in [(0, 0, w, h), (300, 257, 500, 300), (1099, 699, 1, 1), (255, 0, 2, 700)]:
        tl = t.window_tiles(xo, yo, xc, yc, threads=3)
        assert tl is not None and (tl["tile_w"], tl["tile_h"]) == (256, 256)
        assert tl["x_in"] == xo % 256 and tl["y_in"] == yo % 256
        grid = np.zeros((tl["tiles_y"] * 256, tl["tiles_x"] * 256), dtype=np.uint8)
        for i in range(tl["tiles_y"] * tl["tiles_x"]):
            o, n = int(tl["offsets"][i]), int(tl["sizes"][i])
            raw = zlib.decompress(tl["blob"][o:o + n].tobytes())
            r, c = divmod(i, tl["tiles_x"])
            grid[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256] = np.frombuffer(raw, dtype=np.uint8).reshape(256, 256)
        got = grid[tl["y_in"]:tl["y_in"] + yc, tl["x_in"]:tl["x_in"] + xc]
        assert np.array_equal(got, esa[yo:yo + yc, xo:xo + xc])
    assert t.window_tiles(0, 0, w + 1, h) is None              # outside the raster
    t.close()
    # a stripped, uncompressed TIFF (Pillow's default) cannot be handed over compressed
    from PIL import Image
    p2 = str(tmp_path / "plain.tif")
    Image.fromarray(esa[:64, :64]).save(p2)
    t2 = hostlib.Tiff(p2)
    assert t2.window_tiles() is None
    assert np.array_equal(t2.read(), esa[:64, :64])
    t2.close()


from tests.fixtures import write_vrt  # noqa: E402


VRT_PX = 8.3333333333330430e-05          # landcover/esa_worldcover_2021.vrt:3


def test_vrt_mosaic_reader(tmp_path):
    """esa_data_path = *.vrt (the reference's shipped config, raster.c:119): a 3 x 2 mosaic of 700 x 500 tiles with
    one tile missing from the VRT (ocean: reads as NoDataValue) -- size, geotransform (the exact decimal string
    GDAL writes), windows across source borders, host decode and compressed-tile parts."""
    import zlib
    from gcn10_b200 import synth
    tw_, th_ = 700, 500
    full = synth.esa_tile(3 * tw_, 2 * th_, 77, patch=60)
    gt = (-180.0, VRT_PX, 0.0, 84.0, 0.0, -VRT_PX)
    sources = []
    for r in range(2):
        for c in range(3):
            if (r, c) == (1, 2):
                full[r * th_:(r + 1) * th_, c * tw_:(c + 1) * tw_] = 0          # not in the mosaic
                continue
            name = f"tile & {r}_{c}.tif"
            hostlib.tiff_write(str(tmp_path / name), full[r * th_:(r + 1) * th_, c * tw_:(c + 1) * tw_],
                               (gt[0] + c * tw_ * VRT_PX, VRT_PX, 0, gt[3] - r * th_ * VRT_PX, 0, -VRT_PX))
            sources.append((name, 0, 0, c * tw_, r * th_, tw_, th_))
    vrt = write_vrt(str(tmp_path / "mosaic.vrt"), 3 * tw_, 2 * th_, gt, sources)
    r = hostlib.Raster(vrt)
    assert (r.width, r.height) == (3 * tw_, 2 * th_) and r.is_mosaic and r.source_count == 5 and r.fill == 0
    assert r.gt == gt                                            # bit-exact: feeds the window arithmetic
    for (xo, yo, xc, yc) in [(0, 0, 3 * tw_, 2 * th_), (650, 450, 101, 101), (699, 0, 2, 1000), (1390, 490, 30, 20),
                             (1500, 600, 100, 100), (0, 499, 2100, 2)]:
        assert np.array_equal(r.read(xo, yo, xc, yc), full[yo:yo + yc, xo:xo + xc]), (xo, yo, xc, yc)
        rc, parts = r.window_parts(xo, yo, xc, yc)
        assert rc == 0
        got = np.zeros((yc, xc), dtype=np.uint8)
        for p in parts:
            grid = np.zeros((p["tiles_y"] * p["tile_h"], p["tiles_x"] * p["tile_w"]), dtype=np.uint8)
            for i in range(p["tiles_y"] * p["tiles_x"]):
                o, n = int(p["offsets"][i]), int(p["sizes"][i])
                raw = zlib.decompress(p["blob"][o:o + n].tobytes())
                a, b = divmod(i, p["tiles_x"])
                grid[a * 256:(a + 1) * 256, b * 256:(b + 1) * 256] = np.frombuffer(raw, dtype=np.uint8).reshape(256, 256)
            got[p["dst_y"]:p["dst_y"] + p["h"], p["dst_x"]:p["dst_x"] + p["w"]] = \
                grid[p["y_in"]:p["y_in"] + p["h"], p["x_in"]:p["x_in"] + p["w"]]
        assert np.array_equal(got, full[yo:yo + yc, xo:xo + xc])
    with pytest.raises(hostlib.HostError):
        r.read(0, 0, 3 * tw_ + 1, 10)
    r.close()
    # a plain GeoTIFF opens through the same call: one part
    r1 = hostlib.Raster(str(tmp_path / "tile & 0_0.tif"))
    assert not r1.is_mosaic and r1.source_count == 1
    rc, parts = r1.window_parts(10, 20, 300, 300)
    assert rc == 0 and len(parts) == 1 and (parts[0]["dst_x"], parts[0]["w"]) == (0, 300)
    r1.close()


def test_vrt_remote_sources_missing_files_and_bad_documents(tmp_path, monkeypatch):
    from gcn10_b200 import synth
    a = synth.esa_tile(300, 300, 3, patch=30)
    os.makedirs(tmp_path / "tiles")
    hostlib.tiff_write(str(tmp_path / "tiles" / "ESA_A.tif"), a, (0, 1, 0, 0, 0, -1))
    src = [("ESA_A.tif", 0, 0, 0, 0, 300, 300), ("ESA_B.tif", 0, 0, 300, 0, 300, 300)]
    # /vsicurl/ sources (what the shipped VRT names) are looked up by base name in GCN10_VRT_SOURCE_DIR
    vrt = write_vrt(str(tmp_path / "remote.vrt"), 600, 300, (0, 1, 0, 0, 0, -1), src,
                    remote_prefix="/vsicurl/https://esa-worldcover.s3.eu-central-1.amazonaws.com/v200/2021/map/")
    monkeypatch.setenv("GCN10_VRT_SOURCE_DIR", str(tmp_path / "tiles"))
    r = hostlib.Raster(vrt)
    assert np.array_equal(r.read(0, 0, 300, 300), a)
    with pytest.raises(hostlib.HostError) as e:                  # ESA_B.tif does not exist: the read fails (block skipped)
        r.read(250, 0, 100, 100)
    assert "gdal open failed" in e.value.msg
    with pytest.raises(hostlib.HostError):
        r.window_parts(250, 0, 100, 100)
    r.close()
    # SimpleSource, shifted SrcRect, NoDataValue as fill
    vrt2 = write_vrt(str(tmp_path / "simple.vrt"), 400, 250, (5, 0.5, 0, 9, 0, -0.5),
                     [(str(tmp_path / "tiles" / "ESA_A.tif"), 40, 50, 100, 0, 200, 250)], kind="SimpleSource", nodata=80)
    r2 = hostlib.Raster(vrt2)
    want = np.full((250, 400), 80, dtype=np.uint8)
    want[:, 100:300] = a[50:300, 40:240]
    assert r2.fill == 80 and np.array_equal(r2.read(0, 0, 400, 250), want)
    r2.close()
    # scaling sources and non-VRT XML are refused at open
    bad = open(vrt2).read().replace('<DstRect xOff="100" yOff="0" xSize="200"', '<DstRect xOff="100" yOff="0" xSize="100"')
    open(tmp_path / "scaled.vrt", "w").write(bad)
    with pytest.raises(hostlib.HostError):
        hostlib.Raster(str(tmp_path / "scaled.vrt"))
    open(tmp_path / "junk.vrt", "w").write("<html></html>")
    with pytest.raises(hostlib.HostError):
        hostlib.Raster(str(tmp_path / "junk.vrt"))


def test_reference_vrt_if_present():
    vrt = "/root/reference/landcover/esa_worldcover_2021.vrt"
    if not os.path.exists(vrt):
        pytest.skip("reference tree not present")
    r = hostlib.Raster(vrt)
    assert (r.width, r.height) == (4320000, 1728000) and r.source_count == 2651 and r.fill == 0
    assert r.gt == (-180.0, VRT_PX, 0.0, 84.0, 0.0, -VRT_PX)
    # block 2234 (-114..-111, 39..42): the 36001 x 36001 window of SURVEY section 8
    assert hostlib.raster_window(r.width, r.height, r.gt, (-114.0, 39.0, -111.0, 42.0))[:4] == (792000, 504000, 36001, 36001)
    r.close()


def test_geotiff_writer_leaves_no_partial_file(tmp_path):
    """An output that is aborted or fails to close never appears under its final name (ADVICE r1: with overwrite off
    a re-run would keep the junk file and write beside it, cn.c:320-360)."""
    import zlib
    z = zlib.compress(bytes(65536))
    p = tmp_path / "cn_p_i_7.tif"
    tw = hostlib.TiffWriter(str(p), 256, 512, (0, 1, 0, 0, 0, -1))
    assert tw.put_tile_row(0, [z]) == 0
    assert not p.exists()                                       # still under its temporary name
    hostlib.load().gh_tiffw_abort(tw.h)
    assert not p.exists() and not list(tmp_path.glob("cn_p_i_7*"))
    tw = hostlib.TiffWriter(str(p), 256, 512, (0, 1, 0, 0, 0, -1))
    tw.put_tile_row(0, [z])
    assert tw.close() != 0 and not list(tmp_path.glob("cn_p_i_7*"))      # incomplete: removed
    tw = hostlib.TiffWriter(str(p), 256, 512, (0, 1, 0, 0, 0, -1))
    tw.put_tile_row(0, [z])
    tw.put_tile_row(1, [z])
    assert tw.close() == 0 and p.exists() and not (tmp_path / "cn_p_i_7.tif.part").exists()


def test_geokeys_travel_from_the_land_cover_to_the_outputs(tmp_path):
    """The reference copies the source dataset's projection into every raster it writes (raster.c:164-165,
    212-214): the GeoTIFF georeferencing tags of the input are re-emitted verbatim; a RasterPixelIsPoint source gets
    GDAL's half-pixel shift on the way in and the output is tagged PixelIsArea."""
    import struct
    import zlib
    L = hostlib.load()
    src = tmp_path / "utm.tif"
    a = np.arange(64 * 48, dtype=np.uint8).reshape(48, 64)
    # a striped uncompressed TIFF with a projected CRS (EPSG:32612) and RasterPixelIsPoint
    keys = [1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 2, 3072, 0, 1, 32612]
    data = a.tobytes()
    ifd_off = 8 + len(data)
    scale_off = ifd_off + 2 + 12 * 11 + 4
    tie_off = scale_off + 24
    keys_off = tie_off + 48
    ents = [(256, 4, 1, 64), (257, 4, 1, 48), (258, 3, 1, 8), (259, 3, 1, 1), (262, 3, 1, 1), (273, 4, 1, 8),
            (277, 3, 1, 1), (279, 4, 1, len(data)), (33550, 12, 3, scale_off), (33922, 12, 6, tie_off),
            (34735, 3, len(keys), keys_off)]
    with open(src, "wb") as f:
        f.write(struct.pack("<2sHI", b"II", 42, ifd_off) + data + struct.pack("<H", len(ents)))
        for tag, typ, cnt, val in ents:
            f.write(struct.pack("<HHIHH", tag, typ, cnt, val, 0) if typ == 3 and cnt == 1 else struct.pack("<HHII", tag, typ, cnt, val))
        f.write(struct.pack("<I", 0) + struct.pack("<3d", 10.0, 10.0, 0.0) + struct.pack("<6d", 0, 0, 0, 500000.0, 4100000.0, 0.0)
                + struct.pack(f"<{len(keys)}H", *keys))
    t = hostlib.Tiff(str(src))
    assert t.gt == (500000.0 - 5.0, 10.0, 0.0, 4100000.0 + 5.0, 0.0, -10.0)        # PixelIsPoint: half a pixel up-left
    assert np.array_equal(t.read(), a)

    class GK(hostlib.C.Structure):
        _fields_ = [("keys", hostlib.C.c_void_p), ("n_keys", hostlib.C.c_size_t), ("doubles", hostlib.C.c_void_p),
                    ("n_doubles", hostlib.C.c_size_t), ("ascii", hostlib.C.c_void_p), ("n_ascii", hostlib.C.c_size_t)]
    gk = GK()
    L.gh_tiff_geokeys.argtypes = [hostlib.C.c_void_p, hostlib.C.POINTER(GK)]
    L.gh_tiffw_set_geokeys.argtypes = [hostlib.C.c_void_p, hostlib.C.POINTER(GK)]
    assert L.gh_tiff_geokeys(t.h, hostlib.C.byref(gk)) == 0 and gk.n_keys == len(keys)
    out = tmp_path / "out.tif"
    tw = hostlib.TiffWriter(str(out), 256, 256, t.gt)
    assert L.gh_tiffw_set_geokeys(tw.h, hostlib.C.byref(gk)) == 0
    tw.put_tile_row(0, [zlib.compress(bytes(65536))])
    assert tw.close() == 0
    t.close()
    o = hostlib.Tiff(str(out))
    assert o.gt == (499995.0, 10.0, 0.0, 4100005.0, 0.0, -10.0)                    # written as a corner: read back unshifted
    gk2 = GK()
    assert L.gh_tiff_geokeys(o.h, hostlib.C.byref(gk2)) == 0
    got = list((hostlib.C.c_uint16 * gk2.n_keys).from_address(gk2.keys))
    assert got == keys[:11] + [1] + keys[12:]                                       # same keys, RasterType -> PixelIsArea
    o.close()
    # a file without geokeys: the writer keeps its EPSG:4326 default
    hostlib.tiff_write(str(tmp_path / "plain.tif"), a, (0, 1, 0, 0, 0, -1))
    p = hostlib.Tiff(str(tmp_path / "plain.tif"))
    gk3 = GK()
    assert L.gh_tiff_geokeys(p.h, hostlib.C.byref(gk3)) == 0
    assert 4326 in list((hostlib.C.c_uint16 * gk3.n_keys).from_address(gk3.keys))
    p.close()


def test_geotiff_writer_takes_several_ordered_tile_rows_in_one_write(tmp_path):
    """gh_tiffw_put_tile_rows: tiles laid out in table order with alignment gaps (the library's "ordered" strips) go to
    the file with one write; any other layout falls back to tile-by-tile appends.  Both files decode to the raster."""
    import zlib
    from gcn10_b200 import synth
    L = hostlib.load()
    w, h = 700, 600
    a = synth.esa_tile(w, h, 9, patch=30)
    tx, ty = 3, 3
    streams = []
    for r in range(ty):
        for c in range(tx):
            t = np.zeros((256, 256), dtype=np.uint8)
            part = a[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256]
            t[:part.shape[0], :part.shape[1]] = part
            streams.append(zlib.compress(t.tobytes(), 6))
    for name, order in (("ordered", list(range(9))), ("scattered", [4, 0, 8, 2, 6, 1, 7, 3, 5])):
        blob = bytearray()
        offs, sizes = [0] * 9, [0] * 9
        for i in order:
            while len(blob) % 16:
                blob.append(0xAA)                      # alignment padding between the streams
            offs[i], sizes[i] = len(blob), len(streams[i])
            blob += streams[i]
        buf = hostlib.C.create_string_buffer(bytes(blob), len(blob))
        p = tmp_path / f"{name}.tif"
        tw = hostlib.TiffWriter(str(p), w, h, (0, 1, 0, 0, 0, -1))
        o = (hostlib.C.c_uint64 * 9)(*offs)
        z = (hostlib.C.c_uint32 * 9)(*sizes)
        assert L.gh_tiffw_put_tile_rows(tw.h, 0, 2, buf, o, z) == 0
        assert L.gh_tiffw_put_tile_rows(tw.h, 2, 1, buf, hostlib.C.cast(hostlib.C.byref(o, 6 * 8), hostlib.C.POINTER(hostlib.C.c_uint64)),
                                        hostlib.C.cast(hostlib.C.byref(z, 6 * 4), hostlib.C.POINTER(hostlib.C.c_uint32))) == 0
        assert tw.close() == 0
        t = hostlib.Tiff(str(p))
        assert np.array_equal(t.read(), a), name
        t.close()


def _ifd_entries(b):
    ifd = struct.unpack_from("<I", b, 4)[0]
    n = struct.unpack_from("<H", b, ifd)[0]
    return ifd, {struct.unpack_from("<H", b, ifd + 2 + 12 * i)[0]: ifd + 2 + 12 * i for i in range(n)}


def test_geotiff_reader_survives_damaged_directories(tmp_path):
    """Input files are not trusted: a damaged TIFF directory (found by mutation fuzzing under ASan: zero tile sizes
    divided, counts sized allocations) must be refused like GDAL refuses it -- an error, the block is skipped
    (raster.c:121, cn.c:188-192) -- never a crash."""
    a = (np.arange(300 * 520).reshape(300, 520) % 7 * 10).astype(np.uint8)
    p = str(tmp_path / "ok.tif")
    hostlib.tiff_write(p, a, (-114.0, PX, 0.0, 42.0, 0.0, -PX), threads=2)
    good = open(p, "rb").read()
    ifd, ent = _ifd_entries(good)

    def damaged(edit):
        b = bytearray(good)
        edit(b)
        q = str(tmp_path / "bad.tif")
        open(q, "wb").write(b)
        return q

    cases = {
        "tile width 0": lambda b: struct.pack_into("<I", b, ent[322] + 8, 0),
        "tile length 0": lambda b: struct.pack_into("<I", b, ent[323] + 8, 0),
        "tile width type unknown": lambda b: struct.pack_into("<H", b, ent[322] + 2, 99),
        "huge tile": lambda b: (struct.pack_into("<HI", b, ent[322] + 2, 4, 1), struct.pack_into("<I", b, ent[322] + 8, 0x7FFFFFFF),
                                struct.pack_into("<HI", b, ent[323] + 2, 4, 1), struct.pack_into("<I", b, ent[323] + 8, 0x7FFFFFFF)),
        "directory offset outside the file": lambda b: struct.pack_into("<I", b, 4, 0xFFFFFF00),
        "directory longer than the file": lambda b: struct.pack_into("<H", b, ifd, 0xFFFF),
        "offset table outside the file": lambda b: struct.pack_into("<I", b, ent[324] + 8, 0xFFFFFF00),
        "image 2^31 wide": lambda b: struct.pack_into("<I", b, ent[256] + 8, 0x80000000),
        "truncated": lambda b: b.__delitem__(slice(ifd + 20, None)),
    }
    for name, edit in cases.items():
        with pytest.raises(hostlib.HostError) as e:
            hostlib.Raster(damaged(edit))
        assert "gdal open failed" in e.value.msg, name
    # a count larger than the tile grid needs is tolerated: only the grid's entries are read
    r = hostlib.Raster(damaged(lambda b: struct.pack_into("<I", b, ent[324] + 4, 0xFFFFFFFF)))
    assert np.array_equal(r.read(0, 0, 520, 300), a)
    r.close()
    # tile tables that point outside the file: the file opens, the read fails, compressed tiles are not handed out
    def far_tile(b):
        off = struct.unpack_from("<I", b, ent[324] + 8)[0]
        struct.pack_into("<I", b, off, 0xFFFFFF00)
    r = hostlib.Raster(damaged(far_tile))
    with pytest.raises(hostlib.HostError) as e:
        r.read(0, 0, 520, 300)
    assert "gdalrasterio error" in e.value.msg                      # raster.c:182
    rc, parts = r.window_parts(0, 0, 520, 300)
    assert rc == 1 and parts == []
    r.close()
    def long_tile(b):
        cnt = struct.unpack_from("<I", b, ent[325] + 8)[0]
        struct.pack_into("<I", b, cnt, 0xFFFFFFF0)
    r = hostlib.Raster(damaged(long_tile))
    with pytest.raises(hostlib.HostError):
        r.read(0, 0, 520, 300)
    assert r.window_parts(0, 0, 520, 300)[0] == 1
    r.close()


def test_shapefile_reader_survives_damaged_attribute_tables(tmp_path):
    """Same for the block shapefile (cn.c:155-184 reads it through OGR): header lengths, record lengths and field
    widths out of a damaged .dbf must not index past the file."""
    shp = str(tmp_path / "b.shp")
    fixtures.write_block_shapefile(shp, [(2234, -114.0, 39.0, -111.0, 42.0), (7, 0.0, 0.0, 3.0, 3.0)])
    dbf_path = str(tmp_path / "b.dbf")
    good = open(dbf_path, "rb").read()
    assert hostlib.Blocks(shp).bbox(7) == (0.0, 0.0, 3.0, 3.0)
    cases = {
        "header length beyond the file": lambda b: struct.pack_into("<H", b, 8, 0xFFF0),
        "record length 0": lambda b: struct.pack_into("<H", b, 10, 0),
        "record count absurd": lambda b: struct.pack_into("<I", b, 4, 0xFFFFFFFF),
        "field wider than the record": lambda b: b.__setitem__(32 + 16, 255),
        "no field terminator": lambda b: b.__setitem__(b.index(0x0D), 0x41),
    }
    for name, edit in cases.items():
        b = bytearray(good)
        edit(b)
        open(dbf_path, "wb").write(b)
        try:
            blocks = hostlib.Blocks(shp)
            blocks.bbox(2234)               # whatever it holds, reading it back must be safe
        except hostlib.HostError as e:
            assert "ogr open failed" in e.msg, name
    # the geometry file: a record length that points far past the end stops the walk
    open(dbf_path, "wb").write(good)
    sb = bytearray(open(shp, "rb").read())
    struct.pack_into(">I", sb, 100 + 4, 0x7FFFFFFF)
    open(shp, "wb").write(sb)
    blocks = hostlib.Blocks(shp)
    assert len(blocks) == 0
