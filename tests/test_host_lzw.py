"""Host reader: tiled LZW GeoTIFFs without predictor are handed to the GPU as compressed tiles (CPU only).

The files are written by libtiff (gcn10_b200/tiff_lzw.py), so the tile streams are libtiff's; the plan must return
them untouched with the file's compression, per source of a VRT mosaic that mixes DEFLATE and LZW files.  LZW with
predictor 2 and stripped LZW files still go to the host decoder."""
import numpy as np

from gcn10_b200 import hostlib, synth, tiff_lzw
from tests.fixtures import write_vrt


def _assemble(p, decode):
    grid = np.zeros((p["tiles_y"] * p["tile_h"], p["tiles_x"] * p["tile_w"]), dtype=np.uint8)
    for i in range(p["tiles_y"] * p["tiles_x"]):
        o, n = int(p["offsets"][i]), int(p["sizes"][i])
        a, b = divmod(i, p["tiles_x"])
        grid[a * p["tile_h"]:(a + 1) * p["tile_h"], b * p["tile_w"]:(b + 1) * p["tile_w"]] = \
            decode(p["blob"][o:o + n].tobytes(), p["tile_w"], p["tile_h"])
    return grid[p["y_in"]:, p["x_in"]:]


def test_lzw_window_tiles_are_the_files_streams(tmp_path):
    a = synth.esa_tile(517, 333, 7, patch=30)
    path = tmp_path / "lzw.tif"
    tiff_lzw.write_file(path, a, tile=128)
    t = hostlib.Tiff(str(path))
    assert np.array_equal(t.read(), a)
    for (xo, yo, xc, yc) in [(0, 0, 517, 333), (100, 130, 300, 150), (516, 332, 1, 1)]:
        tl = t.window_tiles(xo, yo, xc, yc)
        assert tl is not None and tl["compression"] == 5 and tl["tile_w"] == 128
        got = _assemble(tl, tiff_lzw.decode)[:yc, :xc]
        assert np.array_equal(got, a[yo:yo + yc, xo:xo + xc])
    t.close()


def test_lzw_with_predictor_or_strips_stays_on_the_host(tmp_path):
    a = synth.esa_tile(300, 200, 9, patch=20)
    for name, kw in [("pred2.tif", dict(tile=64, predictor=2)), ("strips.tif", dict(tile=None))]:
        tiff_lzw.write_file(tmp_path / name, a, **kw)
        t = hostlib.Tiff(str(tmp_path / name))
        assert t.window_tiles() is None
        assert np.array_equal(t.read(), a)
        t.close()
        r = hostlib.Raster(str(tmp_path / name))
        assert r.window_parts(0, 0, 300, 200) == (1, [])
        r.close()


def test_vrt_mixing_deflate_and_lzw_sources(tmp_path):
    import zlib
    tw_, th_ = 400, 300
    full = synth.esa_tile(2 * tw_, th_, 21, patch=40)
    gt = (0.0, 1.0, 0.0, 0.0, 0.0, -1.0)
    hostlib.tiff_write(str(tmp_path / "a.tif"), full[:, :tw_], gt)
    tiff_lzw.write_file(tmp_path / "b.tif", full[:, tw_:], tile=256)
    vrt = write_vrt(str(tmp_path / "mix.vrt"), 2 * tw_, th_, gt,
                    [("a.tif", 0, 0, 0, 0, tw_, th_), ("b.tif", 0, 0, tw_, 0, tw_, th_)])
    r = hostlib.Raster(vrt)
    assert np.array_equal(r.read(0, 0, 2 * tw_, th_), full)
    rc, parts = r.window_parts(350, 10, 200, 250)
    assert rc == 0 and [p["compression"] for p in parts] == [8, 5]
    decoders = {8: lambda s, w, h: np.frombuffer(zlib.decompress(s), np.uint8).reshape(h, w), 5: tiff_lzw.decode}
    got = np.zeros((250, 200), dtype=np.uint8)
    for p in parts:
        got[p["dst_y"]:p["dst_y"] + p["h"], p["dst_x"]:p["dst_x"] + p["w"]] = \
            _assemble(p, decoders[p["compression"]])[:p["h"], :p["w"]]
    assert np.array_equal(got, full[10:260, 350:550])
    r.close()
