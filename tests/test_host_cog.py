"""CPU tests of the Cloud Optimized GeoTIFF layout of the GeoTIFF writer (gh_tiffw_set_cog, gh_tiffw_put_level_tile_rows,
gh_tiffw_put_framed_tile_rows, gh_tiff_write_cog) against tests/cog_rule.py; Pillow's libtiff reader reads the pixels
and the tags back independently."""
import os
import zlib

import numpy as np
import pytest
from PIL import Image

from gcn10_b200 import hostlib
from tests import cog_rule, stats_rule
from tests import overview_rule as R
from tests.tiff_cases import GT, SIZES, raster, tile_rows

# the land cover's GeoKeys as the writer copies them (a projected CRS with double and ascii params)
GEOKEYS = ([1, 1, 0, 4, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 32611, 3076, 34736, 1, 0],
           [1.0], "WGS 84 / UTM zone 11N|")


def _frames(path):
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append((np.array(im), dict(im.tag_v2)))
    return out


def _check_pixels(path, a, nlev):
    frames = _frames(path)
    assert len(frames) == nlev + 1
    assert np.array_equal(frames[0][0], a)
    for k in range(1, nlev + 1):
        assert frames[k][1].get(254) == 1, k
        assert np.array_equal(frames[k][0], R.decimate(a, k)), k
    return frames


def _plain(rows):
    """blob, offsets, sizes of tile rows laid end to end, unframed."""
    flat = [z for row in rows for z in row]
    offs = np.cumsum([0] + [len(z) for z in flat[:-1]]).astype(np.uint64)
    return b"".join(flat), offs, np.array([len(z) for z in flat], np.uint32)


def _framed(rows):
    """The same tiles as the library's framed strips lay them: 16-byte aligned streams, the first leader in the first 16
    bytes, each slot round16(size + 8) = stream | trailer | zeros | the next tile's leader."""
    flat = [z for row in rows for z in row]
    buf = bytearray(16)
    offs = []
    for i, z in enumerate(flat):
        at = len(buf)
        offs.append(at)
        slot = (len(z) + 8 + 15) & ~15
        buf += z + z[-4:] + bytes(slot - len(z) - 8) + (len(flat[i + 1]).to_bytes(4, "little") if i + 1 < len(flat)
                                                        else bytes(4))
        buf[at - 4:at] = len(z).to_bytes(4, "little")
    return bytes(buf), np.array(offs, np.uint64), np.array([len(z) for z in flat], np.uint32)


def _put_level(tw, k, img, framed, rows_per_call=3):
    rows = tile_rows(img)
    for r0 in range(0, len(rows), rows_per_call):
        part = rows[r0:r0 + rows_per_call]
        blob, offs, sizes = (_framed if framed else _plain)(part)
        assert tw.put_tile_rows(k, r0, len(part), blob, offs, sizes, framed=framed) == 0, (k, r0)


@pytest.mark.parametrize("w,h", SIZES)
def test_whole_raster_cog(tmp_path, w, h):
    """gh_tiff_write_cog, the CPU reference: rules 1-4 hold and every IFD decodes to the raster and its levels."""
    a = raster(w, h, seed=w * 3 + h)
    path = str(tmp_path / "c.tif")
    hostlib.tiff_write_cog(path, a, GT, 16)
    ifds = cog_rule.check(path)
    assert len(ifds) == R.levels(w, h) + 1
    _check_pixels(path, a, R.levels(w, h))
    t = hostlib.Tiff(path)                       # the project's own reader reads IFD0 of a COG too
    assert np.array_equal(t.read(), a)
    t.close()


@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("tags", ["plain", "stats", "nodata", "geokeys", "stats+geokeys"])
@pytest.mark.parametrize("overviews", [0, 16])
@pytest.mark.parametrize("framed", [False, True])
def test_writer_cog(tmp_path, w, h, tags, overviews, framed):
    a = raster(w, h, seed=w + 5 * h)
    nlev = R.levels(w, h) if overviews else 0
    path = str(tmp_path / "c.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=overviews, stats="stats" in tags, nodata=tags == "nodata",
                            geokeys=GEOKEYS if "geokeys" in tags else None, cog=True)
    assert tw.levels == nlev
    for k in range(nlev, -1, -1):
        _put_level(tw, k, R.decimate(a, k) if k else a, framed)
    if "stats" in tags:
        assert tw.put_histogram(np.bincount(a.ravel(), minlength=256)) == 0
    assert tw.close() == 0
    ifds = cog_rule.check(path)
    assert len(ifds) == nlev + 1
    frames = _check_pixels(path, a, nlev)
    tag0 = frames[0][1]
    if "stats" in tags:
        assert stats_rule.close(stats_rule.parse(tag0[42112]), stats_rule.of_plane(a))
    else:
        assert 42112 not in tag0
    if tags in ("stats", "nodata", "stats+geokeys"):
        assert all(f[1].get(42113) == "255" for f in frames)
    else:
        assert all(42113 not in f[1] for f in frames)
    if "geokeys" in tags:
        assert list(tag0[34735]) == GEOKEYS[0]
        assert tag0[34737] == GEOKEYS[2]


def test_same_streams_as_plain_layout(tmp_path):
    """Same tile streams, different order and framing: the tiles of a COG are byte for byte those of the plain file."""
    w, h = 3001, 517
    a = raster(w, h, seed=11)
    plain, cog = str(tmp_path / "p.tif"), str(tmp_path / "c.tif")
    tw = hostlib.TiffWriter(plain, w, h, GT, overviews=16)
    for y0 in range(0, h, 512):
        assert tw.write_rows(a[y0:y0 + 512], y0) == 0
    assert tw.close() == 0
    hostlib.tiff_write_cog(cog, a, GT, 16)
    ifds = cog_rule.check(cog)
    with open(plain, "rb") as f:
        pdata = f.read()
    with open(cog, "rb") as f:
        cdata = f.read()
    with Image.open(plain) as im:
        for k, d in enumerate(ifds):
            im.seek(k)
            po, pc = im.tag_v2[324], im.tag_v2[325]
            po, pc = (po,) if isinstance(po, int) else po, (pc,) if isinstance(pc, int) else pc
            assert list(pc) == d["counts"]
            for o1, o2, n in zip(po, d["offsets"], d["counts"]):
                assert pdata[o1:o1 + n] == cdata[o2:o2 + n]


def test_rule_rejects_plain_overviews(tmp_path):
    """A file in the plain layout (level data behind the full resolution, IFDs at the end) is not a COG."""
    w, h = 4111, 260
    a = raster(w, h, seed=3)
    path = str(tmp_path / "p.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=16)
    assert tw.write_rows(a, 0) == 0
    assert tw.close() == 0
    with pytest.raises(AssertionError):
        cog_rule.check(path)


def test_rule_rejects_altered_trailer(tmp_path):
    w, h = 4111, 260
    a = raster(w, h, seed=4)
    path = str(tmp_path / "c.tif")
    hostlib.tiff_write_cog(path, a, GT, 16)
    ifds = cog_rule.check(path)
    o, n = ifds[0]["offsets"][5], ifds[0]["counts"][5]
    with open(path, "r+b") as f:
        f.seek(o + n + 2)
        b = f.read(1)
        f.seek(o + n + 2)
        f.write(bytes([b[0] ^ 1]))
    with pytest.raises(AssertionError, match="trailer"):
        cog_rule.check(path)


def _left_behind(tmp_path):
    return sorted(os.listdir(tmp_path))


@pytest.mark.parametrize("order", ["full_first", "largest_first", "skip_level"])
def test_out_of_order_levels_refused(tmp_path, order):
    w, h = 3001, 517
    a = raster(w, h, seed=5)
    nlev = R.levels(w, h)
    assert nlev >= 2
    path = str(tmp_path / "c.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=16, cog=True)
    first = {"full_first": 0, "largest_first": 1, "skip_level": nlev - 1}[order]
    rows = tile_rows(R.decimate(a, first) if first else a)
    blob, offs, sizes = _plain(rows[:1])
    assert tw.put_tile_rows(first, 0, 1, blob, offs, sizes) != 0
    assert tw.close() != 0
    assert _left_behind(tmp_path) == []


def test_bad_framing_refused(tmp_path):
    w, h = 600, 300
    a = raster(w, h, seed=6)
    path = str(tmp_path / "c.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, cog=True)
    blob, offs, sizes = _framed(tile_rows(a))
    bad = bytearray(blob)
    bad[int(offs[1]) - 4] ^= 1                  # tile 1's leader
    assert tw.put_tile_rows(0, 0, 2, bytes(bad), offs, sizes, framed=True) != 0
    assert tw.close() != 0
    assert _left_behind(tmp_path) == []


def test_cog_refuses_bands_and_late_settings(tmp_path):
    w, h = 600, 300
    a = raster(w, h, seed=7)
    path = str(tmp_path / "c.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, stats=True, cog=True)
    assert tw.write_rows(a, 0) != 0                                     # bands: the levels would trail
    assert tw.L.gh_tiffw_set_nodata(tw.h, 1) != 0                       # the header region is sized already
    assert tw.L.gh_tiffw_set_cog(tw.h, 1) != 0
    rows = tile_rows(a)
    blob, offs, sizes = _plain(rows)
    assert tw.put_tile_rows(0, 0, len(rows), blob, offs, sizes) == 0
    assert tw.put_histogram(np.bincount(a.ravel(), minlength=256)) == 0
    assert tw.close() == 0
    cog_rule.check(path)
    assert np.array_equal(_frames(path)[0][0], a)


def test_streams_decode(tmp_path):
    """Each framed tile is still a complete zlib stream of its 256 x 256 tile."""
    w, h = 700, 513
    a = raster(w, h, seed=8)
    path = str(tmp_path / "c.tif")
    hostlib.tiff_write_cog(path, a, GT, 16)
    ifds = cog_rule.check(path)
    with open(path, "rb") as f:
        data = f.read()
    tiles = tile_rows(a)
    flat = [z for row in tiles for z in row]
    for o, n, z in zip(ifds[0]["offsets"], ifds[0]["counts"], flat):
        assert zlib.decompress(data[o:o + n]) == zlib.decompress(z)
