"""CPU tests of the statistics of the GeoTIFF writer (gh_tiffw_set_stats, gh_tiffw_put_histogram, gh_tiffw_write_rows,
gh_tiffw_close): GDAL_NODATA (42113) "255" in every IFD, GDAL_METADATA (42112) with the band statistics in IFD0 only,
equal to tests/stats_rule.py applied to the plane.  Pillow's libtiff reader is the independent reader of the files."""
import os
import zlib

import numpy as np
import pytest
from PIL import Image

from gcn10_b200 import hostlib
from tests import overview_rule as R
from tests import stats_rule as S

GT = (-114.0, 1.0 / 12000.0, 0.0, 42.0, 0.0, -1.0 / 12000.0)


def _plane(kind, w, h, seed):
    rng = np.random.default_rng(seed)
    if kind == "only_nodata":
        return np.full((h, w), 255, np.uint8)
    if kind == "single":
        return np.full((h, w), 77, np.uint8)
    a = rng.integers(0, 12, size=((h + 6) // 7, (w + 4) // 5), dtype=np.uint8) * 21       # patches, like land cover
    a = np.repeat(np.repeat(a, 7, axis=0), 5, axis=1)[:h, :w] + rng.integers(0, 3, size=(h, w), dtype=np.uint8)
    if kind == "with_nodata":
        a[rng.random((h, w)) < 0.3] = 255
    return np.ascontiguousarray(a)                    # "no_nodata": at most 233


def _tags(path):
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append((np.array(im), im.tag_v2.get(42113), im.tag_v2.get(42112)))
    return out


def _check(path, a, nlev):
    frames = _tags(path)
    assert len(frames) == nlev + 1
    assert np.array_equal(frames[0][0], a)
    assert all(nodata == "255" for _, nodata, _ in frames)
    assert all(meta is None for _, _, meta in frames[1:])
    got = S.parse(frames[0][2])
    want = S.of_plane(a)
    assert S.close(got, want), (got, want)
    return got


def _tile_rows(img):
    h, w = img.shape
    out = []
    for ty in range(0, h, 256):
        row = []
        for tx in range(0, w, 256):
            t = np.zeros((256, 256), np.uint8)
            part = img[ty:ty + 256, tx:tx + 256]
            t[:part.shape[0], :part.shape[1]] = part
            row.append(zlib.compress(t.tobytes(), 6))
        out.append(row)
    return out


KINDS = ["no_nodata", "with_nodata", "only_nodata", "single"]
SIZES = [(1, 1), (257, 257), (3001, 517), (48, 1300)]


@pytest.mark.parametrize("overviews", [0, 16], ids=["no_overviews", "overviews"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("w,h", SIZES)
def test_write_rows_stats(tmp_path, w, h, kind, overviews):
    a = _plane(kind, w, h, seed=w + 5 * h)
    path = str(tmp_path / "s.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=overviews, stats=True)
    for y0 in range(0, h, 512):
        assert tw.write_rows(a[y0:y0 + 512], y0) == 0
    assert tw.close() == 0
    got = _check(path, a, R.levels(w, h) if overviews else 0)
    if kind == "only_nodata":
        assert got == {"STATISTICS_VALID_PERCENT": 0.0}
    if kind == "single":
        assert got["STATISTICS_MINIMUM"] == got["STATISTICS_MAXIMUM"] == got["STATISTICS_MEAN"] == 77.0
        assert got["STATISTICS_STDDEV"] == 0.0 and got["STATISTICS_VALID_PERCENT"] == 100.0


def _put(path, a, overviews=0, hist=True):
    h, w = a.shape
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=overviews, stats=True)
    for level in range(tw.levels + 1):
        for r, streams in enumerate(_tile_rows(R.decimate(a, level) if level else a)):
            assert tw.put_tile_row(r, streams, level=level) == 0
    if hist is True:
        hist = np.bincount(a.ravel(), minlength=256)
    if hist is not None:
        assert tw.put_histogram(hist) == 0
    return tw


@pytest.mark.parametrize("kind", KINDS)
def test_put_histogram_same_file_as_write_rows(tmp_path, kind):
    w, h = 3001, 517
    a = _plane(kind, w, h, seed=3)
    p1, p2 = str(tmp_path / "rows.tif"), str(tmp_path / "put.tif")
    tw = hostlib.TiffWriter(p1, w, h, GT, stats=True)
    assert tw.write_rows(a, 0) == 0
    assert tw.close() == 0
    assert _put(p2, a).close() == 0
    assert open(p1, "rb").read() == open(p2, "rb").read()
    # with overviews the tiles lie in another order, the tags are the same
    p3 = str(tmp_path / "put_ov.tif")
    assert _put(p3, a, overviews=16).close() == 0
    _check(p3, a, R.levels(w, h))


def test_histogram_in_two_parts_adds_up(tmp_path):
    a = _plane("with_nodata", 700, 300, seed=4)
    hist = np.bincount(a.ravel(), minlength=256).astype(np.uint64)
    half = hist // np.uint64(2)
    tw = _put(str(tmp_path / "two.tif"), a, hist=half)
    assert tw.put_histogram(hist - half) == 0
    assert tw.close() == 0
    _check(str(tmp_path / "two.tif"), a, 0)


@pytest.mark.parametrize("case", ["short", "long", "missing"])
def test_wrong_or_missing_histogram_fails_and_leaves_no_file(tmp_path, case):
    a = _plane("with_nodata", 600, 300, seed=5)
    hist = np.bincount(a.ravel(), minlength=256).astype(np.uint64)
    if case == "short":
        hist[int(hist.argmax())] -= np.uint64(1)
    elif case == "long":
        hist[255] += np.uint64(1)
    path = str(tmp_path / "bad.tif")
    tw = _put(path, a, hist=None if case == "missing" else hist)
    assert tw.close() != 0
    assert not os.path.exists(path) and not os.path.exists(path + ".part")


def test_without_stats_no_tags(tmp_path):
    a = _plane("with_nodata", 600, 300, seed=6)
    for overviews in (0, 16):
        path = str(tmp_path / f"n{overviews}.tif")
        tw = hostlib.TiffWriter(path, 600, 300, GT, overviews=overviews)
        assert tw.put_histogram(np.zeros(256, np.uint64)) != 0      # no statistics to feed
        assert tw.write_rows(a, 0) == 0
        assert tw.close() == 0
        frames = _tags(path)
        assert len(frames) == (R.levels(600, 300) if overviews else 0) + 1
        assert all(nodata is None and meta is None for _, nodata, meta in frames)
        assert np.array_equal(frames[0][0], a)


def test_set_stats_only_before_data(tmp_path):
    a = _plane("single", 300, 300, seed=7)
    tw = hostlib.TiffWriter(str(tmp_path / "late.tif"), 300, 300, GT)
    assert tw.write_rows(a, 0) == 0
    assert tw.L.gh_tiffw_set_stats(tw.h, 1) != 0
    tw.L.gh_tiffw_abort(tw.h)


def test_exact_at_full_size(tmp_path):
    """36001 x 36001 pixels, 0 and 254 in equal parts and one nodata pixel: N * sum(v^2) is past 64 bits, mean and
    standard deviation stay exact.  (The tiles are all one stream: only the histogram matters here.)"""
    n = 36001
    hist = np.zeros(256, np.uint64)
    hist[0] = hist[254] = (n * n) // 2
    hist[255] = 1
    assert int(hist[0]) * int(hist[254]) * 254 * 254 > 2 ** 64
    z = zlib.compress(bytes(256 * 256), 6)
    path = str(tmp_path / "big.tif")
    tw = hostlib.TiffWriter(path, n, n, GT, stats=True)
    tiles = (n + 255) // 256
    for r in range(tiles):
        assert tw.put_tile_row(r, [z] * tiles) == 0
    assert tw.put_histogram(hist) == 0
    assert tw.close() == 0
    limit, Image.MAX_IMAGE_PIXELS = Image.MAX_IMAGE_PIXELS, None      # (only the tags are read)
    try:
        with Image.open(path) as im:
            got = S.parse(im.tag_v2.get(42112))
    finally:
        Image.MAX_IMAGE_PIXELS = limit
    want = S.from_histogram(hist, n * n)
    assert want["STATISTICS_MEAN"] == 127.0 and want["STATISTICS_STDDEV"] == 127.0
    assert S.close(got, want), (got, want)


def _ifd0_entries(path):
    import struct
    data = open(path, "rb").read()
    (off,) = struct.unpack_from("<I", data, 4)
    (n,) = struct.unpack_from("<H", data, off)
    return {tag: (typ, cnt, val) for tag, typ, cnt, val in
            (struct.unpack_from("<HHII", data, off + 2 + 12 * i) for i in range(n))}, data


@pytest.mark.parametrize("ascii_len", [7, 8])
def test_metadata_offset_word_aligned(tmp_path, ascii_len):
    """GeoAsciiParams of odd length copied from a source: the GDAL_METADATA value still starts on a word boundary
    (TIFF 6.0), and the tags keep ascending order."""
    import ctypes as C

    class GeoKeys(C.Structure):
        _fields_ = [("keys", C.POINTER(C.c_uint16)), ("n_keys", C.c_size_t), ("doubles", C.POINTER(C.c_double)),
                    ("n_doubles", C.c_size_t), ("ascii", C.c_char_p), ("n_ascii", C.c_size_t)]

    keys = (C.c_uint16 * 16)(1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2049, 34737, ascii_len, 0)
    text = (b"WGS 84|" + b"x" * 8)[:ascii_len - 1] + b"\0"
    gk = GeoKeys(keys, 16, None, 0, text, ascii_len)
    a = _plane("with_nodata", 300, 200, seed=8)
    path = str(tmp_path / "g.tif")
    tw = hostlib.TiffWriter(path, 300, 200, GT, stats=True)
    tw.L.gh_tiffw_set_geokeys.argtypes = [C.c_void_p, C.POINTER(GeoKeys)]
    assert tw.L.gh_tiffw_set_geokeys(tw.h, C.byref(gk)) == 0
    assert tw.write_rows(a, 0) == 0
    assert tw.close() == 0
    ent, data = _ifd0_entries(path)
    assert list(ent) == sorted(ent) and ent[34737][1] == ascii_len
    typ, cnt, off = ent[42112]
    assert typ == 2 and off % 2 == 0
    assert S.close(S.parse(data[off:off + cnt - 1].decode()), S.of_plane(a))
    assert _check(path, a, 0)
