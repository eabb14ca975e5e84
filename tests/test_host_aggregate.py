"""CPU tests of the host's mean rasters (gh_aggregate_rows, gh_aggregate_write_rows) and of the NoData tag alone
(gh_tiffw_set_nodata): the host aggregation must equal tests/aggregate_rule.py, the numpy restatement of the rule in
include/gcn10_cuda.h, for any band split; the mean file must be ceil(w / f) x ceil(h / f) with the scaled geotransform,
the writer's GeoKeys, GDAL_NODATA "255" in every IFD and no GDAL_METADATA.  Pillow's libtiff reader is the independent
reader of the files."""
import numpy as np
import pytest
from PIL import Image

from gcn10_b200 import hostlib
from tests import aggregate_rule as A

GT = (-114.0, 1.0 / 12000.0, 0.0, 42.0, 0.0, -1.0 / 12000.0)


def _plane(w, h, seed, nodata=0.2):
    rng = np.random.default_rng(seed)
    a = rng.integers(30, 100, size=((h + 8) // 9, (w + 10) // 11), dtype=np.uint8)     # patches, like land cover
    a = np.repeat(np.repeat(a, 9, axis=0), 11, axis=1)[:h, :w] + rng.integers(0, 3, size=(h, w), dtype=np.uint8)
    a[rng.random((h, w)) < nodata] = 255
    return np.ascontiguousarray(a)


def _host(plane, f, bands):
    """The host aggregation fed in the given band heights; every completed cell row comes back once, in order."""
    h, w = plane.shape
    ag = hostlib.Aggregate(w, h, f)
    rows, y0 = [], 0
    try:
        for b in bands:
            r0, out = ag.rows(plane[y0:y0 + b], y0)
            assert r0 == sum(len(r) for r in rows)
            rows.append(out)
            y0 += b
    finally:
        ag.free()
    assert y0 == h
    return np.concatenate(rows) if rows else np.zeros((0, A.dim(w, f)), np.uint8)


def _split(h, step):
    return [min(step, h - y) for y in range(0, h, step)]


@pytest.mark.parametrize("f", [2, 7, 25, 256, 1024])
@pytest.mark.parametrize("w,h", [(1000, 777), (53, 1301), (2049, 300)])
def test_rule_ragged_sizes(f, w, h):
    p = _plane(w, h, f + w)
    want = A.mean(p, f)
    assert want.shape == (A.dim(h, f), A.dim(w, f))
    assert np.array_equal(_host(p, f, [h]), want)
    assert np.array_equal(_host(p, f, _split(h, 256)), want)


@pytest.mark.parametrize("bands", [[1] * 60, [13, 1, 25, 21], [24, 26, 10], [59, 1]])
def test_bands_that_split_cell_rows(bands):
    p = _plane(300, 60, 3)
    assert np.array_equal(_host(p, 25, bands), A.mean(p, 25))


def test_factor_larger_than_block():
    p = _plane(40, 30, 4)
    got = _host(p, 1024, [30])
    assert got.shape == (1, 1)
    v = p[p != 255].astype(np.int64)
    assert int(got[0, 0]) == (2 * int(v.sum()) + len(v)) // (2 * len(v))


def test_all_nodata_cells_half_means_and_254():
    p = np.full((50, 75), 255, np.uint8)
    p[25:, 25:50] = 254                                 # one cell of 254 everywhere
    p[0, 50], p[0, 51] = 10, 11                         # 10.5 -> 11 (half up), 255 left out
    p[30, 60] = 3                                       # a single valid pixel: the mean is that pixel
    got = _host(p, 25, [50])
    assert got.tolist() == [[255, 255, 11], [255, 254, 3]]
    assert np.array_equal(got, A.mean(p, 25))
    q = np.full((2100, 1100), 254, np.uint8)            # 254 everywhere stays 254, also in a full 1024 x 1024 cell
    for f in (7, 1024):
        assert np.array_equal(_host(q, f, _split(2100, 256)), np.full((A.dim(2100, f), A.dim(1100, f)), 254, np.uint8))


def test_value_rule_edges():
    assert A.value(0, 0) == 255
    assert A.value(1, 2) == 1                           # 0.5 rounds up
    assert A.value(3, 2) == 2                           # 1.5 rounds up
    assert A.value(254 * 1024 * 1024, 1024 * 1024) == 254
    assert A.value(5, 4) == 1                           # 1.25 rounds down


def test_bands_out_of_order_are_refused():
    p = _plane(100, 100, 5)
    ag = hostlib.Aggregate(100, 100, 25)
    try:
        ag.rows(p[:30], 0)
        with pytest.raises(hostlib.HostError):
            ag.rows(p[40:], 40)
    finally:
        ag.free()


def _ifds(path):
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append((np.array(im), dict(im.tag_v2)))
    return out


@pytest.mark.parametrize("f,w,h,band", [(25, 1000, 777, 256), (2, 600, 520, 512), (7, 300, 2049, 2048),
                                        (1024, 100, 90, 256)])
def test_mean_file(tmp_path, f, w, h, band):
    p = _plane(w, h, 6 + f)
    full = hostlib.TiffWriter(str(tmp_path / "full.tif"), w, h, GT)
    tw = hostlib.TiffWriter(str(tmp_path / "mean.tif"), w, h, GT, aggregate=f)
    for y0 in range(0, h, band):
        assert full.write_rows(p[y0:y0 + band], y0) == 0
        assert tw.write_plane_rows(p[y0:y0 + band], y0) == 0
    assert full.close() == 0 and tw.close() == 0
    frames = _ifds(str(tmp_path / "mean.tif"))
    assert len(frames) == 1
    img, tags = frames[0]
    assert img.shape == (A.dim(h, f), A.dim(w, f))
    assert np.array_equal(img, A.mean(p, f))
    assert tags[42113] == "255" and 42112 not in tags
    (_, ftags), = _ifds(str(tmp_path / "full.tif"))
    assert 42113 not in ftags
    assert tags[34735] == ftags[34735]                  # the same GeoKeys
    assert tuple(tags[33922]) == tuple(ftags[33922])    # the same corner
    assert tuple(tags[33550])[:2] == pytest.approx((GT[1] * f, -GT[5] * f), rel=1e-15)
    assert tuple(A.gt(GT, f)) == (GT[0], GT[1] * f, 0.0, GT[3], 0.0, GT[5] * f)


def test_incomplete_mean_file_is_removed(tmp_path):
    p = _plane(300, 600, 7)
    tw = hostlib.TiffWriter(str(tmp_path / "mean.tif"), 300, 600, GT, aggregate=25)
    assert tw.write_plane_rows(p[:512], 0) == 0
    assert tw.close() != 0
    assert not (tmp_path / "mean.tif").exists()


def test_nodata_alone_with_overviews(tmp_path):
    p = _plane(700, 600, 8)
    tw = hostlib.TiffWriter(str(tmp_path / "n.tif"), 700, 600, GT, overviews=16, nodata=True)
    assert tw.write_rows(p, 0) == 0 and tw.close() == 0
    frames = _ifds(str(tmp_path / "n.tif"))
    assert len(frames) == 1 + tw.levels and tw.levels == 2
    assert np.array_equal(frames[0][0], p)
    assert all(t.get(42113) == "255" and 42112 not in t for _, t in frames)


def test_vrt_windows_overlap_by_one_pixel():
    """The edge wart of include/gcn10_cuda.h: with the shipped VRT's geotransform a 3-degree block's window is 36001
    pixels wide and tall, and its last column and row are the first of the next block's window.  So at f = 25 the
    one-pixel edge cell is a pixel that the neighbour's first cell covers in full."""
    px = 8.3333333333330430e-05
    t = (-180.0, px, 0.0, 84.0, 0.0, -px)
    rw, rh = 4320000, 1728000
    for lon in range(-180, 180, 3):
        for lat in range(84, -57, -3):
            xoff, yoff, xc, yc, _ = hostlib.raster_window(rw, rh, t, (lon, lat - 3, lon + 3, lat))
            assert (xoff, yoff) == ((lon + 180) // 3 * 36000, (84 - lat) // 3 * 36000), (lon, lat)
            assert xc == (36001 if xoff + 36001 <= rw else rw - xoff), (lon, lat)
            assert yc == (36001 if yoff + 36001 <= rh else rh - yoff), (lon, lat)
    assert A.dim(36001, 25) == 1441 and 36001 - 1440 * 25 == 1
