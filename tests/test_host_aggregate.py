"""CPU tests of the mean-raster rule and of the NoData tag alone (gh_tiffw_set_nodata).  tests/aggregate_rule.py, the
numpy restatement of the rule in include/gcn10_cuda.h, is what the GPU tests compare every mean tile with, so its edge
cases are pinned here with literal values.  A file with the NoData tag alone must carry GDAL_NODATA "255" in every IFD
and no GDAL_METADATA; Pillow's libtiff reader is the independent reader of the files."""
import numpy as np
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


def test_rule_factor_larger_than_block():
    p = _plane(40, 30, 4)
    got = A.mean(p, 1024)
    assert got.shape == (1, 1)
    v = p[p != 255].astype(np.int64)
    assert int(got[0, 0]) == (2 * int(v.sum()) + len(v)) // (2 * len(v))


def test_rule_all_nodata_cells_half_means_and_254():
    p = np.full((50, 75), 255, np.uint8)
    p[25:, 25:50] = 254                                 # one cell of 254 everywhere
    p[0, 50], p[0, 51] = 10, 11                         # 10.5 -> 11 (half up), 255 left out
    p[30, 60] = 3                                       # a single valid pixel: the mean is that pixel
    got = A.mean(p, 25)
    assert got.tolist() == [[255, 255, 11], [255, 254, 3]]
    q = np.full((2100, 1100), 254, np.uint8)            # 254 everywhere stays 254, also in a full 1024 x 1024 cell
    for f in (7, 1024):
        assert np.array_equal(A.mean(q, f), np.full((A.dim(2100, f), A.dim(1100, f)), 254, np.uint8))


def test_value_rule_edges():
    assert A.value(0, 0) == 255
    assert A.value(1, 2) == 1                           # 0.5 rounds up
    assert A.value(3, 2) == 2                           # 1.5 rounds up
    assert A.value(254 * 1024 * 1024, 1024 * 1024) == 254
    assert A.value(5, 4) == 1                           # 1.25 rounds down


def _ifds(path):
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append((np.array(im), dict(im.tag_v2)))
    return out


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
