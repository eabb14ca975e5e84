"""CPU tests of the overview levels of the GeoTIFF writer (gh_tiffw_set_overviews, gh_tiffw_write_rows,
gh_tiffw_put_level_tile_rows, gh_tiffw_close) and of the three overview rules of include/gcn10_cuda.h.  Pillow's
libtiff reader is the independent reader of the files."""
import os
import subprocess

import numpy as np
import pytest
from PIL import Image

from gcn10_b200 import hostlib
from tests import overview_rule as R
from tests.tiff_cases import GT, SIZES, raster, tile_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
def _frames(path):
    out = []
    with Image.open(path) as im:
        for k in range(im.n_frames):
            im.seek(k)
            out.append((np.array(im), im.tag_v2.get(254)))
    return out


def _check_file(path, a, nlev):
    frames = _frames(path)
    assert len(frames) == nlev + 1
    assert np.array_equal(frames[0][0], a)
    assert frames[0][1] in (None, 0)
    for k in range(1, nlev + 1):
        img, subfile = frames[k]
        assert subfile == 1, k
        assert img.shape == (R.dim(a.shape[0], k), R.dim(a.shape[1], k)), k
        assert np.array_equal(img, R.decimate(a, k)), k


@pytest.mark.parametrize("w,h", SIZES)
def test_write_rows_levels(tmp_path, w, h):
    a = raster(w, h, seed=w * 7 + h)
    path = str(tmp_path / "o.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=16)
    assert tw.levels == R.levels(w, h)
    # bands of 512 rows: level rows whose source lies in the next band stay in the writer's tile row
    for y0 in range(0, h, 512):
        assert tw.write_rows(a[y0:y0 + 512], y0) == 0
    assert tw.close() == 0
    _check_file(path, a, R.levels(w, h))
    t = hostlib.Tiff(path)                      # the project's own reader keeps reading IFD0
    assert (t.width, t.height) == (w, h)
    assert np.array_equal(t.read(), a)
    t.close()


@pytest.mark.parametrize("w,h", SIZES)
def test_put_level_tile_rows(tmp_path, w, h):
    a = raster(w, h, seed=w + 3 * h)
    nlev = R.levels(w, h)
    path = str(tmp_path / "p.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=16)
    for level in range(nlev + 1):
        for r, streams in enumerate(tile_rows(R.decimate(a, level) if level else a)):
            assert tw.put_tile_row(r, streams, level=level) == 0, (level, r)
    assert tw.close() == 0
    _check_file(path, a, nlev)


def test_level_cap_and_order(tmp_path):
    a = raster(3001, 517, seed=5)
    tw = hostlib.TiffWriter(str(tmp_path / "c.tif"), 3001, 517, GT, overviews=2)
    assert tw.levels == 2
    rows = tile_rows(R.decimate(a, 1))
    assert tw.put_tile_row(1, rows[1], level=1) != 0         # tile rows of a level come in order
    assert tw.put_tile_row(0, rows[0], level=3) != 0         # no such level
    tw.L.gh_tiffw_abort(tw.h)


def test_incomplete_level_fails_and_leaves_no_file(tmp_path):
    w, h = 3001, 517
    a = raster(w, h, seed=9)
    path = str(tmp_path / "i.tif")
    tw = hostlib.TiffWriter(path, w, h, GT, overviews=16)
    for r, streams in enumerate(tile_rows(a)):
        assert tw.put_tile_row(r, streams) == 0
    for level in range(1, R.levels(w, h)):                  # the last level is missing
        for r, streams in enumerate(tile_rows(R.decimate(a, level))):
            assert tw.put_tile_row(r, streams, level=level) == 0
    assert tw.close() != 0
    assert not os.path.exists(path) and not os.path.exists(path + ".part")


def test_without_overviews_one_ifd(tmp_path):
    a = raster(600, 300, seed=1)
    path = str(tmp_path / "n.tif")
    tw = hostlib.TiffWriter(path, 600, 300, GT)
    assert tw.levels == 0
    assert tw.write_rows(a, 0) == 0
    assert tw.close() == 0
    _check_file(path, a, 0)


def test_header_rules(tmp_path):
    """gcn10_overview_dim / _src / _levels compiled from the header itself."""
    src = tmp_path / "rules.c"
    src.write_text(
        '#include <stdio.h>\n#include "gcn10_cuda.h"\n'
        "int main(void) {\n"
        "  int n[] = {36000, 36001};\n"
        "  for (int a = 0; a < 2; a++) {\n"
        "    int L = gcn10_overview_levels(n[a], n[a], 16);\n"
        "    printf(\"%d\", L);\n"
        "    for (int k = 1; k <= L; k++) printf(\" %d\", gcn10_overview_dim(n[a], k));\n"
        "    printf(\"\\n\");\n"
        "  }\n"
        "  printf(\"%d %d %d %d\\n\", gcn10_overview_levels(256, 256, 16), gcn10_overview_levels(257, 1, 16),\n"
        "         gcn10_overview_levels(36000, 36000, 3), gcn10_overview_levels(1, 1, 16));\n"
        "  printf(\"%d %d %d %d %d\\n\", gcn10_overview_src(0, 1, 5), gcn10_overview_src(2, 1, 5),\n"
        "         gcn10_overview_src(0, 3, 3), gcn10_overview_src(140, 8, 36000), gcn10_overview_src(140, 8, 36001));\n"
        "  return 0;\n}\n")
    exe = tmp_path / "rules"
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           str(src)])
    lines = subprocess.check_output([str(exe)], text=True).splitlines()
    assert lines[0] == "8 18000 9000 4500 2250 1125 563 282 141"
    assert lines[1] == "8 18001 9001 4501 2251 1126 563 282 141"
    assert lines[2] == "0 1 3 0"
    # centre of the cell, clamped to the last pixel: 140 * 256 + 128 = 35968 < 35999
    assert lines[3] == "1 4 2 35968 35968"
    assert [R.dim(36001, k) for k in range(1, 9)] == [18001, 9001, 4501, 2251, 1126, 563, 282, 141]
    assert R.levels(36000, 36000) == R.levels(36001, 36001) == 8
    assert int(R.src(17999, 1, 36000)) == 35999 and int(R.src(18000, 1, 36001)) == 36000
