"""End to end on a GPU: the gcn10 executable (C host program + libgcn10cuda) against the reference's
own process_block() on the same rasters -- decoded planes must be identical, file names, log lines
and the no-overwrite underscore rule must match the reference's observable behaviour.  Where the reference's object
code (oracle/_ref) is not built, the expected rasters come from the plain-C restatement the golden fixtures pin to it."""
import os
import re
import subprocess

import numpy as np
import pytest

from gcn10_b200 import hostlib, synth
from tests import lookups
from oracle import oracle as O
from tests import fixtures

pytestmark = pytest.mark.gpu

PX = 1.0 / 12000.0
HSG_PX = 1.0 / 480.0


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    root = tmp_path_factory.mktemp("gcn10_run")
    W, H = 3000, 2200
    esa_t = (-114.0, PX, 0.0, 42.0, 0.0, -PX)
    esa = synth.esa_tile(W, H, 41, patch=96)
    hw, hh = 130, 100
    hsg_t = (-114.0 - 1.3 * HSG_PX, HSG_PX, 0.0, 42.0 + 2.6 * HSG_PX, 0.0, -HSG_PX)
    hsg = synth.hsg_tile(hw, hh, 42, "coastal", patch=3)
    hostlib.tiff_write(str(root / "esa.tif"), esa, esa_t)
    hostlib.tiff_write(str(root / "hsg.tif"), hsg, hsg_t)
    blocks = [
        (11, -114.0 + 100 * PX, 42.0 - 1500 * PX, -114.0 + 1400 * PX, 42.0 - 200 * PX),     # inside, 1300 x 1300
        (12, -114.0 + 1700 * PX, 42.0 - 2500 * PX, -114.0 + 3300 * PX, 42.0 - 900 * PX),    # hangs over the SE corner
        (13, -120.0, 10.0, -119.0, 11.0),                                                   # outside both rasters
    ]
    fixtures.write_block_shapefile(str(root / "blocks.shp"), blocks)
    lookups.write_default_lookups(str(root / "lookups"))
    fixtures.write_config(str(root / "config.txt"), str(root / "esa.tif"), str(root / "hsg.tif"),
                          str(root / "blocks.shp"), str(root / "lookups"), str(root / "logs"))
    (root / "blocks.txt").write_text("11\n12\n13\n99\n")
    return dict(root=root, esa=esa, esa_t=esa_t, hsg=hsg, hsg_t=hsg_t, blocks=blocks)


def _run(world, *extra, host_deflate=False, host_inflate=False):
    exe = hostlib.EXE_PATH
    assert os.path.exists(exe), "gcn10 executable not built (make host)"
    root = world["root"]
    env = dict(os.environ, GCN10_HOST_DEFLATE="1" if host_deflate else "0",
               GCN10_HOST_INFLATE="1" if host_inflate else "0")
    return subprocess.run([exe, "-c", str(root / "config.txt"), "-l", str(root / "blocks.txt"), "--gpus", "1",
                           "--io-threads", "4", *extra], cwd=str(root), capture_output=True, text=True, timeout=300,
                          env=env)


@pytest.mark.parametrize("host_deflate,host_inflate", [(False, False), (False, True), (True, True)],
                         ids=["gpu_inflate_gpu_deflate", "host_inflate_gpu_deflate", "host_inflate_host_deflate"])
def test_program_matches_reference_process_block(world, reference, host_deflate, host_inflate):
    from PIL import Image
    import shutil
    shutil.rmtree(world["root"] / "logs", ignore_errors=True)      # log files are opened for append (log.c:79)
    r = _run(world, "-o", host_deflate=host_deflate, host_inflate=host_inflate)
    assert r.returncode == 0, r.stderr
    log_all = (world["root"] / "logs" / "rank_0.log").read_text()
    assert ("land cover inflated on the gpu" in log_all) == (not host_deflate and not host_inflate)
    root = world["root"]
    for bid, x0, y0, x1, y1 in world["blocks"][:2]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                             str(root / "lookups"), block_id=bid)
        assert want["nplanes"] == 18
        for k, rel in enumerate(want["paths"]):                 # the reference's own file names, save order
            t = hostlib.Tiff(str(root / rel))
            assert (t.width, t.height) == (want["w"], want["h"]), rel
            assert t.gt == want["gt"], rel
            got = t.read()
            t.close()
            assert np.array_equal(got, want["planes"][k]), f"{rel}: {(got != want['planes'][k]).sum()} px differ"
            if k in (0, 17):                                    # independent decoder (libtiff) on the same file
                assert np.array_equal(np.array(Image.open(str(root / rel))), want["planes"][k]), rel
    # blocks 13 (no overlap) and 99 (not in the shapefile) are skipped with the reference's messages
    assert "esa load failed for block 13" in r.stderr and "invalid raster bounds" in r.stderr
    assert "block 99 not found" in r.stderr
    assert not (root / "cn_rasters_drained" / "cn_p_i_13.tif").exists()
    log = (root / "logs" / "rank_0.log").read_text()
    for c in O.CONDS:
        for h in O.HCS:
            for a in O.ARCS:
                assert f"completed condition for 11: {c}/{h}/{a}" in log                # cn.c:366-369
    assert len(re.findall(r"progress: completed block 12 / total 4", log)) == 18        # log.c:199-207, 18 per block
    assert "processing block 11" in log and "processed 4 blocks on 1 ranks" in log      # main.c:172,191


def test_damaged_land_cover_tile_skips_the_block(world, tmp_path):
    """A land-cover tile that is not a valid zlib stream: the GPU inflater reports it, the block is skipped with
    the reference's recoverable-error messages (raster.c:182-186 -> cn.c:188-192), the other block is written."""
    import shutil
    root = world["root"]
    data = bytearray((root / "esa.tif").read_bytes())
    t = hostlib.Tiff(str(root / "esa.tif"))
    tl = t.window_tiles(0, 0, 256, 256)             # first tile of the file = inside block 11 only
    t.close()
    first = bytes(tl["blob"][:int(tl["sizes"][0])].tobytes())
    at = bytes(data).find(first)
    assert at > 0
    data[at + 2:at + 40] = b"\xff" * 38
    shutil.copy(str(root / "esa.tif"), str(tmp_path / "esa_good.tif"))
    try:
        (root / "esa.tif").write_bytes(bytes(data))
        r = _run(world, "-o")
    finally:
        shutil.copy(str(tmp_path / "esa_good.tif"), str(root / "esa.tif"))
    assert r.returncode == 0, r.stderr
    assert "gdalrasterio error 3" in r.stderr and "esa load failed for block 11" in r.stderr
    assert "esa load failed for block 12" not in r.stderr
    _run(world, "-o")                               # leave intact outputs behind for the following tests


def test_no_overwrite_appends_underscore(world):
    root = world["root"]
    first = root / "cn_rasters_undrained" / "cn_g_iii_11.tif"
    if not first.exists():
        assert _run(world, "-o").returncode == 0
    before = first.read_bytes()
    r = _run(world)                                             # no -o: existing outputs are kept (cn.c:320-360)
    assert r.returncode == 0, r.stderr
    second = root / "cn_rasters_undrained" / "cn_g_iii_11_.tif"
    assert second.exists() and first.read_bytes() == before
    a = hostlib.Tiff(str(first)).read()
    b = hostlib.Tiff(str(second)).read()
    assert np.array_equal(a, b)


def test_block_rows_bands_equal_whole_block(gpu_ctx, port, tables):
    from tests.cases import make_block
    b = make_block(w=1300, h=1111, seed=77, shift=(0.0007, 0.0002), margin=1)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    for y0, n in [(0, 256), (256, 512), (768, 343), (1110, 1)]:
        got = gpu_ctx.block_rows(np.ascontiguousarray(b["esa"][y0:y0 + n]), 1111, y0, b["gt"], b["hsg"], b["soil_gt"])
        assert np.array_equal(got, want[:, y0:y0 + n]), (y0, n)


def test_program_reads_a_vrt_mosaic(world, reference, tmp_path):
    """esa_data_path = *.vrt, as in the reference's shipped config (landcover/esa_worldcover_2021.vrt, opened at
    raster.c:119): the land cover is a 2 x 2 mosaic of GeoTIFFs whose borders (x = 1290, y = 1210) cross both block
    windows, so every block is assembled from four sources -- on the GPU from their compressed tiles, and on the
    host with GCN10_HOST_INFLATE=1.  The rasters must equal the reference's process_block() on the assembled raster."""
    import shutil
    from tests.fixtures import write_vrt
    root = world["root"]
    vroot = tmp_path
    esa, esa_t = world["esa"], world["esa_t"]
    H, W = esa.shape
    cx, cy = 1290, 1210
    srcs = []
    for r, (y0, y1) in enumerate([(0, cy), (cy, H)]):
        for c, (x0, x1) in enumerate([(0, cx), (cx, W)]):
            name = f"lc_{r}{c}.tif"
            hostlib.tiff_write(str(vroot / name), esa[y0:y1, x0:x1],
                               (esa_t[0] + x0 * PX, PX, 0, esa_t[3] - y0 * PX, 0, -PX))
            srcs.append((name, 0, 0, x0, y0, x1 - x0, y1 - y0))
    write_vrt(str(vroot / "mosaic.vrt"), W, H, esa_t, srcs)
    fixtures.write_config(str(vroot / "config.txt"), str(vroot / "mosaic.vrt"), str(root / "hsg.tif"),
                          str(root / "blocks.shp"), str(root / "lookups"), str(vroot / "logs"))
    exe = hostlib.EXE_PATH
    for host_inflate in ("0", "1"):
        out = vroot / f"out{host_inflate}"
        out.mkdir()
        shutil.rmtree(vroot / "logs", ignore_errors=True)
        r = subprocess.run([exe, "-c", str(vroot / "config.txt"), "-l", str(root / "blocks.txt"), "--gpus", "1", "-o",
                            "--io-threads", "4", "--outdir", str(out)], cwd=str(vroot), capture_output=True, text=True,
                           timeout=300, env=dict(os.environ, GCN10_HOST_INFLATE=host_inflate, GCN10_HOST_DEFLATE="0"))
        assert r.returncode == 0, r.stderr
        log = (vroot / "logs" / "rank_0.log").read_text()
        assert ("mosaic parts inflated on the gpu" in log) == (host_inflate == "0")
        for bid, x0, y0, x1, y1 in world["blocks"][:2]:
            want = reference.run_block(esa, esa_t, world["hsg"], world["hsg_t"], (x0, y0, x1, y1), str(root / "lookups"),
                                 block_id=bid)
            for k, rel in enumerate(want["paths"]):
                t = hostlib.Tiff(str(out / rel))
                assert t.gt == want["gt"] and np.array_equal(t.read(), want["planes"][k]), (host_inflate, rel)
                t.close()
    # a source file that is missing: GDAL's read fails, the block is skipped, no output appears (cn.c:188-192)
    os.remove(vroot / "lc_11.tif")
    out = vroot / "out_missing"
    out.mkdir()
    r = subprocess.run([exe, "-c", str(vroot / "config.txt"), "-l", str(root / "blocks.txt"), "--gpus", "1", "-o",
                        "--outdir", str(out)], cwd=str(vroot), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0
    assert "gdal open failed" in r.stderr and "esa load failed for block 12" in r.stderr
    assert not list(out.glob("cn_rasters_*/cn_*_12*"))


def test_program_with_the_gdal_backend(world, reference, tmp_path):
    """The optional GDAL input backend (host_raster_gdal.c, make GDAL=1) inside the whole program: gcn10 is rebuilt
    here with -DGCN10_WITH_GDAL against the oracle's RAM stand-in for GDAL, the land cover is served by that GDAL under
    a /vsicurl/ name no file has (the soil raster stays a GeoTIFF on disk, read by the built-in reader), and the 18
    rasters per block must equal the reference's process_block().  The land cover then arrives as decoded pixels and
    goes through the raster-in entry point (gcn10_cuda_block_deflate_rows)."""
    host = os.path.join(os.path.dirname(hostlib.EXE_PATH))
    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "refshim")
    esa, esa_t = world["esa"], world["esa_t"]
    root = world["root"]
    esa.tofile(str(tmp_path / "esa.raw"))
    # the stand-in's registry lives in the process: a constructor fills it from a raw file before main() runs
    (tmp_path / "preload.c").write_text(
        '#include <stdio.h>\n#include <stdlib.h>\n#include <stdint.h>\n#include "refshim.h"\n'
        'void refshim_sink_deliver(refshim_sink *s, const char *p, const void *b, int w, int h)\n'
        '{ (void)s; (void)p; (void)b; (void)w; (void)h; }\n'
        'double refshim_now(void) { return 0.0; }\n'
        '__attribute__((constructor)) static void preload(void)\n{\n'
        '    const char *raw = getenv("REFSHIM_RAW"), *name = getenv("REFSHIM_NAME");\n'
        '    if (!raw || !name) return;\n'
        '    int w = atoi(getenv("REFSHIM_W")), h = atoi(getenv("REFSHIM_H"));\n'
        '    double t[6];\n'
        '    sscanf(getenv("REFSHIM_GT"), "%lf,%lf,%lf,%lf,%lf,%lf", &t[0], &t[1], &t[2], &t[3], &t[4], &t[5]);\n'
        '    uint8_t *d = malloc((size_t)w * h);\n'
        '    FILE *f = fopen(raw, "rb");\n'
        '    if (!d || !f || fread(d, 1, (size_t)w * h, f) != (size_t)w * h) abort();\n'
        '    fclose(f);\n'
        '    refshim_add_raster(name, d, w, h, t);\n}\n')
    exe = str(tmp_path / "gcn10_gdal")
    srcs = [os.path.join(host, f) for f in ("gcn10_main.c", "host_pipeline.c", "host_core.c", "host_tiff.c", "host_raster.c",
                                            "host_raster_gdal.c")]
    cmd = ["gcc", "-std=gnu11", "-O2", "-fPIC", "-ffp-contract=off", "-pthread", "-DGCN10_WITH_GDAL",
           "-I" + os.path.join(shim, "include"), "-I" + shim, "-o", exe, *srcs, os.path.join(shim, "fake_gdal.c"),
           str(tmp_path / "preload.c"), "-L" + os.path.dirname(host), "-lgcn10cuda",
           "-Wl,-rpath," + os.path.dirname(host), "-lz", "-lm", "-lstdc++"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    name = "/vsicurl/https://example.invalid/esa_worldcover.tif"
    fixtures.write_config(str(tmp_path / "config.txt"), name, str(root / "hsg.tif"), str(root / "blocks.shp"),
                          str(root / "lookups"), str(tmp_path / "logs"))
    out = tmp_path / "out"
    out.mkdir()
    env = dict(os.environ, REFSHIM_RAW=str(tmp_path / "esa.raw"), REFSHIM_NAME=name, REFSHIM_W=str(esa.shape[1]),
               REFSHIM_H=str(esa.shape[0]), REFSHIM_GT=",".join(repr(float(v)) for v in esa_t))
    env.pop("GCN10_RASTER_BACKEND", None)
    r = subprocess.run([exe, "-c", str(tmp_path / "config.txt"), "-l", str(root / "blocks.txt"), "--gpus", "1", "-o",
                        "--io-threads", "4", "--outdir", str(out)], cwd=str(tmp_path), capture_output=True, text=True,
                       timeout=300, env=env)
    assert r.returncode == 0, r.stderr
    log = (tmp_path / "logs" / "rank_0.log").read_text()
    assert f"{name} opened with gdal" in log and "hsg.tif opened with gdal" not in log
    assert "inflated on the gpu" not in log
    for bid, x0, y0, x1, y1 in world["blocks"][:2]:
        want = reference.run_block(esa, esa_t, world["hsg"], world["hsg_t"], (x0, y0, x1, y1), str(root / "lookups"),
                             block_id=bid)
        for k, rel in enumerate(want["paths"]):
            t = hostlib.Tiff(str(out / rel))
            assert t.gt == want["gt"] and np.array_equal(t.read(), want["planes"][k]), rel
            t.close()
    assert "esa load failed for block 13" in r.stderr and "block 99 not found" in r.stderr
