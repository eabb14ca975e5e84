"""GPU tests of option "stats": the compressed-tile calls count the histogram of every selected plane while they encode
(gcn10_cuda_last_histograms).  Every histogram must equal np.bincount of the oracle's planes, and the tiles must be
byte-identical to the same call without the option.  The program's --stats outputs must carry the tags of
tests/stats_rule.py applied to their decoded planes."""
import numpy as np
import pytest

from gcn10_b200 import capi, hostlib, synth
from tests import fixtures
from tests import overview_rule as R
from tests import stats_rule as S
from tests.block_options import (CALLS, FULL_SIZE, config_for, ctx, full_size_block, full_size_parts,  # noqa: F401
                                 options, run_call, world)
from tests.cases import SMALL_CASES, make_block

pytestmark = pytest.mark.gpu


def _want(planes, mask):
    """[18, 256] bincount of the selected planes of an oracle block, zero rows elsewhere."""
    out = np.zeros((18, 256), np.uint64)
    for p in range(18):
        if mask >> p & 1:
            out[p] = np.bincount(planes[p].ravel(), minlength=256)
    return out


@pytest.mark.parametrize("call", CALLS)
@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_histograms_equal_oracle(name, kw, call, ctx, port, tables):
    mask, fused, ordered, ship = config_for(name, call)
    b = make_block(**kw)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    with options(ctx, fused=fused, ordered=ordered, ship=ship):
        base = run_call(ctx, call, b, mask)
    assert base["histograms"] is None
    with options(ctx, stats=1, fused=fused, ordered=ordered, ship=ship):
        res = run_call(ctx, call, b, mask)
        assert np.array_equal(ctx.last_histograms(), res["histograms"])
    assert res["tiles"] == base["tiles"]            # the same bytes as without the option
    assert np.array_equal(res["histograms"], _want(want, mask))


@pytest.mark.parametrize("fused", [1, 0], ids=["fused_on", "fused_off"])
def test_random_tables_two_kernel_path(fused, ctx, port, tables):
    """Random tables give more than 255 distinct value records: the two-kernel path runs with option fused on too."""
    rng = np.random.default_rng(1)
    t = rng.integers(0, 256, size=tables.shape).astype(np.int32)
    b = make_block(w=1040, h=700, profile="random", seed=9)
    b["esa"] = rng.integers(0, 256, size=b["esa"].shape, dtype=np.uint8)
    b["hsg"] = rng.integers(0, 15, size=b["hsg"].shape, dtype=np.uint8)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    try:
        ctx.set_luts(t)
        with options(ctx, fused=fused, strip_rows=256):
            for mask in (capi.MASK_ALL, capi.MASK_UNDRAINED):
                ctx.set_option("stats", 1)
                n0 = ctx.launch_count()
                res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], mask)
                n_on = ctx.launch_count() - n0
                ctx.set_option("stats", 0)
                n0 = ctx.launch_count()
                ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], mask)
                assert n_on - (ctx.launch_count() - n0) == 3        # one histogram kernel per strip (3 of 256 rows)
                assert np.array_equal(res["histograms"], _want(want, mask)), mask
    finally:
        ctx.set_luts(tables)


def test_with_overviews_level_zero_only(ctx, port, tables):
    b = make_block(w=2100, h=1900, seed=41)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    for fused in (1, 0):
        with options(ctx, stats=1, overviews=16, fused=fused):
            res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        assert sorted(res["overviews"]) == list(range(1, R.levels(2100, 1900) + 1))
        assert np.array_equal(res["histograms"], _want(want, capi.MASK_ALL)), fused
        assert all(int(res["histograms"][p].sum()) == 2100 * 1900 for p in range(18))


def test_bands_order_and_restart(ctx, port, tables):
    b = make_block(w=700, h=1100, seed=23)
    esa, h = b["esa"], 1100
    want = port.block_rows(esa, b["gt"], b["hsg"], b["soil_gt"], tables)
    with options(ctx, stats=1):
        with pytest.raises(capi.Gcn10Error) as e:       # no block open
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        assert e.value.code == -1
        with pytest.raises(capi.Gcn10Error):            # nothing completed since the option was set
            ctx.last_histograms()
        ctx.block_deflate_rows(esa[:256], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        with pytest.raises(capi.Gcn10Error):            # a gap
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        ctx.block_deflate_rows(esa[:256], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        with pytest.raises(capi.Gcn10Error):            # another plane mask inside the block
            ctx.block_deflate_rows(esa[256:512], h, 256, b["gt"], b["hsg"], b["soil_gt"], capi.MASK_DRAINED)
        # a block that starts over at row 0 counts from zero: the rows of the abandoned bands are not in it
        ctx.block_deflate_rows(esa[:512], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        r1 = ctx.block_deflate_rows(esa[:512], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        assert r1["histograms"] is None
        r2 = ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        assert np.array_equal(r2["histograms"], _want(want, capi.MASK_ALL))
        # the whole block again in one call: the same counts, not twice them
        r3 = ctx.block_deflate(esa, b["gt"], b["hsg"], b["soil_gt"])
        assert np.array_equal(r3["histograms"], r2["histograms"])
    ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])     # free again without the option


def test_launch_counts(ctx, tables):
    b = make_block(w=1300, h=1100, seed=22)
    args = (b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    with capi.Context(0) as fresh:
        fresh.set_luts(tables)
        n0 = fresh.launch_count()
        fresh.block_deflate(*args)
        base = fresh.launch_count() - n0

    def count(stats, fused):
        with options(ctx, stats=stats, fused=fused, strip_rows=512):
            n0 = ctx.launch_count()
            ctx.block_deflate(*args)
            return ctx.launch_count() - n0

    with options(ctx, stats=1):
        ctx.set_option("stats", 0)                      # set, then back off: exactly the launches of a fresh context
        n0 = ctx.launch_count()
        ctx.block_deflate(*args)
        assert ctx.launch_count() - n0 == base
    assert count(1, 1) == count(0, 1)                   # fused: no launch of its own
    assert count(1, 0) == count(0, 0) + 3               # two-kernel path: one per strip (1100 rows in 512-row strips)


def test_prefetch_and_ship_paths(ctx, port, tables):
    blocks = [make_block(w=2100, h=1900, seed=24 + i) for i in range(3)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    for ordered, ship in ((0, 0), (1, 1)):
        with options(ctx, stats=1, ordered=ordered, ship=ship):
            ctx.tiles_prefetch(srcs[0], 2100, 1900)
            results = []
            for i, b in enumerate(blocks):
                if i + 1 < len(blocks):
                    ctx.tiles_prefetch(srcs[i + 1], 2100, 1900)
                results.append(ctx.block_tiles_deflate(srcs[i], 2100, 1900, b["gt"], b["hsg"], b["soil_gt"]))
        for b, res in zip(blocks, results):
            want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
            assert np.array_equal(res["histograms"], _want(want, capi.MASK_ALL))


def _oracle_histograms(port, tables, esa, gt, hsg, sgt, n):
    """The oracle's planes of an n x n block in 256-row bands, counted (with torch on the GPU: numpy's bincount would
    take minutes for 23 G pixels)."""
    import torch
    hist = torch.zeros((18, 256), dtype=torch.int64, device="cuda")
    for y in range(0, n, 256):
        y1 = min(n, y + 256)
        planes = torch.from_numpy(port.block_rows(esa[y:y1], gt, hsg, sgt, tables, y0=y, y1=y1, h=n)).cuda()
        for p in range(18):
            hist[p] += torch.bincount(planes[p].flatten(), minlength=256)
    return hist.cpu().numpy().astype(np.uint64)


@pytest.mark.parametrize("shape", FULL_SIZE)
def test_full_size_block(shape, ctx, port, tables):
    n, gt, sgt, esa, hsg = full_size_block(shape)
    parts = full_size_parts(shape, esa)
    with options(ctx, stats=1):
        if len(parts) == 1:
            res = ctx.block_tiles_deflate(parts[0][0], n, n, gt, hsg, sgt, on_strip=lambda st: 0)
        else:
            res = ctx.block_parts_deflate(parts, 0, n, n, gt, hsg, sgt, on_strip=lambda st: 0)
    got = res["histograms"]
    assert all(int(got[p].sum()) == n * n for p in range(18))
    assert np.array_equal(got, _oracle_histograms(port, tables, esa, gt, hsg, sgt, n))


# ---- the program, file to file ---------------------------------------------------------------------------------

def _tags(path):
    from PIL import Image
    with Image.open(path) as im:
        return np.array(im), im.tag_v2.get(42113), im.tag_v2.get(42112)


@pytest.mark.parametrize("config", ["config.txt", "config_vrt.txt"], ids=["geotiff", "vrt_mosaic"])
def test_program_stats(world, reference, config, tmp_path):
    root = world["root"]
    modes = dict(gpu=False, host_inflate=True)
    for mode, hi in modes.items():
        r = fixtures.run_program(root, config, "-o", "--outdir", str(tmp_path / mode), "--stats", host_inflate=hi)
        assert r.returncode == 0, r.stderr
    r = fixtures.run_program(root, config, "-o", "--outdir", str(tmp_path / "plain"))
    assert r.returncode == 0, r.stderr
    for bid, x0, y0, x1, y1 in world["blocks"]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                                   str(root / "lookups"), block_id=bid)
        for k, rel in enumerate(want["paths"]):
            tags = {m: _tags(str(tmp_path / m / rel)) for m in modes}
            img, nodata, meta = tags["gpu"]
            assert np.array_equal(img, want["planes"][k]), rel
            assert nodata == "255", rel
            assert S.close(S.parse(meta), S.of_plane(img)), rel
            for m in modes:                             # both paths write the same tags
                assert tags[m][1:] == tags["gpu"][1:], (rel, m)
                assert np.array_equal(tags[m][0], img), (rel, m)
            img, nodata, meta = _tags(str(tmp_path / "plain" / rel))
            assert nodata is None and meta is None, rel
            assert np.array_equal(img, want["planes"][k]), rel


@pytest.fixture(scope="module")
def tall_world(tmp_path_factory):
    """A block of 4500 rows: three 2048-row bands on the host-decode path of the program."""
    from tests import lookups
    root = tmp_path_factory.mktemp("gcn10_stats_tall")
    px, hpx = 1.0 / 12000.0, 1.0 / 480.0
    esa_t = (-114.0, px, 0.0, 42.0, 0.0, -px)
    esa = synth.esa_tile(1200, 4800, 61, patch=96)
    esa[::37, ::11] = 255                               # some nodata land cover too
    hsg_t = (-114.0 - 1.3 * hpx, hpx, 0.0, 42.0 + 2.6 * hpx, 0.0, -hpx)
    hsg = synth.hsg_tile(60, 200, 62, "coastal", patch=3)
    hostlib.tiff_write(str(root / "esa.tif"), esa, esa_t)
    hostlib.tiff_write(str(root / "hsg.tif"), hsg, hsg_t)
    blocks = [(31, -114.0 + 100 * px, 42.0 - 4600 * px, -114.0 + 1000 * px, 42.0 - 100 * px)]
    fixtures.write_block_shapefile(str(root / "blocks.shp"), blocks)
    lookups.write_default_lookups(str(root / "lookups"))
    (root / "blocks.txt").write_text("31\n")
    fixtures.write_config(str(root / "config.txt"), str(root / "esa.tif"), str(root / "hsg.tif"), str(root / "blocks.shp"),
                          str(root / "lookups"), str(root / "logs"))
    return dict(root=root, esa=esa, esa_t=esa_t, hsg=hsg, hsg_t=hsg_t, blocks=blocks)


def test_program_stats_multi_band_block(tall_world, reference, tmp_path):
    """A block taller than two 2048-row bands: the host-decode path hands the GPU's histograms over after its last band;
    both paths write the tags of the decoded planes."""
    root = tall_world["root"]
    modes = dict(gpu=False, host_inflate=True)
    for mode, hi in modes.items():
        r = fixtures.run_program(root, "config.txt", "-o", "--outdir", str(tmp_path / mode), "--stats", host_inflate=hi)
        assert r.returncode == 0, r.stderr
    bid, x0, y0, x1, y1 = tall_world["blocks"][0]
    want = reference.run_block(tall_world["esa"], tall_world["esa_t"], tall_world["hsg"], tall_world["hsg_t"],
                               (x0, y0, x1, y1), str(root / "lookups"), block_id=bid)
    assert want["h"] > 2 * 2048
    for k, rel in enumerate(want["paths"]):
        for m in modes:
            img, nodata, meta = _tags(str(tmp_path / m / rel))
            assert np.array_equal(img, want["planes"][k]), (rel, m)
            assert nodata == "255", (rel, m)
            assert S.close(S.parse(meta), S.of_plane(img)), (rel, m)
