"""GPU tests of option "aggregate": the compressed-tile calls deliver the f x f mean raster of every selected plane
behind the block's full-resolution strips and overview levels.  Every mean tile is inflated with CPython's zlib and
must equal the rule of include/gcn10_cuda.h (tests/aggregate_rule.py) applied to the oracle's planes, byte for byte;
the full-resolution strips must be byte-identical to the same call without the option."""
import os

import numpy as np
import pytest

from gcn10_b200 import capi
from tests import aggregate_rule as A
from tests import fixtures
from tests import overview_rule as R
from tests.block_options import (CALLS, FULL_SIZE, T, assemble, config_for, ctx, full_size_block,  # noqa: F401
                                 full_size_parts, options, run_call, world)
from tests.cases import SMALL_CASES, make_block

pytestmark = pytest.mark.gpu

FACTORS = [25, 2, 7, 100, 256, 1024]


def _check_means(res, want, mask, f, w, h):
    planes = [p for p in range(18) if mask >> p & 1]
    assert sorted(res["aggregate"]) == planes
    for p in planes:
        got = assemble(res["aggregate"][p], A.dim(w, f), A.dim(h, f))
        assert np.array_equal(got, A.mean(want[p], f)), f"plane {p} f={f}"


@pytest.mark.parametrize("call", CALLS)
@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_means_equal_oracle(name, kw, call, ctx, port, tables):
    mask, fused, ordered, ship = config_for(name, call)
    f = config_for(name, call, FACTORS)
    b = make_block(**kw)
    h, w = b["esa"].shape
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    with options(ctx, fused=fused, ordered=ordered, ship=ship):
        base = run_call(ctx, call, b, mask)
    assert base["aggregate"] == {}
    with options(ctx, aggregate=f, fused=fused, ordered=ordered, ship=ship):
        res = run_call(ctx, call, b, mask)
    assert res["tiles"] == base["tiles"]            # the same bytes as without the option
    _check_means(res, want, mask, f, w, h)


def test_strip_fields_and_order(ctx):
    b = make_block(w=3001, h=2600, seed=21)
    h, w = b["esa"].shape
    seen = []
    with options(ctx, aggregate=2, overviews=16, strip_rows=512):
        ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], capi.MASK_DRAINED,
                          on_strip=lambda st: seen.append((st.aggregate, st.level, st.tile_row0, st.n_tile_rows,
                                                           st.tiles_x, st.level_w, st.level_h)))
    expect = []
    for k in range(R.levels(w, h) + 1):             # full resolution, then the overview levels
        lw, lh = R.dim(w, k), R.dim(h, k)
        for y0 in range(0, lh, 512):
            expect.append((0, k, y0 // T, (min(512, lh - y0) + T - 1) // T, (lw + T - 1) // T, lw, lh))
    cw, ch = A.dim(w, 2), A.dim(h, 2)               # then the mean raster, in strips of at most strip_rows rows
    for y0 in range(0, ch, 512):
        expect.append((2, 0, y0 // T, (min(512, ch - y0) + T - 1) // T, (cw + T - 1) // T, cw, ch))
    assert seen == expect


@pytest.mark.parametrize("f", [2, 7, 25, 300])
def test_factors_and_strip_sizes(f, ctx, port, tables):
    """Cell rows that straddle strips of 256 rows, and a factor larger than the block's height."""
    b = make_block(w=1777, h=1290, seed=31 + f)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    for fused in (1, 0):
        with options(ctx, aggregate=f, fused=fused, strip_rows=256):
            res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        _check_means(res, want, capi.MASK_ALL, f, 1777, 1290)
    b = make_block(w=300, h=200, seed=5)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    with options(ctx, aggregate=1024):
        res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])       # one cell holds the whole block
    _check_means(res, want, capi.MASK_ALL, 1024, 300, 200)


def test_option_values(ctx):
    for bad in (1, -1, 1025):
        with pytest.raises(capi.Gcn10Error):
            ctx.set_option("aggregate", bad)
    for good in (2, 1024, 0):
        ctx.set_option("aggregate", good)


def test_launch_counts(ctx, tables):
    b = make_block(w=1300, h=1100, seed=22)
    args = (b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    with capi.Context(0) as fresh:
        fresh.set_luts(tables)
        n0 = fresh.launch_count()
        fresh.block_deflate(*args)
        base = fresh.launch_count() - n0

    def count(agg, fused):
        with options(ctx, aggregate=agg, fused=fused, strip_rows=512):
            n0 = ctx.launch_count()
            ctx.block_deflate(*args)
            return ctx.launch_count() - n0

    with options(ctx, aggregate=25):
        ctx.set_option("aggregate", 0)                  # set, then back off: exactly the launches of a fresh context
        n0 = ctx.launch_count()
        ctx.block_deflate(*args)
        assert ctx.launch_count() - n0 == base
    # three accumulate kernels (1100 rows in 512-row strips), the finish kernel, one encoder for the 52 x 44 mean
    for fused in (1, 0):
        assert count(25, fused) == count(0, fused) + 3 + 1 + 1


def test_with_overviews_and_stats(ctx, port, tables):
    """The levels and the histograms are those of the call without the option; the mean strips are not counted."""
    b = make_block(w=2100, h=1900, seed=41)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    for fused in (1, 0):
        with options(ctx, overviews=16, stats=1, fused=fused):
            base = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        with options(ctx, aggregate=25, overviews=16, stats=1, fused=fused):
            res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        assert res["tiles"] == base["tiles"] and res["overviews"] == base["overviews"]
        assert np.array_equal(res["histograms"], base["histograms"])
        assert all(int(res["histograms"][p].sum()) == 2100 * 1900 for p in range(18))
        _check_means(res, want, capi.MASK_ALL, 25, 2100, 1900)


def test_bands_order_restart_and_mask(ctx, port, tables):
    b = make_block(w=700, h=1100, seed=23)
    esa, h = b["esa"], 1100
    want = port.block_rows(esa, b["gt"], b["hsg"], b["soil_gt"], tables)
    with options(ctx, aggregate=25):
        with pytest.raises(capi.Gcn10Error) as e:       # no block open
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        assert e.value.code == -1
        ctx.block_deflate_rows(esa[:256], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        with pytest.raises(capi.Gcn10Error):            # a gap
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        ctx.block_deflate_rows(esa[:256], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        with pytest.raises(capi.Gcn10Error) as e:       # another plane mask inside the block
            ctx.block_deflate_rows(esa[256:512], h, 256, b["gt"], b["hsg"], b["soil_gt"], capi.MASK_DRAINED)
        assert e.value.code == -1
        # a block that starts over at row 0 sums from zero: the rows of the abandoned bands are not in it
        ctx.block_deflate_rows(esa[:512], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        r1 = ctx.block_deflate_rows(esa[:512], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        assert r1["aggregate"] == {}
        r2 = ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        _check_means(r2, want, capi.MASK_ALL, 25, 700, h)
        # the whole block again in one call: the same means, not sums of two blocks
        r3 = ctx.block_deflate(esa, b["gt"], b["hsg"], b["soil_gt"])
        assert r3["aggregate"] == r2["aggregate"]
    ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])     # free again without the option


def test_prefetch_and_ship_paths(ctx, port, tables):
    blocks = [make_block(w=2100, h=1900, seed=24 + i) for i in range(3)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    for ordered, ship in ((0, 0), (1, 1)):
        with options(ctx, aggregate=25, ordered=ordered, ship=ship):
            ctx.tiles_prefetch(srcs[0], 2100, 1900)
            results = []
            for i, b in enumerate(blocks):
                if i + 1 < len(blocks):
                    ctx.tiles_prefetch(srcs[i + 1], 2100, 1900)
                results.append(ctx.block_tiles_deflate(srcs[i], 2100, 1900, b["gt"], b["hsg"], b["soil_gt"]))
        for b, res in zip(blocks, results):
            want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
            for p in (0, 17):
                assert np.array_equal(assemble(res["tiles"][p], 2100, 1900), want[p])
            _check_means(res, want, capi.MASK_ALL, 25, 2100, 1900)


def test_sink_failure_and_damaged_tile(ctx, port, tables):
    b = make_block(w=1500, h=1300, seed=30)
    h, w = b["esa"].shape
    with options(ctx, aggregate=7, strip_rows=256):
        seen = []

        def fail_in_mean(st):
            seen.append(st.aggregate)
            return 7 if st.aggregate else 0

        with pytest.raises(capi.Gcn10Error):
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=fail_in_mean)
        assert seen[-1] == 7 and seen.count(7) == 1
        src = capi.TileSource.from_raster(b["esa"], 256, 256)
        blob = src.blob.copy()
        o = int(src.offsets[5])
        blob[o + 2:o + 40] ^= 0x5A
        bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
        seen.clear()
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_tiles_deflate(bad, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=lambda st: seen.append(1))
        assert e.value.code == -6 and seen == []
        # the context is usable afterwards: the aborted blocks left nothing in the accumulators
        res = ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"])
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    _check_means(res, want, capi.MASK_ALL, 7, w, h)


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
        for mask in (capi.MASK_ALL, capi.MASK_UNDRAINED, 0x3 | 1 << 10):
            with options(ctx, aggregate=25, fused=fused, strip_rows=256):
                res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], mask)
            _check_means(res, want, mask, 25, 1040, 700)
    finally:
        ctx.set_luts(tables)


def _oracle_means(port, tables, esa, gt, hsg, sgt, n, f):
    """The rule applied to the oracle's planes of an n x n block, made in 256-row bands (with torch on the GPU: numpy
    would take minutes for 23 G pixels)."""
    import torch
    cw = A.dim(n, f)
    s = torch.zeros((18, cw, cw), dtype=torch.int64, device="cuda")
    cnt = torch.zeros_like(s)
    for y in range(0, n, 256):
        y1 = min(n, y + 256)
        pl = torch.from_numpy(port.block_rows(esa[y:y1], gt, hsg, sgt, tables, y0=y, y1=y1, h=n)).cuda().to(torch.int64)
        valid = (pl != 255).to(torch.int64)
        pad = cw * f - n
        v = torch.nn.functional.pad(pl * valid, (0, pad)).reshape(18, y1 - y, cw, f).sum(-1)
        c = torch.nn.functional.pad(valid, (0, pad)).reshape(18, y1 - y, cw, f).sum(-1)
        idx = torch.arange(y, y1, device="cuda") // f
        s.index_add_(1, idx, v)
        cnt.index_add_(1, idx, c)
    return A.value(s.cpu().numpy().astype(np.uint64), cnt.cpu().numpy().astype(np.uint64))


@pytest.mark.parametrize("shape", FULL_SIZE)
def test_full_size_block(shape, ctx, port, tables):
    n, gt, sgt, esa, hsg = full_size_block(shape)
    esa[::41, ::13] = 0                                 # land cover without a Curve Number: nodata pixels in every cell
    parts = full_size_parts(shape, esa)
    with options(ctx, aggregate=25):
        if len(parts) == 1:
            res = ctx.block_tiles_deflate(parts[0][0], n, n, gt, hsg, sgt)
        else:
            res = ctx.block_parts_deflate(parts, 0, n, n, gt, hsg, sgt)
    cw = A.dim(n, 25)
    assert cw == (1440 if n == 36000 else 1441)
    want = _oracle_means(port, tables, esa, gt, hsg, sgt, n, 25)
    for p in range(18):
        assert np.array_equal(assemble(res["aggregate"][p], cw, cw), want[p]), p


# ---- the program, file to file ---------------------------------------------------------------------------------

def _read(path):
    from PIL import Image
    with Image.open(path) as im:
        return (np.array(im), im.n_frames, im.tag_v2.get(33922), im.tag_v2.get(33550), im.tag_v2.get(34735),
                im.tag_v2.get(42113), im.tag_v2.get(42112))


@pytest.mark.parametrize("config", ["config.txt", "config_vrt.txt"], ids=["geotiff", "vrt_mosaic"])
def test_program_aggregate(world, reference, config, tmp_path):
    root = world["root"]
    modes = dict(gpu=False, host_inflate=True)
    for mode, hi in modes.items():
        r = fixtures.run_program(root, config, "-o", "--outdir", str(tmp_path / mode), "--aggregate", "25",
                                 host_inflate=hi)
        assert r.returncode == 0, r.stderr
    for bid, x0, y0, x1, y1 in world["blocks"]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                                   str(root / "lookups"), block_id=bid)
        for k, rel in enumerate(want["paths"]):
            # the full-resolution files are where they always were, and the mean files beside them
            full = _read(str(tmp_path / "gpu" / rel))
            assert np.array_equal(full[0], want["planes"][k]), rel
            d, name = os.path.split(rel)
            agg_rel = os.path.join(d + "_agg25", name)
            got = {m: _read(str(tmp_path / m / agg_rel)) for m in modes}
            img, nframes, tie, scale, keys, nodata, meta = got["gpu"]
            assert np.array_equal(img, A.mean(want["planes"][k], 25)), agg_rel
            assert nframes == 1 and nodata == "255" and meta is None, agg_rel
            assert keys == full[4], agg_rel                 # the land cover's GeoKeys
            assert tuple(scale)[:2] == pytest.approx((full[3][0] * 25, full[3][1] * 25), rel=1e-15)
            assert tuple(tie) == tuple(full[2])
            for m in modes:                                 # both paths write the same file contents
                assert np.array_equal(got[m][0], img) and got[m][1:] == got["gpu"][1:], (agg_rel, m)
