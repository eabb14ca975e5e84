"""GPU tests of option "cog": the whole-block compressed-tile calls deliver the overview levels first, smallest first,
then the full resolution, then the mean rasters, and with "ordered" every tile leaves the device framed for a Cloud
Optimized GeoTIFF.  The tile streams must be byte-identical to the same call without the option; the framing is
checked on every tile; the program's outputs must pass tests/cog_rule.py and equal the reference."""
import numpy as np
import pytest

from gcn10_b200 import capi
from tests import cog_rule, fixtures
from tests import overview_rule as R
from tests.block_options import (FULL_SIZE, assemble, config_for, ctx, frames, full_size_block,  # noqa: F401
                                 full_size_parts, options, run_call, strip_collector, world)
from tests.cases import SMALL_CASES, make_block

pytestmark = pytest.mark.gpu

CALLS = ["deflate", "tiles", "parts"]
# (mask, fused, ordered, ship), dealt out over the cases x calls below: every (fused, ordered) pair several times
CONFIGS = [(m, f, o, s) for m in (capi.MASK_ALL, capi.MASK_DRAINED, 1 << 13) for o in (1, 0) for f in (1, 0)
           for s in (0, 1)]
AGG = 25


def _check_order(strips, nlev, agg=True):
    """Levels nlev .. 1, then level 0, then the mean rasters; tile rows in order within each."""
    kinds = [("agg", 0) if a else ("lv", lv) for a, lv, *_ in strips]
    want_kinds = [("lv", k) for k in range(nlev, -1, -1)] + ([("agg", 0)] if agg else [])
    seen = [k for i, k in enumerate(kinds) if i == 0 or kinds[i - 1] != k]
    assert seen == want_kinds, seen
    for kind in want_kinds:
        rows = [(r0, n) for (a, lv, r0, n, _), k in zip(strips, kinds) if k == kind]
        at = 0
        for r0, n in rows:
            assert r0 == at, (kind, rows)
            at += n


@pytest.mark.parametrize("call", CALLS)
@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_cog_order_same_streams_framed(name, kw, call, ctx, port, tables):
    mask, fused, ordered, ship = config_for(name, call, CONFIGS, CALLS)
    b = make_block(**kw)
    h, w = b["esa"].shape
    nlev = R.levels(w, h)
    got = {}
    for cog in (0, 1):
        strips, tiles = [], {}
        with options(ctx, cog=cog, overviews=16, aggregate=AGG, fused=fused, ordered=ordered, ship=ship):
            run_call(ctx, call, b, mask, on_strip=strip_collector(strips, tiles))
        got[cog] = (strips, tiles)
    strips, tiles = got[1]
    assert tiles == got[0][1]                       # every stream byte-identical to the call without the option
    _check_order(strips, nlev)
    assert all(f == (ordered == 1) for *_, f in strips)
    assert not any(f for *_, f in got[0][0])
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    for p in [p for p in range(18) if mask >> p & 1][:2]:
        assert np.array_equal(assemble(tiles[0][p], w, h), want[p])
        for k in range(1, nlev + 1):
            lv = assemble(tiles[k][p], R.dim(w, k), R.dim(h, k))
            assert np.array_equal(lv, R.decimate(want[p], k)), (p, k)


def test_rows_refuses_cog(ctx):
    b = make_block(w=700, h=600, seed=40)
    with options(ctx, cog=1, overviews=16):
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_deflate_rows(b["esa"], 600, 0, b["gt"], b["hsg"], b["soil_gt"])
        assert e.value.code == -1


def test_option_off_launches_nothing_new(ctx, tables):
    b = make_block(w=1300, h=1100, seed=41)
    counts = []
    with capi.Context(0) as fresh:
        fresh.set_luts(tables)
        fresh.set_option("overviews", 16)
        fresh.set_option("ordered", 1)
        n0 = fresh.launch_count()
        fresh.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        counts.append(fresh.launch_count() - n0)
    with options(ctx, overviews=16, ordered=1):
        for cog in (1, 0):                              # set, then back off: exactly the launches of a fresh context
            ctx.set_option("cog", cog)
            n0 = ctx.launch_count()
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
            counts.append(ctx.launch_count() - n0)
    assert counts[2] == counts[0]
    # the levels in one decimation instead of one per full-resolution strip (a single strip here): same count
    assert counts[1] == counts[0]


def test_prefetch_next_block_and_host_raster_between(ctx, port, tables):
    """A prefetched block survives a host-raster call in between, whose whole upload takes the other slot."""
    blocks = [make_block(w=2100, h=1900, seed=42 + i) for i in range(3)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    other = make_block(w=1700, h=1500, seed=49)
    results, res_other = [], None
    with options(ctx, cog=1, overviews=16, ordered=1):
        ctx.tiles_prefetch(srcs[0], 2100, 1900)
        for i, b in enumerate(blocks):
            if i + 1 < len(blocks):
                ctx.tiles_prefetch(srcs[i + 1], 2100, 1900)
            results.append(ctx.block_tiles_deflate(srcs[i], 2100, 1900, b["gt"], b["hsg"], b["soil_gt"]))
            if i == 0:
                res_other = ctx.block_deflate(other["esa"], other["gt"], other["hsg"], other["soil_gt"])
    for b, res, (w, h) in list(zip(blocks, results, [(2100, 1900)] * 3)) + [(other, res_other, (1700, 1500))]:
        want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
        for p in (0, 17):
            assert np.array_equal(assemble(res["tiles"][p], w, h), want[p])
            for k in range(1, R.levels(w, h) + 1):
                assert np.array_equal(assemble(res["overviews"][k][p], R.dim(w, k), R.dim(h, k)), R.decimate(want[p], k))


def test_sink_failure_in_a_level_and_damaged_tile(ctx, port, tables):
    b = make_block(w=1500, h=1300, seed=50)
    h, w = b["esa"].shape
    with options(ctx, cog=1, overviews=16, aggregate=AGG, ordered=1):
        strips = []
        with pytest.raises(capi.Gcn10Error):
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"],
                              on_strip=strip_collector(strips, {}, fail_at=lambda st: st.level == 1))
        assert [lv for _, lv, *_ in strips] == list(range(R.levels(w, h), 0, -1))     # stopped at level 1
        src = capi.TileSource.from_raster(b["esa"], 256, 256)
        blob = src.blob.copy()
        o = int(src.offsets[5])
        blob[o + 2:o + 40] ^= 0x5A
        bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
        strips.clear()
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_tiles_deflate(bad, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=strip_collector(strips, {}))
        assert e.value.code == -6 and strips == []
        strips, tiles = [], {}
        ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=strip_collector(strips, tiles))
    _check_order(strips, R.levels(w, h))
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    assert np.array_equal(assemble(tiles[0][3], w, h), want[3])


@pytest.mark.parametrize("shape", FULL_SIZE)
def test_full_size_block(shape, ctx, port, tables):
    n, gt, sgt, esa, hsg = full_size_block(shape)
    strips, tiles = [], {}
    with options(ctx, cog=1, overviews=16, ordered=1):
        ctx.block_parts_deflate(full_size_parts(shape, esa), 0, n, n, gt, hsg, sgt,
                                on_strip=strip_collector(strips, tiles))
    _check_order(strips, 8, agg=False)
    assert all(f for *_, f in strips)
    for p in (0, 17):
        full = assemble(tiles[0][p], n, n)
        for k in range(1, 9):
            lv = assemble(tiles[k][p], R.dim(n, k), R.dim(n, k))
            assert np.array_equal(lv, R.decimate(full, k)), (p, k)
        for y in list(range(0, n, 997)) + [n - 1]:
            want = port.block_rows(esa[y:y + 1], gt, hsg, sgt, tables, y0=y, y1=y + 1, h=n)[p][0]
            assert np.array_equal(full[y], want), f"plane {p} row {y}"


# ---- the program, file to file ---------------------------------------------------------------------------------

@pytest.mark.parametrize("config,host_inflate", [("config.txt", False), ("config_vrt.txt", False), ("config.txt", True)],
                         ids=["geotiff", "vrt_mosaic", "host_inflate"])
def test_program_cog(world, reference, config, host_inflate, tmp_path):
    root = world["root"]
    r = fixtures.run_program(root, config, "-o", "--outdir", str(tmp_path), "--cog", "--stats", "--aggregate", str(AGG),
                             host_inflate=host_inflate)
    assert r.returncode == 0, r.stderr
    for bid, x0, y0, x1, y1 in world["blocks"]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                                   str(root / "lookups"), block_id=bid)
        for k, rel in enumerate(want["paths"]):
            path = str(tmp_path / rel)
            ifds = cog_rule.check(path)
            f = frames(path)
            assert len(f) == len(ifds) == R.levels(want["w"], want["h"]) + 1, rel
            assert np.array_equal(f[0], want["planes"][k]), rel
            for lv in range(1, len(f)):
                assert np.array_equal(f[lv], R.decimate(f[0], lv)), (rel, lv)
            cond, name = rel.split("/")[-2:]
            agg = str(tmp_path / f"{cond}_agg{AGG}" / name)
            assert len(cog_rule.check(agg)) == 1, agg               # the mean raster: a COG without levels
            assert len(frames(agg)) == 1
