"""GPU tests of option "overviews": the compressed-tile calls deliver nearest-neighbour overview levels of every
selected plane behind the block's full-resolution strips.  Every level tile is inflated with CPython's zlib and must
equal the rule of include/gcn10_cuda.h (tests/overview_rule.py) applied to the oracle's planes; the full-resolution
strips must be byte-identical to the same call without the option."""
import numpy as np
import pytest

from gcn10_b200 import capi, hostlib
from tests import fixtures
from tests import overview_rule as R
from tests.block_options import (CALLS, FULL_SIZE, T, assemble, config_for, ctx, frames, full_size_block,  # noqa: F401
                                 full_size_parts, options, run_call, world)
from tests.cases import SMALL_CASES, make_block

pytestmark = pytest.mark.gpu


def _check_levels(res, want, mask, w, h):
    nlev = R.levels(w, h)
    assert sorted(res["overviews"]) == list(range(1, nlev + 1))
    for k in range(1, nlev + 1):
        lw, lh = R.dim(w, k), R.dim(h, k)
        planes = res["overviews"][k]
        assert sorted(planes) == [p for p in range(18) if mask >> p & 1]
        for p, tiles in planes.items():
            got = assemble(tiles, lw, lh)
            assert np.array_equal(got, R.decimate(want[p], k)), f"level {k} plane {p}"


@pytest.mark.parametrize("call", CALLS)
@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_levels_equal_decimated_oracle(name, kw, call, ctx, port, tables):
    mask, fused, ordered, ship = config_for(name, call)
    b = make_block(**kw)
    h, w = b["esa"].shape
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    with options(ctx, fused=fused, ordered=ordered, ship=ship):
        base = run_call(ctx, call, b, mask)
    assert base["overviews"] == {}
    with options(ctx, overviews=16, fused=fused, ordered=ordered, ship=ship):
        res = run_call(ctx, call, b, mask)
    assert res["tiles"] == base["tiles"]            # level 0: byte-identical to the call without overviews
    _check_levels(res, want, mask, w, h)


def test_strip_fields_and_order(ctx, port, tables):
    b = make_block(w=3001, h=2600, seed=21)
    h, w = b["esa"].shape
    seen = []

    def on_strip(st):
        seen.append((st.level, st.tile_row0, st.n_tile_rows, st.tiles_x, st.level_w, st.level_h))

    with options(ctx, overviews=16, strip_rows=512):
        ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], capi.MASK_DRAINED, on_strip=on_strip)
    nlev = R.levels(w, h)
    expect = []
    for k in range(nlev + 1):
        lw, lh = R.dim(w, k), R.dim(h, k)
        for y0 in range(0, lh, 512):
            rows = min(512, lh - y0)
            expect.append((k, y0 // T, (rows + T - 1) // T, (lw + T - 1) // T, lw, lh))
    assert seen == expect


def test_option_off_launches_nothing_new(ctx, tables):
    b = make_block(w=1300, h=1100, seed=22)
    counts = []
    with capi.Context(0) as fresh:
        fresh.set_luts(tables)
        n0 = fresh.launch_count()
        fresh.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        counts.append(fresh.launch_count() - n0)
    with options(ctx):
        for ov in (3, 0):                               # set, then back off: exactly the launches of a fresh context
            ctx.set_option("overviews", ov)
            n0 = ctx.launch_count()
            levels = []
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=lambda st: levels.append(st.level))
            counts.append(ctx.launch_count() - n0)
            assert (max(levels) > 0) == (ov > 0)
    assert counts[2] == counts[0]
    assert counts[1] > counts[0]


def test_bands_out_of_order_are_refused(ctx):
    b = make_block(w=700, h=1100, seed=23)
    esa, h = b["esa"], 1100
    with options(ctx, overviews=16):
        with pytest.raises(capi.Gcn10Error) as e:       # no block open
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        assert e.value.code == -1
        ctx.block_deflate_rows(esa[:256], h, 0, b["gt"], b["hsg"], b["soil_gt"])
        with pytest.raises(capi.Gcn10Error):            # a gap
            ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])
        r = ctx.block_deflate_rows(esa, h, 0, b["gt"], b["hsg"], b["soil_gt"])      # a new block starts at row 0
        assert sorted(r["overviews"]) == list(range(1, R.levels(700, h) + 1))
    # without the option the band calls are as free as before
    ctx.block_deflate_rows(esa[512:], h, 512, b["gt"], b["hsg"], b["soil_gt"])


def test_prefetch_next_block_while_levels_run(ctx, port, tables):
    blocks = [make_block(w=2100, h=1900, seed=24 + i) for i in range(3)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    with options(ctx, overviews=16):
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
        _check_levels(res, want, capi.MASK_ALL, 2100, 1900)


def test_sink_failure_in_a_level_aborts_and_damaged_tile_gives_no_strip(ctx, port, tables):
    b = make_block(w=1500, h=1300, seed=30)
    h, w = b["esa"].shape
    with options(ctx, overviews=16):
        seen = []

        def fail_in_level_2(st):
            seen.append(st.level)
            return 7 if st.level == 2 else 0

        with pytest.raises(capi.Gcn10Error):
            ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=fail_in_level_2)
        assert seen[-1] == 2 and 3 not in seen
        src = capi.TileSource.from_raster(b["esa"], 256, 256)
        blob = src.blob.copy()
        o = int(src.offsets[5])
        blob[o + 2:o + 40] ^= 0x5A
        bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
        seen.clear()
        with pytest.raises(capi.Gcn10Error) as e:
            ctx.block_tiles_deflate(bad, w, h, b["gt"], b["hsg"], b["soil_gt"], on_strip=lambda st: seen.append(st.level))
        assert e.value.code == -6 and seen == []
        # the context is usable afterwards, levels included
        res = ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"])
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    _check_levels(res, want, capi.MASK_ALL, w, h)


def _levels_of_decoded(res, planes, w, h):
    """Every level tile of the given planes equals the rule applied to the decoded level-0 tiles."""
    for p in planes:
        full = assemble(res["tiles"][p], w, h)
        for k in range(1, R.levels(w, h) + 1):
            got = assemble(res["overviews"][k][p], R.dim(w, k), R.dim(h, k))
            assert np.array_equal(got, R.decimate(full, k)), f"level {k} plane {p}"
        yield p, full


@pytest.mark.parametrize("shape", FULL_SIZE)
def test_full_size_block_all_levels(shape, ctx, port, tables):
    n, gt, sgt, esa, hsg = full_size_block(shape)
    with options(ctx, overviews=16):
        res = ctx.block_parts_deflate(full_size_parts(shape, esa), 0, n, n, gt, hsg, sgt)
    assert sorted(res["overviews"]) == list(range(1, 9))
    assert all(len(res["overviews"][k]) == 18 for k in res["overviews"])
    assert sum(len(res["overviews"][k][0]) for k in res["overviews"]) == 6781        # level tiles of one plane
    cols = R.src(np.arange(R.dim(n, 1)), 1, n)
    for p, _ in _levels_of_decoded(res, (0, 17), n, n):
        # level 1 against the oracle on the sampled pixels of every 997th level row
        lv1 = assemble(res["overviews"][1][p], R.dim(n, 1), R.dim(n, 1))
        for r in range(0, R.dim(n, 1), 997):
            y = int(R.src(r, 1, n))
            want = port.block_rows(esa[y:y + 1], gt, hsg, sgt, tables, y0=y, y1=y + 1, h=n)[p][0]
            assert np.array_equal(lv1[r], want[cols]), f"plane {p} level 1 row {r}"


# ---- the program, file to file ---------------------------------------------------------------------------------

@pytest.mark.parametrize("config", ["config.txt", "config_vrt.txt"], ids=["geotiff", "vrt_mosaic"])
def test_program_overviews(world, reference, config, tmp_path):
    root = world["root"]
    modes = dict(gpu=False, host_inflate=True)
    for mode, hi in modes.items():
        r = fixtures.run_program(root, config, "-o", "--overviews", "--outdir", str(tmp_path / mode), host_inflate=hi)
        assert r.returncode == 0, r.stderr
    for bid, x0, y0, x1, y1 in world["blocks"]:
        want = reference.run_block(world["esa"], world["esa_t"], world["hsg"], world["hsg_t"], (x0, y0, x1, y1),
                                   str(root / "lookups"), block_id=bid)
        for k, rel in enumerate(want["paths"]):
            got = {m: frames(str(tmp_path / m / rel)) for m in modes}
            f = got["gpu"]
            assert len(f) == R.levels(want["w"], want["h"]) + 1, rel
            assert np.array_equal(f[0], want["planes"][k]), rel
            for lv in range(1, len(f)):
                assert np.array_equal(f[lv], R.decimate(f[0], lv)), (rel, lv)
            for m in modes:
                assert len(got[m]) == len(f) and all(np.array_equal(a, c) for a, c in zip(got[m], f)), (rel, m)
            t = hostlib.Tiff(str(tmp_path / "gpu" / rel))       # the project's reader: IFD0
            assert np.array_equal(t.read(), want["planes"][k])
            t.close()
