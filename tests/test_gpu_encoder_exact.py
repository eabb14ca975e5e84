"""Every tile stream the GPU encoders write equals the scalar reference's (tests/stream_ref.py), byte for byte.

Decoding a tile with zlib only shows that the stream is valid.  These tests also hold the kernels to the streams of
DESIGN.md section 4.5: the same parse, tie-break, code, stored fallbacks and encoder choice.  They sweep:

  * the code regimes build_fused_tables picks from the lookup tables: the ten shapes of the tuned code, the fixed code
    beyond 240 values, the 255-record edge, and the two-kernel path at 256 records or 4 literal classes; checked with
    launch_count() too;
  * the modes step 6 of cn_deflate_fused_kernel picks per tile (template or per-plane streams, rounds, checkpoint
    pieces or items, stored planes among compressed ones, MAXP 9 and 18), counted and required to occur;
  * overview levels, mean rasters and histograms of one call under tables the shipped ones do not reach;
  * one full 36000 x 36000 block.
"""
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from gcn10_b200 import capi
from tests import aggregate_rule, overview_rule
from tests import stream_ref as S
from tests.block_options import assemble
from tests.cases import make_block
from tests.encoder_cases import (SHAPES, noisy_tile, random_block, tables_with_classes, tables_with_records,
                                  tables_with_values)

pytestmark = pytest.mark.gpu

T = 256
ONE, NINE, ALL = 1 << 7, capi.MASK_DRAINED, capi.MASK_ALL


def _launches(ctx, fn):
    a = ctx.launch_count()
    res = fn()
    return res, ctx.launch_count() - a


REGIME_CASES = [(f"values_{n}", "values", n) for n in (2, 4, 8, 16, 32, 64, 128, 192, 224, 240)] + [
    ("values_241", "values", 241), ("records_255", "records", 255), ("records_256", "records", 256),
    ("classes_4", "classes", 4)]
EXPECT = {"values_241": "fixed", "records_255": None, "records_256": "two_kernel", "classes_4": "two_kernel"}
_regime_table = []


@pytest.fixture(scope="module", autouse=True)
def _print_regime_table():
    yield
    if _regime_table:
        print("\nregime / shape                 planes  call                  path (launches fused / fused=0)")
        for row in _regime_table:
            print("%-30s %6d  %-20s  %s" % row)


@pytest.mark.parametrize("call", ["block_deflate", "block_tiles_deflate"])
@pytest.mark.parametrize("mask", [ONE, NINE, ALL], ids=["1_plane", "9_planes", "18_planes"])
@pytest.mark.parametrize("name,kind,n", REGIME_CASES, ids=[c[0] for c in REGIME_CASES])
def test_code_regimes(name, kind, n, mask, call, gpu_ctx, port, tables):
    """One value count per tuned-code shape, the 241-value drop to the fixed code, the 255/256-record edge and four
    literal classes: the predicted path is the one the library takes (a fallback makes exactly the launches of the
    same call with fused=0, a fused regime fewer), and every tile is the reference's."""
    if kind == "classes" and mask == ONE:
        pytest.skip("one plane has one literal class")
    if kind == "values":
        t = tables_with_values(n, mask, seed=n)
    elif kind == "records":
        t = tables_with_records(n, mask)
    else:
        t = tables_with_classes(tables, n)
    tuned_code = 0 if kind == "classes" else 1
    reg = S.regime(t, mask, tuned_code=tuned_code)
    if kind == "values":
        assert reg.n_values == n and reg.n_records <= 255
        if n <= 240:
            assert reg.path == "tuned" and reg.shape == SHAPES[n], reg.shape
        else:
            assert reg.path == EXPECT[name]
    elif kind == "records":
        assert reg.n_records == n
        assert reg.path == (EXPECT[name] or ("fixed" if mask == ONE else "tuned"))
    else:
        assert reg.path == EXPECT[name]
    w, h = 700, 530
    b = random_block(w, h, seed=n + mask % 97)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    sel = [k for k in range(18) if mask >> k & 1]

    def run():
        if call == "block_deflate":
            return gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)
        src = capi.TileSource.from_raster(b["esa"], 256, 256, level=1)
        return gpu_ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)

    try:
        gpu_ctx.set_luts(t)
        gpu_ctx.set_option("tuned_code", tuned_code)
        res, n_fused = _launches(gpu_ctx, run)
        gpu_ctx.set_option("fused", 0)
        res0, n_plain = _launches(gpu_ctx, run)
    finally:
        gpu_ctx.set_option("fused", 1)
        gpu_ctx.set_option("tuned_code", 1)
        gpu_ctx.set_luts(tables)
    if reg.fused:
        assert n_fused < n_plain, (n_fused, n_plain)
    else:
        assert n_fused == n_plain, (n_fused, n_plain)
    _regime_table.append((f"{name} {reg.shape or reg.path}", len(sel), call, f"{reg.path} ({n_fused} / {n_plain})"))
    planes = {k: want[k] for k in sel}
    for k, tiles in res["tiles"].items():
        assert np.array_equal(assemble(tiles, w, h), planes[k]), k
    S.check_tiles(res["tiles"], planes, reg, name)
    S.check_tiles(res0["tiles"], planes, S.regime(t, mask, fused=0), name + " fused=0")


# ---- kernel modes --------------------------------------------------------------------------------------------------

def _one_tile_planes(port, esa, t):
    b = make_block(w=T, h=T, seed=1)
    b["esa"] = esa
    b["hsg"][:] = 2
    return b, port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)


def _stored(port, t, reg, n, seed, pool, plane=0):
    """Whether the j-th selected plane of the tile with n new pixels falls back to a stored stream."""
    _, want = _one_tile_planes(port, noisy_tile(n, seed, pool), t)
    tiles, _, _ = S.fused_tiles({k: want[k] for k in reg.planes}, reg)
    return len(tiles[reg.planes[plane]][(0, 0)]) == S.STORED_BYTES


def _threshold_n(port, t, reg, seed, pool, plane=0):
    """Largest n whose stream stays compressed (at most 31 680 bytes); with n + 1 new pixels it is stored."""
    lo, hi = 0, T * T
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if _stored(port, t, reg, mid, seed, pool, plane):
            hi = mid
        else:
            lo = mid
    return lo


MODE_CONFIGS = [
    # (name, tables kind, mask, tuned_code, densities)
    ("tuned_9", "shipped", NINE, 1, [0, 300, 2000, 5000, 9000, 16000, 30000, 65536]),
    ("tuned_18", "shipped", ALL, 1, [0, 2000, 9000, 30000, 65536]),
    ("fixed_1cls", "classes1", NINE, 0, [0, 2000, 9000, 65536]),
    ("fixed_2cls", "classes2", NINE, 0, [0, 2000, 9000]),
    ("fixed_3cls", "classes3", NINE, 0, [0, 2000, 9000]),
    ("mixed_stored", "mixed", NINE, 0, []),
]


def _mode_tables(kind, tables):
    if kind == "shipped":
        return tables
    if kind.startswith("classes"):
        return tables_with_classes(tables, int(kind[-1]))
    # variants 0, 2 and 5 hold 9-bit literals (>= 144) for every land cover, the others 8-bit ones
    rng = np.random.default_rng(5)
    t = rng.integers(1, 144, size=(9, 256, 5)).astype(np.int32)
    for v in (0, 2, 5):
        t[v] = rng.integers(144, 255, size=(256, 5))
    t[:, 50:] = 255                                 # 251 records
    return t


def mode_blocks(port, tables):
    """The blocks of the mode sweep, one tile row each: (name, regime, tables, tuned_code, block, planes, reference
    tiles, reference modes)."""
    pool = np.array([10, 20, 30, 40, 50, 60, 80, 90, 100], np.uint8)
    for name, kind, mask, tuned_code, dens in MODE_CONFIGS:
        t = _mode_tables(kind, tables)
        reg = S.regime(t, mask, tuned_code=tuned_code)
        assert reg.fused, name
        tiles_lc = [noisy_tile(n, 100 + i, pool) for i, n in enumerate(dens)]
        if name == "tuned_9":
            # one tile on each side of the stored threshold
            n0 = _threshold_n(port, t, reg, 77, pool)
            tiles_lc += [noisy_tile(n0, 77, pool), noisy_tile(n0 + 1, 77, pool)]
        if name == "mixed_stored":
            # plane 0 (9-bit literals) just stored, the 8-bit planes compressed
            lcpool = np.arange(0, 50, dtype=np.uint8)
            n0 = _threshold_n(port, t, reg, 78, lcpool, plane=0)
            tiles_lc += [noisy_tile(n0 + 1, 78, lcpool)]
        esa = np.concatenate(tiles_lc, axis=1)
        b = make_block(w=esa.shape[1], h=T, seed=3)
        b["esa"] = esa
        b["hsg"][:] = 2
        want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
        planes = {k: want[k] for k in reg.planes}
        ref, modes, _ = S.fused_tiles(planes, reg)
        yield name, reg, t, tuned_code, b, planes, ref, modes


def mode_counts(blocks):
    count = {m: 0 for m in ("template", "per_plane", "one_round", "rounds_2+", "fine", "coarse", "items",
                            "all_stored", "some_stored", "stored_noncontiguous", "just_below_threshold",
                            "just_above_threshold", "classes_0", "classes_1", "classes_2", "classes_3", "maxp_9",
                            "maxp_18")}
    for name, reg, _, _, _, _, ref, modes in blocks:
        nsel = len(reg.planes)
        for i, m in enumerate(modes):
            md = dict(zip(S.MODE_FIELDS, m.tolist()))
            count["template" if md["template"] else "per_plane"] += 1
            count["one_round" if md["rounds"] == 1 else "rounds_2+"] += 1
            count[{1: "fine", 0: "coarse", -1: "items"}[md["fine"]]] += 1
            if md["stored"] == nsel:
                count["all_stored"] += 1
            elif md["stored"]:
                count["some_stored"] += 1
                bits = [k for k in range(nsel) if md["stored_mask"] >> k & 1]
                if bits != list(range(bits[0], bits[-1] + 1)):
                    count["stored_noncontiguous"] += 1
            if name in ("tuned_9", "mixed_stored") and i >= len(modes) - (2 if name == "tuned_9" else 1):
                count["just_above_threshold" if md["stored"] else "just_below_threshold"] += 1
            count[f"classes_{md['classes']}"] += 1
            count[f"maxp_{md['maxp']}"] += 1
    return count


def test_kernel_modes(gpu_ctx, port, tables):
    """Tiles with a controlled number of new pixels drive cn_deflate_fused_kernel through its per-tile modes; every
    tile equals the reference, and each mode is reached at least once."""
    blocks = list(mode_blocks(port, tables))
    for name, reg, t, tuned_code, b, planes, ref, modes in blocks:
        try:
            gpu_ctx.set_luts(t)
            gpu_ctx.set_option("tuned_code", tuned_code)
            res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=reg.mask)
        finally:
            gpu_ctx.set_option("tuned_code", 1)
            gpu_ctx.set_luts(tables)
        for k, tiles in res["tiles"].items():
            assert np.array_equal(assemble(tiles, b["esa"].shape[1], T), planes[k]), k
        S.check_tiles(res["tiles"], planes, reg, name)
    count = mode_counts(blocks)
    print("\nmode coverage:", count)
    missing = [m for m, v in count.items() if v == 0]
    assert not missing, f"modes never reached: {missing}"


# ---- everything a call emits ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("fused,ordered,ship", [(1, 0, 0), (1, 1, 1), (0, 0, 1), (0, 1, 0)])
@pytest.mark.parametrize("nvals", [230, 241])
def test_overviews_stats_and_means_are_exact(nvals, fused, ordered, ship, gpu_ctx, port, tables):
    """Under tables the shipped ones do not reach (225..240 values: the tuned code's longest shape; 241: the fixed
    code), with overviews, stats and 25 x 25 means on: level tiles are the reference's encoding of the sampled planes,
    mean tiles the two-kernel encoding of the mean rasters, histograms the oracle's."""
    mask = NINE
    t = tables_with_values(nvals, mask, seed=nvals)
    reg = S.regime(t, mask, fused=fused)
    assert reg.path == ("two_kernel" if not fused else "tuned" if nvals <= 240 else "fixed")
    w, h = 1100, 900
    b = random_block(w, h, seed=nvals + 3)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    sel = reg.planes
    opts = dict(fused=fused, ordered=ordered, ship=ship, overviews=16, stats=1, aggregate=25, strip_rows=512)
    try:
        gpu_ctx.set_luts(t)
        for k, v in opts.items():
            gpu_ctx.set_option(k, v)
        res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)
    finally:
        for k, v in dict(fused=1, ordered=0, ship=0, overviews=0, stats=0, aggregate=0, strip_rows=2048).items():
            gpu_ctx.set_option(k, v)
        gpu_ctx.set_luts(tables)
    planes = {k: want[k] for k in sel}
    S.check_tiles(res["tiles"], planes, reg, "level 0")
    nlev = overview_rule.levels(w, h)
    assert sorted(res["overviews"]) == list(range(1, nlev + 1))
    for lev in range(1, nlev + 1):
        S.check_tiles(res["overviews"][lev], {k: overview_rule.decimate(want[k], lev) for k in sel}, reg,
                      f"level {lev}")
    S.check_tiles(res["aggregate"], {k: aggregate_rule.mean(want[k], 25) for k in sel}, S.regime(t, mask, fused=0),
                  "mean rasters")
    for k in sel:
        assert np.array_equal(res["histograms"][k], np.bincount(want[k].ravel(), minlength=256)), k


# ---- one full block ------------------------------------------------------------------------------------------------

def test_full_block_nine_planes(gpu_ctx, port, tables):
    """A 36000 x 36000 block, nine planes, shipped tables: every one of the 178 929 tiles equals the reference's.  The
    oracle runs one tile row at a time, the reference encoder beside it, on every core."""
    from gcn10_b200 import synth
    w = h = 36000
    gt, sgt, hsx, hsy = synth.block_geometry(-114.0, 42.0, w, h)
    esa = synth.esa_tile(w, h, seed=2234, patch=192)
    hsg = synth.hsg_tile(hsx, hsy, seed=3234, patch=9)
    t0 = time.time()
    res = gpu_ctx.block_deflate(esa, gt, hsg, sgt, plane_mask=NINE)
    t_gpu = time.time() - t0
    reg = S.regime(tables, NINE)
    assert reg.path == "tuned"
    sel = reg.planes

    def one_row(r):
        y0, y1 = r * T, min(h, (r + 1) * T)
        band = port.block_rows(esa[y0:y1], gt, hsg, sgt, tables, y0=y0, y1=y1, h=h)
        ref, _, _ = S.fused_tiles({k: band[k] for k in sel}, reg)
        bad = [(k, (r, c)) for k in sel for (_, c), z in ref[k].items() if res["tiles"][k][(r, c)] != z]
        return bad

    t0 = time.time()
    with ThreadPoolExecutor(max(4, len(os.sched_getaffinity(0)))) as ex:
        bad = [x for row in ex.map(one_row, range((h + T - 1) // T)) for x in row]
    print(f"\nfull block: GPU call {t_gpu:.1f} s, reference + oracle {time.time() - t0:.1f} s, {len(bad)} tiles differ")
    assert not bad, bad[:10]
