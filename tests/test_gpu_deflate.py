"""GPU tile DEFLATE (gcn10_cuda_block_deflate): every tile must be a valid zlib stream (decoded here with
CPython's zlib, an independent inflate) whose 256 x 256 bytes equal the oracle's plane, zero padded at
the right / bottom edge exactly like the CPU GeoTIFF writer pads; and every stream must equal, byte for byte, the
scalar reference of the encoder the library picks (tests/stream_ref.py)."""
import zlib

import numpy as np
import pytest

from gcn10_b200 import capi
from tests import stream_ref as S
from tests.cases import make_block

pytestmark = pytest.mark.gpu

T = 256
_PATH = [None]          # the encoder path of the running test (fixture encoder_path)


@pytest.fixture(autouse=True, params=["fused_tuned_code", "fused_fixed_code", "two_kernel"])
def encoder_path(request, gpu_ctx):
    """Every test runs through the compressed-tile paths: cn_deflate_fused_kernel (Curve Numbers and all
    planes' zlib streams from one parse of the record-id tile) with the tuned Huffman code of tile_code.h or
    with RFC 1951's fixed code, and cn_block_kernel + deflate_tiles_kernel."""
    gpu_ctx.set_option("fused", 0 if request.param == "two_kernel" else 1)
    gpu_ctx.set_option("tuned_code", 1 if request.param == "fused_tuned_code" else 0)
    _PATH[0] = request.param
    yield request.param
    gpu_ctx.set_option("fused", 1)
    gpu_ctx.set_option("tuned_code", 1)


def _reference(want, tables, mask=capi.MASK_ALL):
    """The reference's streams of the selected planes of ``want`` (the oracle's [18, h, w]) under the encoder path
    the test runs: {plane: {(tile_row, tile_x): bytes}}."""
    p = _PATH[0]
    reg = S.regime(tables, mask, fused=int(p != "two_kernel"), tuned_code=int(p == "fused_tuned_code"))
    return S.expected_tiles({k: want[k] for k in reg.planes}, reg)


def _assemble(tiles, w, h, exact=None):
    """The plane the tiles decode to; with ``exact`` (the reference's tiles of the plane) every stream must equal the
    reference's, byte for byte."""
    tx_n, ty_n = (w + T - 1) // T, (h + T - 1) // T
    full = np.zeros((ty_n * T, tx_n * T), dtype=np.uint8)
    assert sorted(tiles) == [(r, c) for r in range(ty_n) for c in range(tx_n)], "tile grid incomplete"
    for (r, c), z in tiles.items():
        if exact is not None:
            assert z == exact[(r, c)], f"{_PATH[0]}: tile {(r, c)}: {len(z)} bytes, reference {len(exact[(r, c)])}"
        raw = zlib.decompress(z)
        assert len(raw) == T * T
        full[r * T:(r + 1) * T, c * T:(c + 1) * T] = np.frombuffer(raw, dtype=np.uint8).reshape(T, T)
    return full


CASES = [
    ("one_tile", dict(w=256, h=256)),
    ("ragged", dict(w=1300, h=777, seed=4)),
    ("tiny", dict(w=5, h=3)),
    ("multi_strip", dict(w=700, h=2600, seed=6)),
    ("coastal", dict(w=1000, h=600, profile="coastal", seed=7)),
    ("random_incompressible", dict(w=600, h=520, profile="random", seed=8)),
    ("busy_multi_round", dict(w=600, h=520, seed=9, esa_patch=5, hsg_patch=1)),
    ("busy_ragged_vrt", dict(w=1031, h=300, seed=10, esa_patch=9, hsg_patch=2, px=8.3333333333330430e-05, lon0=-3.0,
                             lat0=3.0, shift=(0.0011, 0.0004), margin=2)),
    ("ratio3", dict(w=700, h=300, seed=11, hsg_px=3.0 / 12000.0)),
    ("hsg_too_small_clamp", dict(w=800, h=400, hsx=20, hsy=5)),
]


@pytest.mark.parametrize("name,kw", CASES, ids=[c[0] for c in CASES])
def test_deflate_tiles_decode_to_oracle_planes(name, kw, gpu_ctx, port, tables):
    b = make_block(**kw)
    h, w = b["esa"].shape
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    gpu_ctx.set_option("strip_rows", 1024)
    try:
        res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_option("strip_rows", 2048)
    assert sorted(res["tiles"]) == list(range(18))
    ref = _reference(want, tables)
    for k in range(18):
        full = _assemble(res["tiles"][k], w, h, ref[k])
        assert np.array_equal(full[:h, :w], want[k]), f"{name}: plane {k}"
        assert not full[h:, :].any() and not full[:, w:].any(), "edge padding must be zero"


def test_deflate_stored_fallback_and_masks(gpu_ctx, port, tables):
    """Noise through a noisy table cannot be compressed: tiles must fall back to stored blocks and still
    decode; a mask selects planes."""
    rng = np.random.default_rng(1)
    t = rng.integers(0, 255, size=tables.shape).astype(np.int32)
    b = make_block(w=520, h=300, profile="random", seed=9)
    b["esa"] = rng.integers(0, 256, size=b["esa"].shape, dtype=np.uint8)
    b["hsg"] = rng.integers(1, 5, size=b["hsg"].shape, dtype=np.uint8)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    mask = capi.MASK_DRAINED
    try:
        gpu_ctx.set_luts(t)
        res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)
    finally:
        gpu_ctx.set_luts(tables)
    assert sorted(res["tiles"]) == list(range(9))
    sizes = [len(z) for d in res["tiles"].values() for z in d.values()]
    assert max(sizes) == 2 + 10 + 65536 + 4, "expected at least one stored tile"
    ref = _reference(want, t, mask)
    for k in range(9):
        assert np.array_equal(_assemble(res["tiles"][k], 520, 300, ref[k])[:300, :520], want[k])


@pytest.mark.parametrize("holes", [1, 2, 5], ids=["2_literal_classes", "3_literal_classes", "too_many_classes"])
def test_tables_with_missing_rows_per_variant(holes, gpu_ctx, port, tables):
    """Variants whose lookup CSV lacks rows for some land-cover classes put nodata (255, a 9-bit literal)
    where the other planes hold a value: the fused kernel keeps one bit-position counter per such pattern
    (up to 3) and the library falls back to the two-kernel path beyond that.  Negative, >= 255 and column-0
    entries ride along."""
    t = tables.copy()
    for q in range(holes):
        t[1 + q, 10 * (q + 1), :] = 255                    # variant 1+q has no rows for class 10 (q+1)
    t[0, 30, 2] = -3                                       # (uint8_t)(-3) = 253, a 9-bit literal in plane 0 only ...
    t[0, 30, 2] = t[0, 30, 2] if holes < 2 else tables[0, 30, 2]
    t[7, 50, 0] = 77                                       # column 0: reached by soil code 0
    b = make_block(w=700, h=540, seed=31, esa_patch=30, hsg_patch=2)
    b["hsg"][::7, ::5] = 0
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    try:
        gpu_ctx.set_luts(t)
        res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_luts(tables)
    ref = _reference(want, t)
    for k in range(18):
        assert np.array_equal(_assemble(res["tiles"][k], 700, 540, ref[k])[:540, :700], want[k]), f"plane {k}"


@pytest.mark.parametrize("mask", [1 << 7, (1 << 0) | (1 << 4) | (1 << 9) | (1 << 17), 0x3FFFF & ~(1 << 8), 0x2AAAA])
def test_arbitrary_plane_masks(mask, gpu_ctx, port, tables):
    """Any subset of the 18 rasters, across both drainage conditions: only the selected planes come back, in
    ascending plane order, and each decodes to the oracle's plane."""
    b = make_block(w=777, h=515, seed=17, esa_patch=40, hsg_patch=2, profile="coastal")
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)
    sel = [k for k in range(18) if mask & (1 << k)]
    assert sorted(res["tiles"]) == sel
    ref = _reference(want, tables, mask)
    for k in sel:
        assert np.array_equal(_assemble(res["tiles"][k], 777, 515, ref[k])[:515, :777], want[k]), f"plane {k}"


def test_deflate_compresses_cn_rasters(gpu_ctx):
    b = make_block(w=2048, h=2048, seed=10, esa_patch=192, hsg_patch=9)
    res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=capi.MASK_DRAINED)
    ratio = 9 * 2048 * 2048 / res["bytes"]
    assert ratio > 4.0, f"compression ratio only {ratio:.2f}"


def test_tuned_code_is_smaller_than_fixed_and_close_to_zlib(gpu_ctx, encoder_path):
    """The tuned Huffman code (tile_code.h) against RFC 1951's fixed code on the same tiles, and both against
    zlib level 6 (what the reference's save_raster() would write)."""
    if encoder_path != "fused_tuned_code":
        pytest.skip("size comparison runs once")
    b = make_block(w=2048, h=2048, seed=10, esa_patch=192, hsg_patch=9)
    tuned = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=capi.MASK_DRAINED)
    gpu_ctx.set_option("tuned_code", 0)
    fixed = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=capi.MASK_DRAINED)
    gpu_ctx.set_option("tuned_code", 1)
    zl = sum(len(zlib.compress(zlib.decompress(z), 6)) for d in tuned["tiles"].values() for z in d.values())
    assert tuned["bytes"] < 0.85 * fixed["bytes"]
    assert tuned["bytes"] < 1.6 * zl, (tuned["bytes"], zl)
    print(f"tile streams: tuned {tuned['bytes']}, fixed {fixed['bytes']}, zlib-6 {zl}")


def test_deflate_rows_bands_equal_whole_block(gpu_ctx, port, tables):
    """Band form: tiles of rows [row0, row0+n) carry the block's tile-row numbers and decode to the same
    bytes as the whole-block call."""
    import ctypes as C
    b = make_block(w=900, h=1400, seed=21, shift=(0.0005, 0.0003), margin=1)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    lib = gpu_ctx.lib
    h, w = b["esa"].shape
    hsy, hsx = b["hsg"].shape
    got = {}

    def _sink(_u, sp):
        st = sp.contents
        blob = C.string_at(st.blob, st.blob_bytes)
        for k in range(st.n_planes):
            for tr in range(st.n_tile_rows):
                for tx in range(st.tiles_x):
                    i = (k * st.n_tile_rows + tr) * st.tiles_x + tx
                    got[(st.plane_ids[k], st.tile_row0 + tr, tx)] = blob[st.offsets[i]: st.offsets[i] + st.sizes[i]]
        return 0

    cb = capi.TILE_SINK(_sink)
    gt6 = (C.c_double * 6)(*b["gt"])
    sgt6 = (C.c_double * 6)(*b["soil_gt"])
    for row0, n in [(0, 512), (512, 768), (1280, 120)]:
        band = np.ascontiguousarray(b["esa"][row0:row0 + n])
        rc = lib.gcn10_cuda_block_deflate_rows(gpu_ctx.h, band.ctypes.data, w, h, row0, n, w, gt6, b["hsg"].ctypes.data,
                                               hsx, hsy, hsx, sgt6, capi.MASK_UNDRAINED, cb, None)
        assert rc == 0, lib.gcn10_cuda_last_error()
    # a band that does not start on a tile boundary is refused
    band = np.ascontiguousarray(b["esa"][100:356])
    assert lib.gcn10_cuda_block_deflate_rows(gpu_ctx.h, band.ctypes.data, w, h, 100, 256, w, gt6, b["hsg"].ctypes.data,
                                             hsx, hsy, hsx, sgt6, capi.MASK_UNDRAINED, cb, None) == -1
    ref = _reference(want, tables, capi.MASK_UNDRAINED)
    for k in range(9, 18):
        tiles = {(r, c): z for (p, r, c), z in got.items() if p == k}
        full = _assemble(tiles, w, h, ref[k])
        assert np.array_equal(full[:h, :w], want[k]), k


@pytest.mark.parametrize("break_row", [None, 129, 2, 255, 130, 3])
def test_long_row_runs(break_row, gpu_ctx, port, tables, encoder_path):
    """Uniform rasters: every tile row repeats the row above, so whole tiles are coded as runs of length-258
    matches across the rows (fused_row_run).  break_row starts a new run there: run lengths 255, 128 (the case whose
    remainder of 2 bytes has to be merged into the last two matches), 1, 254, 129, 2 ..."""
    w, h = 700, 600
    b = make_block(w=w, h=h, seed=3)
    b["esa"][:] = 20
    b["hsg"][:] = 2
    if break_row is not None:
        b["esa"][break_row:] = 40
        b["esa"][256 + break_row:] = 10            # the second tile row gets the same structure
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    ref = _reference(want, tables)
    for k in range(18):
        assert np.array_equal(_assemble(res["tiles"][k], w, h, ref[k])[:h, :w], want[k]), f"plane {k}"
    # a tile of 256 repeated rows: 254 tokens of 10 bits (tuned code), 19 bits (fixed code), or one 24-bit token per
    # row (two-kernel path), plus a few tokens where the raster changes
    per_tile = {"fused_tuned_code": 450, "fused_fixed_code": 750, "two_kernel": 900}[encoder_path]
    assert res["bytes"] < 18 * 9 * per_tile, "uniform tiles must collapse to a few hundred bytes each"


def test_strip_hand_over_paths_agree(gpu_ctx, port, tables, encoder_path):
    """The ship kernel (exact bytes + tables written straight into page-locked memory behind the encoder) and the
    two-phase path (size read-back, then a copy) deliver the same tiles; a host arena that is too small for a strip
    is grown and the strip fetched again.  A failing sink drains the strips in flight and leaves the context usable."""
    b = make_block(w=1100, h=2300, seed=61, esa_patch=7, hsg_patch=1)
    h, w = b["esa"].shape
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    got = {}
    gpu_ctx.set_option("strip_rows", 512)
    try:
        for ship in (1, 0):
            gpu_ctx.set_option("ship", ship)
            got[ship] = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
        calls = [0]

        def failing(_st):
            calls[0] += 1
            return 3 if calls[0] == 2 else 0

        gpu_ctx.set_option("ship", 1)
        with pytest.raises(capi.Gcn10Error):
            gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=failing)
        again = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_option("ship", 0)
        gpu_ctx.set_option("strip_rows", 2048)
    assert got[0]["bytes"] == got[1]["bytes"] == again["bytes"]
    ref = _reference(want, tables)
    for k in range(18):
        assert got[0]["tiles"][k] == got[1]["tiles"][k] == again["tiles"][k]
        full = _assemble(got[1]["tiles"][k], w, h, ref[k])
        assert np.array_equal(full[:h, :w], want[k])


def test_ordered_strips(gpu_ctx, port, tables, encoder_path):
    """Option "ordered": every strip arrives laid out in table order ([plane][tile row][tile column], 16-byte
    aligned, offsets ascending, no bytes unaccounted for) and decodes to the same rasters."""
    b = make_block(w=1100, h=1500, seed=63, esa_patch=20, hsg_patch=2)
    h, w = b["esa"].shape
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    plain = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    seen = []

    def on_strip(st):
        n = st.n_planes * st.n_tile_rows * st.tiles_x
        offs = np.ctypeslib.as_array(st.offsets, (n,)).astype(np.int64)
        sizes = np.ctypeslib.as_array(st.sizes, (n,)).astype(np.int64)
        assert offs[0] == 0 and (offs % 16 == 0).all()
        assert (offs[1:] == offs[:-1] + (sizes[:-1] + 15) // 16 * 16).all()
        assert offs[-1] + (sizes[-1] + 15) // 16 * 16 == st.blob_bytes
        seen.append(n)
        return 0

    gpu_ctx.set_option("strip_rows", 512)
    gpu_ctx.set_option("ordered", 1)
    try:
        gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], on_strip=on_strip)
        res = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_option("ordered", 0)
        gpu_ctx.set_option("strip_rows", 2048)
    assert len(seen) == 3 and res["bytes"] == plain["bytes"]
    ref = _reference(want, tables)
    for k in range(18):
        assert res["tiles"][k] == plain["tiles"][k]
        full = _assemble(res["tiles"][k], w, h, ref[k])
        assert np.array_equal(full[:h, :w], want[k])
