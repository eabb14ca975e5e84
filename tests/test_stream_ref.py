"""CPU checks of the scalar reference of the GPU tile encoders (tests/stream_ref.py, tests/harness/tile_code_host.cpp).

The GPU tests hold every tile the kernels write to this reference byte for byte, so the reference itself must be
right: its streams decode with zlib to the oracle's tiles in every regime, every shape of the tuned code and on both
sides of both stored thresholds; its parse is the one the token statistics count; and the regime it predicts changes
exactly at the edges build_fused_tables has (240 / 241 values, 255 / 256 records, 3 / 4 literal classes)."""
from __future__ import annotations

import zlib

import numpy as np
import pytest

from gcn10_b200 import capi
from tests import stream_ref as S
from tests.cases import make_block
from tests.encoder_cases import (SHAPES, noisy_tile, random_block, tables_with_classes, tables_with_records,
                                  tables_with_values)

T = 256
NINE = capi.MASK_DRAINED


def _decodes(tiles, planes):
    for k, d in tiles.items():
        h, w = planes[k].shape
        for (r, c), z in d.items():
            raw = np.frombuffer(zlib.decompress(z), np.uint8).reshape(T, T)
            part = planes[k][r * T:(r + 1) * T, c * T:(c + 1) * T]
            assert np.array_equal(raw[:part.shape[0], :part.shape[1]], part), (k, r, c)
            assert not raw[part.shape[0]:].any() and not raw[:, part.shape[1]:].any(), "padding must be zero"


@pytest.mark.parametrize("mask", [1 << 7, NINE, capi.MASK_ALL], ids=["1_plane", "9_planes", "18_planes"])
@pytest.mark.parametrize("nvals", sorted(SHAPES) + [241])
def test_streams_decode_in_every_shape(nvals, mask, port):
    """Every tuned-code shape and the fixed code past 240 values: the fused reference's streams, and the two-kernel
    reference's, decode to the oracle's tiles."""
    t = tables_with_values(nvals, mask, seed=nvals)
    reg = S.regime(t, mask)
    assert reg.n_values == nvals
    assert reg.path == ("tuned" if nvals <= 240 else "fixed")
    if nvals <= 240:
        assert reg.shape == SHAPES[nvals]
    b = random_block(300, 270, seed=nvals)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    planes = {k: want[k] for k in reg.planes}
    _decodes(S.fused_tiles(planes, reg)[0], planes)
    _decodes(S.expected_tiles(planes, S.regime(t, mask, fused=0)), planes)


def _one_tile(port, tables, n, pool, seed=77):
    b = make_block(w=T, h=T, seed=1)
    b["esa"] = noisy_tile(n, seed, pool)
    b["hsg"][:] = 2
    return port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)


def _first_stored(size_of, limit):
    """Smallest n whose stream passes ``limit`` bytes (size_of is non-decreasing enough for a bisection)."""
    lo, hi = 0, T * T
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if size_of(mid) > limit:
            hi = mid
        else:
            lo = mid
    return hi


def test_fused_stored_threshold(port, tables):
    """cn_deflate_fused_kernel stores a plane whose stream would pass 31 * 1024 - 64 = 31 680 bytes: the tile one
    new pixel below the switch is compressed (within a few bytes of it), the tile at the switch is stored, and both
    decode."""
    reg = S.regime(tables, NINE)
    pool = np.array([10, 20, 30, 40, 50, 60, 80, 90, 100], np.uint8)
    sizes = {}

    def size_of(n):
        want = _one_tile(port, tables, n, pool)
        z = S.fused_tiles({k: want[k] for k in reg.planes}, reg)[0][0][(0, 0)]
        sizes[n] = (len(z), want)
        return 10 ** 6 if len(z) == S.STORED_BYTES else len(z)

    n = _first_stored(size_of, 31680)
    size_of(n - 1)
    below, want_b = sizes[n - 1]
    above, want_a = sizes[n]
    assert 31680 - 24 <= below <= 31680, below
    assert above == S.STORED_BYTES
    for want in (want_b, want_a):
        planes = {k: want[k] for k in reg.planes}
        _decodes(S.fused_tiles(planes, reg)[0], planes)


def test_two_kernel_stored_threshold(port, tables):
    """deflate_tiles_kernel stores a tile whose stream would pass 40 KB."""
    pool = np.array([10, 20, 30, 40, 50, 60, 80, 90, 100], np.uint8)
    sizes = {}

    def size_of(n):
        want = _one_tile(port, tables, n, pool)
        z = S.plain_tiles(want[0])[(0, 0)]
        sizes[n] = (len(z), want[0])
        return 10 ** 6 if len(z) == S.STORED_BYTES else len(z)

    n = _first_stored(size_of, 40 * 1024)
    size_of(n - 1)
    assert 40 * 1024 - 24 <= sizes[n - 1][0] <= 40 * 1024 and sizes[n][0] == S.STORED_BYTES
    for _, plane in (sizes[n - 1], sizes[n]):
        _decodes({0: S.plain_tiles(plane)}, {0: plane})


def test_tokens_of_the_encoder_are_the_token_statistics(port, tables):
    """The encoder's parse and gcn10_test_tile_tokens (the statistics behind the tuned code's model) are one parse: on
    record-id tiles (here: the bytes of a one-plane tile, whose records are its values) the token counts agree."""
    L = S.lib()
    reg = S.regime(tables, 1 << 7)
    for seed in range(4):
        b = random_block(T, T, seed=seed)
        want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
        _, _, ntok = S.fused_tiles({7: want[7]}, reg)
        hist = np.zeros(34, np.uint64)
        L.gcn10_test_tile_tokens(np.ascontiguousarray(want[7]).ctypes.data, hist.ctypes.data)
        assert int(hist[0]) + int(hist[2:31].sum()) == ntok[0], seed


def test_regime_edges(tables):
    """build_fused_tables' edges: 240 values keep the tuned code, 241 take the fixed code; 255 records stay fused,
    256 go to the two-kernel path; three literal classes stay fused, four do not."""
    assert S.regime(tables_with_values(240, NINE), NINE).path == "tuned"
    assert S.regime(tables_with_values(241, NINE), NINE).path == "fixed"
    assert S.regime(tables_with_values(240, NINE), NINE, tuned_code=0).path == "fixed"
    for mask in (1 << 7, NINE, capi.MASK_ALL):
        assert S.regime(tables_with_records(255, mask), mask).n_records == 255
        assert S.regime(tables_with_records(255, mask), mask).fused
        r = S.regime(tables_with_records(256, mask), mask)
        assert r.n_records == 256 and r.path == "two_kernel"
    r3 = S.regime(tables_with_classes(tables, 3), NINE, tuned_code=0)
    assert r3.path == "fixed" and sorted(set(r3.cls)) == [0, 1, 2]
    assert S.regime(tables_with_classes(tables, 4), NINE, tuned_code=0).path == "two_kernel"
    assert S.regime(tables_with_classes(tables, 4), NINE).path == "tuned", "the tuned code has no literal classes"
    assert S.regime(tables, NINE, fused=0).path == "two_kernel"


def test_all_zero_record_beside_the_padding(port):
    """A real record whose values are all zero is not the padding: the fused parse keeps the raster's zeros and the
    padding apart, though both are zero bytes in every plane, so a ragged tile of zeros costs more tokens than a full
    one.  The two-kernel parse sees plain bytes: its stream of the same tile is that of a tile of zeros."""
    t = np.zeros((9, 256, 5), np.int32)
    reg = S.regime(t, NINE)
    assert reg.n_records == 2 and reg.n_values == 2 and reg.path == "tuned"     # zeros, and soil class 9's nodata
    b = make_block(w=200, h=180, seed=5)
    b["hsg"][:] = 1
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    assert not want[0].any()
    planes = {k: want[k] for k in reg.planes}
    ragged = S.fused_tiles(planes, reg)[0][0][(0, 0)]
    full = S.fused_tiles({k: np.zeros((T, T), np.uint8) for k in reg.planes}, reg)[0][0][(0, 0)]
    assert zlib.decompress(ragged) == zlib.decompress(full) == bytes(T * T)
    # ragged: row 0 = literal, run, literal (padding), run; a row run; row 180 = literal, run; a row run
    assert len(ragged) > len(full)
    assert S.plain_tiles(want[0]) == S.plain_tiles(np.zeros((T, T), np.uint8))


def test_plane_stream_depends_on_the_mask(port, tables):
    """A plane's fused stream is parsed on the records of ALL selected planes: plane 7 alone merges pixels that differ
    only in other planes, inside MASK_ALL it does not.  Both decode to the same plane; the streams differ.  That is
    part of the format, not an error."""
    b = random_block(512, 300, seed=9)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    alone = S.fused_tiles({7: want[7]}, S.regime(tables, 1 << 7))[0][7]
    inside = S.fused_tiles({k: want[k] for k in range(18)}, S.regime(tables, capi.MASK_ALL))[0][7]
    assert sorted(alone) == sorted(inside)
    for key in alone:
        assert zlib.decompress(alone[key]) == zlib.decompress(inside[key])
    assert any(alone[key] != inside[key] for key in alone)


def test_tie_goes_to_the_pixel_above():
    """Where the pixel above and the run of the left pixel match equally far, the match is at distance 256.  Row 0 =
    4 then 255 x 5, row 1 = 256 x 5: from pixel 1 of row 1 both distances match 255 pixels.  Rows 2..255 are 7s."""
    tile = np.full((T, T), 7, np.uint8)
    tile[0] = 5
    tile[0, 0] = 4
    tile[1] = 5
    hist = np.zeros(34, np.uint64)
    S.lib().gcn10_test_tile_tokens(tile.ctypes.data, hist.ctypes.data)
    # literals: 4 and 5 (row 0), 5 (row 1, pixel 0), 7 (row 2); runs: rows 0 and 2; above: row 1's tie + the row run of
    # rows 3..255 (253 rows = 251 x 258 + 10)
    assert int(hist[0]) == 4
    assert int(hist[33]) == 2
    assert int(hist[32]) == 1 + 252
