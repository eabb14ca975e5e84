"""GPU tile inflate (gcn10_cuda_inflate_tiles / gcn10_cuda_block_tiles_deflate) against zlib and the oracle.

The reference's load_raster() lets GDAL/zlib decode the land-cover tiles on the CPU
(/root/reference/src/raster.c:177-179); the checker is therefore zlib itself: every tile handed to the GPU
was produced by zlib.compress from a known raster, and the inflated window must equal that raster
byte for byte.  The chained call (compressed tiles in -> Curve Numbers -> compressed tiles out) is checked
against the oracle planes after decoding the output tiles with zlib."""
import zlib

import numpy as np
import pytest

from gcn10_b200 import capi, synth
from tests.block_options import assemble
from tests.cases import make_block

pytestmark = pytest.mark.gpu


def _raster(w, h, seed, profile="worldcover", patch=48):
    return synth.esa_tile(w, h, seed, profile=profile, patch=patch)


GEOMS = [
    # name, grid w, grid h, tile w, tile h, window (x_off, y_off, w, h) or None, level
    ("tiles256", 1300, 777, 256, 256, None, 6),
    ("tiles1024", 2500, 2100, 1024, 1024, None, 6),
    ("tiles512_level9", 1500, 1100, 512, 512, None, 9),
    ("tiles_not_pow2", 1000, 500, 240, 112, None, 6),
    ("window_inside", 3000, 2200, 1024, 1024, (700, 300, 1500, 1300), 6),
    ("window_inside_small_tiles", 1200, 900, 256, 256, (255, 257, 600, 500), 1),
    ("stored_only", 700, 600, 256, 256, None, 0),
    ("one_pixel_window", 600, 600, 256, 256, (300, 299, 1, 1), 6),
]


@pytest.mark.parametrize("name,gw,gh,tw,th,win,level", GEOMS, ids=[g[0] for g in GEOMS])
@pytest.mark.parametrize("profile", ["worldcover", "random"])
def test_inflate_equals_zlib_source(name, gw, gh, tw, th, win, level, profile, gpu_ctx):
    grid = _raster(gw, gh, seed=len(name) * 7 + gw, profile=profile)
    x_off, y_off, w, h = win if win else (0, 0, gw, gh)
    src = capi.TileSource.from_raster(grid, tw, th, level=level, x_off=x_off, y_off=y_off, gap=3)
    # guard band: a destination wider than the window must keep its padding
    out = np.full((h + 2, w + 37), 0xEE, dtype=np.uint8)
    view = out[1:h + 1, :w]
    rc, _, status = gpu_ctx.inflate_tiles(src, w, h, out=view, want_status=True)
    assert rc == 0, gpu_ctx.lib.gcn10_cuda_last_error().decode()
    assert not status.any()
    assert np.array_equal(view, grid[y_off:y_off + h, x_off:x_off + w])
    assert (out[0] == 0xEE).all() and (out[-1] == 0xEE).all() and (out[:, w:] == 0xEE).all()
    assert gpu_ctx.last_inflate_ms() > 0


def test_every_stream_alignment_and_strategy(gpu_ctx):
    """Streams at all 16 byte alignments inside the blob; fixed-Huffman, RLE, Huffman-only and filtered
    strategies; tiny windows (wbits 9) and short blocks (memLevel 1)."""
    tw = th = 256
    variants = [(6, zlib.Z_DEFAULT_STRATEGY, 15, 8), (6, zlib.Z_FIXED, 15, 8), (6, zlib.Z_RLE, 15, 8),
                (6, zlib.Z_HUFFMAN_ONLY, 15, 8), (6, zlib.Z_FILTERED, 15, 8), (6, zlib.Z_DEFAULT_STRATEGY, 9, 1),
                (9, zlib.Z_DEFAULT_STRATEGY, 12, 9), (1, zlib.Z_DEFAULT_STRATEGY, 15, 1)]
    n = 32
    grid = _raster(tw * n, th, seed=5, patch=20)
    grid[:, tw * 8:tw * 12] = _raster(tw * 4, th, seed=6, profile="random")
    blob, offsets, sizes = bytearray(), [], []
    for i in range(n):
        level, strat, wbits, mem = variants[i % len(variants)]
        c = zlib.compressobj(level, zlib.DEFLATED, wbits, mem, strat)
        z = c.compress(np.ascontiguousarray(grid[:, i * tw:(i + 1) * tw]).tobytes()) + c.flush()
        while len(blob) % 16 != (i * 5 + 1) % 16:
            blob.append(0x5A)
        offsets.append(len(blob))
        sizes.append(len(z))
        blob += z
    src = capi.TileSource(tw, th, n, 1, 0, 0, np.frombuffer(bytes(blob), dtype=np.uint8).copy(), offsets, sizes)
    assert len({o % 16 for o in offsets}) == 16
    out = gpu_ctx.inflate_tiles(src, tw * n, th)
    assert np.array_equal(out, grid)


def test_long_codes_far_matches_and_block_mixes(gpu_ctx):
    """Skewed byte statistics (Huffman codes longer than the 10-bit lookup), matches at distance ~30000
    (the batch-closing rule of the decode lane), and stored/fixed/dynamic blocks mixed by flushes."""
    rng = np.random.default_rng(3)
    tw, th = 1024, 512
    skew = rng.choice(np.arange(256, dtype=np.uint8), size=tw * th, p=np.r_[[0.6], np.full(255, 0.4 / 255)])
    period = rng.integers(0, 256, 30011, dtype=np.uint8)
    far = np.resize(period, tw * th)
    mixed_raw, parts = [], []
    c = zlib.compressobj(6)
    left = tw * th
    k = 0
    while left:
        m = min(left, 20000 + 1000 * k)
        chunk = (rng.integers(0, 256, m, dtype=np.uint8) if k % 3 == 0
                 else np.resize(_raster(300, 40, k, patch=16).ravel(), m))
        mixed_raw.append(chunk)
        parts.append(c.compress(chunk.tobytes()))
        parts.append(c.flush(zlib.Z_FULL_FLUSH if k % 2 else zlib.Z_SYNC_FLUSH))
        left -= m
        k += 1
    parts.append(c.flush())
    tiles = [skew, far, np.concatenate(mixed_raw)]
    streams = [zlib.compress(skew.tobytes(), 6), zlib.compress(far.tobytes(), 9), b"".join(parts)]
    offsets, pos = [], 0
    for z in streams:
        offsets.append(pos)
        pos += len(z)
    src = capi.TileSource(tw, th, 3, 1, 0, 0, np.frombuffer(b"".join(streams), dtype=np.uint8).copy(), offsets,
                          [len(z) for z in streams])
    out = gpu_ctx.inflate_tiles(src, 3 * tw, th)
    for i, t in enumerate(tiles):
        assert np.array_equal(out[:, i * tw:(i + 1) * tw], t.reshape(th, tw)), f"tile {i}"


def test_sparse_tiles_read_as_zero(gpu_ctx):
    grid = _raster(1024, 768, seed=12)
    src = capi.TileSource.from_raster(grid, 256, 256, sparse={(0, 1), (2, 3)})
    out = np.full(grid.shape, 7, dtype=np.uint8)
    gpu_ctx.inflate_tiles(src, 1024, 768, out=out)
    want = grid.copy()
    want[0:256, 256:512] = 0
    want[512:768, 768:1024] = 0
    assert np.array_equal(out, want)


def test_damaged_tiles_are_reported_not_fatal(gpu_ctx):
    grid = _raster(1024, 512, seed=13)
    src = capi.TileSource.from_raster(grid, 256, 256)
    blob = src.blob.copy()
    blob[int(src.offsets[2])] = 0x79                             # tile 2: bad zlib method
    o5, s5 = int(src.offsets[5]), int(src.sizes[5])
    blob[o5 + 2:o5 + s5] = 0xFF                                   # tile 5: garbage body
    bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
    rc, out, status = gpu_ctx.inflate_tiles(bad, 1024, 512, want_status=True)
    assert rc == -6, "GCN10_EDATA expected"
    assert status[2] == 1 and status[5] != 0
    good = [i for i in range(8) if i not in (2, 5)]
    assert not status[good].any()
    for i in good:
        r, c = divmod(i, 4)
        assert np.array_equal(out[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256],
                              grid[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256])
    # truncated tile: the size table says fewer bytes than the stream needs
    sizes = src.sizes.copy()
    sizes[1] = sizes[1] // 2
    cut = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, src.blob, src.offsets, sizes)
    rc, _, status = gpu_ctx.inflate_tiles(cut, 1024, 512, want_status=True)
    assert rc == -6 and status[1] != 0
    # the context stays usable
    assert np.array_equal(gpu_ctx.inflate_tiles(src, 1024, 512), grid)


def test_adler32_mismatch_is_reported(gpu_ctx):
    """A tile whose payload was altered without breaking the DEFLATE structure decodes to wrong land cover; zlib
    (GDAL's codec, raster.c:177-186) rejects it by its Adler-32 trailer and so does the GPU inflater: status 10,
    GCN10_EDATA, the other tiles unaffected."""
    grid = _raster(768, 512, seed=17)
    src = capi.TileSource.from_raster(grid, 256, 256, level=0)            # stored blocks: payload bytes are literals
    blob = src.blob.copy()
    blob[int(src.offsets[1]) + 7 + 4000] ^= 0x20                         # tile 1: one land-cover byte changed
    blob[int(src.offsets[4]) + int(src.sizes[4]) - 1] ^= 0x01            # tile 4: trailer changed
    bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
    rc, out, status = gpu_ctx.inflate_tiles(bad, 768, 512, want_status=True)
    assert rc == -6
    assert list(status) == [0, 10, 0, 0, 10, 0]
    # Huffman-coded tiles: a flipped bit deep in a stream is either a structural error or a checksum error
    src6 = capi.TileSource.from_raster(grid, 256, 256, level=6)
    for k in range(12):
        blob = src6.blob.copy()
        t = k % 6
        blob[int(src6.offsets[t]) + int(src6.sizes[t]) // 2 + k] ^= 1 << (k % 8)
        rc, out, status = gpu_ctx.inflate_tiles(capi.TileSource(256, 256, 3, 2, 0, 0, blob, src6.offsets, src6.sizes),
                                                768, 512, want_status=True)
        if rc == 0:
            assert np.array_equal(out, grid)
        else:
            assert status[t] != 0 and not np.delete(status, t).any()
    assert np.array_equal(gpu_ctx.inflate_tiles(src6, 768, 512), grid)
    # the chained call refuses the block (the reference skips a block whose land cover cannot be read, cn.c:188-192)
    b = make_block(w=768, h=512, seed=17)
    with pytest.raises(capi.Gcn10Error) as ei:
        gpu_ctx.block_tiles_deflate(bad, 768, 512, b["gt"], b["hsg"], b["soil_gt"])
    assert ei.value.code == -6


def test_bad_arguments(gpu_ctx):
    grid = _raster(512, 512, seed=1)
    src = capi.TileSource.from_raster(grid, 256, 256)
    rc, _, _ = gpu_ctx.inflate_tiles(src, 513, 512, want_status=True)            # grid does not cover the window
    assert rc == -1
    sizes = src.sizes.copy()
    sizes[3] = 1 << 30
    rc, _, _ = gpu_ctx.inflate_tiles(capi.TileSource(256, 256, 2, 2, 0, 0, src.blob, src.offsets, sizes), 512, 512,
                                     want_status=True)
    assert rc == -1


@pytest.mark.parametrize("kw,tile,off", [
    (dict(w=1300, h=777, seed=4), 256, (0, 0)),
    (dict(w=2300, h=2600, seed=6), 1024, (100, 900)),
    (dict(w=1000, h=600, profile="coastal", seed=7), 512, (511, 1)),
], ids=["t256", "t1024_window", "coastal_t512"])
def test_compressed_in_compressed_out_matches_oracle(kw, tile, off, gpu_ctx, port, tables):
    b = make_block(**kw)
    h, w = b["esa"].shape
    x_off, y_off = off
    grid = _raster(w + x_off + 50, h + y_off + 70, seed=99, profile="random")
    grid[y_off:y_off + h, x_off:x_off + w] = b["esa"]
    src = capi.TileSource.from_raster(grid, tile, tile, x_off=x_off, y_off=y_off)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    res = gpu_ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"])
    assert sorted(res["tiles"]) == list(range(18))
    for k in range(18):
        assert np.array_equal(assemble(res["tiles"][k], w, h), want[k]), f"plane {k}"
    # identical to the raw-raster entry point, tile for tile
    ref = gpu_ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    assert ref["tiles"] == res["tiles"]


def test_damaged_land_cover_stops_the_block(gpu_ctx):
    b = make_block(w=600, h=520, seed=3)
    src = capi.TileSource.from_raster(b["esa"], 256, 256)
    blob = src.blob.copy()
    blob[int(src.offsets[4]) + 1] ^= 0x01
    bad = capi.TileSource(256, 256, src.tiles_x, src.tiles_y, 0, 0, blob, src.offsets, src.sizes)
    calls = []
    with pytest.raises(capi.Gcn10Error) as ei:
        gpu_ctx.block_tiles_deflate(bad, 600, 520, b["gt"], b["hsg"], b["soil_gt"], on_strip=lambda s: calls.append(1))
    assert ei.value.code == -6 and not calls


def test_prefetch_overlaps_the_next_block_and_results_do_not_change(gpu_ctx, port, tables):
    """gcn10_cuda_tiles_prefetch: block i+1's tiles are uploaded and inflated while block i's strips run; each
    block_tiles_deflate call picks up its own prefetched land cover (oldest first), a call without a prefetch still
    works, and a third prefetch is refused while two are waiting."""
    blocks = [make_block(w=900, h=700, seed=60 + i, esa_patch=30) for i in range(4)]
    srcs = [capi.TileSource.from_raster(b["esa"], 256, 256) for b in blocks]
    wants = [port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables) for b in blocks]

    def check(res, want):
        for k in range(18):
            assert np.array_equal(assemble(res["tiles"][k], 900, 700), want[k])

    gpu_ctx.tiles_prefetch(srcs[0], 900, 700)
    for i in range(4):
        if i + 1 < 4:
            gpu_ctx.tiles_prefetch(srcs[i + 1], 900, 700)
        b = blocks[i]
        check(gpu_ctx.block_tiles_deflate(srcs[i], 900, 700, b["gt"], b["hsg"], b["soil_gt"]), wants[i])
    # no prefetch: inflated inside the call
    check(gpu_ctx.block_tiles_deflate(srcs[2], 900, 700, blocks[2]["gt"], blocks[2]["hsg"], blocks[2]["soil_gt"]), wants[2])
    # two waiting, a third is refused; a call for another block drops nothing it needs and still works
    gpu_ctx.tiles_prefetch(srcs[0], 900, 700)
    gpu_ctx.tiles_prefetch(srcs[1], 900, 700)
    with pytest.raises(capi.Gcn10Error):
        gpu_ctx.tiles_prefetch(srcs[2], 900, 700)
    check(gpu_ctx.block_tiles_deflate(srcs[3], 900, 700, blocks[3]["gt"], blocks[3]["hsg"], blocks[3]["soil_gt"]), wants[3])
    check(gpu_ctx.block_tiles_deflate(srcs[1], 900, 700, blocks[1]["gt"], blocks[1]["hsg"], blocks[1]["soil_gt"]), wants[1])
    out = gpu_ctx.inflate_tiles(srcs[0], 900, 700)
    assert np.array_equal(out, blocks[0]["esa"])


def test_mosaic_parts(gpu_ctx, port, tables):
    """A block window over a mosaic of four source files whose tile grids do not line up (the structure of the
    reference's landcover/esa_worldcover_2021.vrt, where a 36001-pixel window spills one pixel into the
    neighbouring 36000-pixel files): every part is inflated into its rectangle by one launch, pixels no part
    covers read as the fill value, and the chained call gives the oracle's planes."""
    w, h = 1531, 1203
    b = make_block(w=w, h=h, seed=71)
    esa = b["esa"]
    cut_x, cut_y = 1530, 700                      # the last column comes from the right-hand neighbours
    rects = [(0, 0, cut_x, cut_y), (cut_x, 0, w - cut_x, cut_y), (0, cut_y, cut_x, h - cut_y), (cut_x, cut_y, w - cut_x, h - cut_y)]
    parts = []
    for i, (x, y, pw, ph) in enumerate(rects):
        # each source file holds more than the part: the window starts (ox, oy) pixels into its tile grid
        ox, oy = 13 * i, 300 * (i % 2)
        grid = synth.esa_tile(ox + pw + 9, oy + ph + 5, seed=100 + i, patch=40)
        grid[oy:oy + ph, ox:ox + pw] = esa[y:y + ph, x:x + pw]
        tw = (256, 240, 512, 1024)[i]
        src = capi.TileSource.from_raster(grid, tw, tw if i != 1 else 112, x_off=ox, y_off=oy, level=6 if i else 1)
        parts.append((src, x, y, pw, ph))
    got = gpu_ctx.inflate_parts(parts, 0, w, h)
    assert np.array_equal(got, esa)
    want = port.block_rows(esa, b["gt"], b["hsg"], b["soil_gt"], tables)
    res = gpu_ctx.block_parts_deflate(parts, 0, w, h, b["gt"], b["hsg"], b["soil_gt"])
    for k in range(18):
        assert np.array_equal(assemble(res["tiles"][k], w, h), want[k]), k
    # a missing source: its rectangle reads as the fill value (VRT NoDataValue)
    holed = esa.copy()
    x, y, pw, ph = rects[2]
    holed[y:y + ph, x:x + pw] = 80
    got = gpu_ctx.inflate_parts([parts[0], parts[1], parts[3]], 80, w, h)
    assert np.array_equal(got, holed)
    # damaged tile in the second part: reported with its global tile number, GCN10_EDATA
    src1 = parts[1][0]
    blob = src1.blob.copy()
    blob[int(src1.offsets[1])] = 0x79
    bad = capi.TileSource(src1.tile_w, src1.tile_h, src1.tiles_x, src1.tiles_y, src1.x_off, src1.y_off, blob,
                          src1.offsets, src1.sizes)
    rc, _, status = gpu_ctx.inflate_parts([parts[0], (bad,) + parts[1][1:], parts[2], parts[3]], 0, w, h, want_status=True)
    n0 = parts[0][0].tiles_x * parts[0][0].tiles_y
    assert rc == -6 and status[n0 + 1] == 1 and np.count_nonzero(status) == 1
    # parts outside the window / too many parts are refused
    rc, _, _ = gpu_ctx.inflate_parts([(parts[0][0], 5, 0, cut_x, cut_y)], 0, cut_x, cut_y, want_status=True)
    assert rc == -1
    rc, _, _ = gpu_ctx.inflate_parts([parts[3]] * 10, 0, w, h, want_status=True)
    assert rc == -1
