"""Property-style GPU parity: seeded random block shapes, pixel sizes, HSG ratios, origin shifts, data
profiles and plane masks; every output byte must equal the oracle's."""
import numpy as np
import pytest

from gcn10_b200 import capi
from tests import stream_ref as S
from tests.cases import make_block, PX, PX_VRT

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", range(24))
def test_random_block(seed, gpu_ctx, port, tables):
    rng = np.random.default_rng(1000 + seed)
    w = int(rng.choice([1, 7, 16, 31, 255, 256, 257, 1023, 4095, 4096, 4097, 6000, int(rng.integers(1, 9000))]))
    h = int(rng.choice([1, 2, 11, 12, 13, 25, 255, 256, 257, int(rng.integers(1, 1200))]))
    px = float(rng.choice([PX, PX_VRT, 1.0 / 3600.0, 0.00025]))
    ratio = float(rng.choice([25.0, 25.0, 10.0, 3.0, 1.0, 0.5, 7.3, 60.0]))
    shift = (float(rng.uniform(0, 2)) * px * ratio, float(rng.uniform(0, 2)) * px * ratio)
    kw = dict(w=w, h=h, px=px, hsg_px=px * ratio, shift=shift, margin=int(rng.integers(0, 3)),
              lon0=float(rng.integers(-180, 177)), lat0=float(rng.integers(-57, 84)), seed=seed,
              profile=str(rng.choice(["worldcover", "random", "coastal"])),
              esa_patch=int(rng.choice([8, 48, 192])), hsg_patch=int(rng.choice([1, 3, 9])))
    b = make_block(**kw)
    mask = int(rng.choice([capi.MASK_ALL, capi.MASK_DRAINED, capi.MASK_UNDRAINED, int(rng.integers(1, 1 << 18))]))
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)
    for k in range(18):
        if mask & (1 << k):
            assert np.array_equal(got[k], want[k]), (kw, hex(mask), k)
        else:
            assert not got[k].any()


@pytest.mark.parametrize("seed", range(16))
def test_random_block_through_the_compressed_tile_chain(seed, gpu_ctx, port, tables):
    """The same property through gcn10_cuda_block_tiles_deflate: random input tile sizes and zlib levels, the
    window at a random position inside the tile grid, random plane masks; every output tile is inflated with
    zlib and compared with the oracle's plane, and equals the reference encoder's stream byte for byte."""
    import zlib
    rng = np.random.default_rng(5000 + seed)
    w = int(rng.choice([1, 16, 255, 256, 257, 700, 1023, 1025, int(rng.integers(1, 2600))]))
    h = int(rng.choice([1, 12, 255, 256, 257, 511, int(rng.integers(1, 1500))]))
    px = float(rng.choice([PX, PX_VRT]))
    ratio = float(rng.choice([25.0, 25.0, 25.0, 10.0, 3.0, 1.0, 7.3, 60.0]))
    shift = (float(rng.uniform(0, 2)) * px * ratio, float(rng.uniform(0, 2)) * px * ratio)
    kw = dict(w=w, h=h, px=px, hsg_px=px * ratio, shift=shift, margin=int(rng.integers(0, 3)),
              lon0=float(rng.integers(-180, 177)), lat0=float(rng.integers(-57, 84)), seed=seed,
              profile=str(rng.choice(["worldcover", "worldcover", "random", "coastal"])),
              esa_patch=int(rng.choice([8, 48, 192])), hsg_patch=int(rng.choice([1, 3, 9])))
    b = make_block(**kw)
    tw, th = [(256, 256), (512, 512), (1024, 1024), (128, 64), (240, 112), (1024, 256)][int(rng.integers(0, 6))]
    x_off, y_off = int(rng.integers(0, 2 * tw)), int(rng.integers(0, 2 * th))
    grid = rng.integers(0, 256, size=(y_off + h + int(rng.integers(0, th)), x_off + w + int(rng.integers(0, tw))),
                        dtype=np.uint8)
    grid[y_off:y_off + h, x_off:x_off + w] = b["esa"]
    src = capi.TileSource.from_raster(grid, tw, th, level=int(rng.choice([0, 1, 6, 9])), x_off=x_off, y_off=y_off,
                                      gap=int(rng.integers(0, 9)))
    mask = int(rng.choice([capi.MASK_ALL, capi.MASK_DRAINED, capi.MASK_UNDRAINED, int(rng.integers(1, 1 << 18))]))
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    res = gpu_ctx.block_tiles_deflate(src, w, h, b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask)
    assert sorted(res["tiles"]) == [k for k in range(18) if mask & (1 << k)]
    T = 256
    for k, tiles in res["tiles"].items():
        full = np.zeros(((h + T - 1) // T * T, (w + T - 1) // T * T), dtype=np.uint8)
        for (r, c), z in tiles.items():
            full[r * T:(r + 1) * T, c * T:(c + 1) * T] = np.frombuffer(zlib.decompress(z), dtype=np.uint8).reshape(T, T)
        assert np.array_equal(full[:h, :w], want[k]), (kw, (tw, th, x_off, y_off), hex(mask), k)
        assert not full[h:, :].any() and not full[:, w:].any()
    S.check_tiles(res["tiles"], {k: want[k] for k in res["tiles"]}, S.regime(tables, mask), f"seed {seed}")
