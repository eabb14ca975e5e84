"""Rasters shared by the CPU tests of the GeoTIFF writer's overview levels and Cloud Optimized GeoTIFF layout."""
import zlib

import numpy as np

GT = (-114.0, 1.0 / 12000.0, 0.0, 42.0, 0.0, -1.0 / 12000.0)
SIZES = [(1, 1), (15, 7), (257, 257), (4111, 260), (48, 3000), (3001, 517)]


def raster(w, h, seed):
    rng = np.random.default_rng(seed)
    # patches, so that the tiles compress like land cover and the levels differ from plain subsampling by rows
    a = rng.integers(0, 12, size=((h + 6) // 7, (w + 4) // 5), dtype=np.uint8) * 10
    a = np.repeat(np.repeat(a, 7, axis=0), 5, axis=1)[:h, :w]
    return np.ascontiguousarray(a + rng.integers(0, 2, size=(h, w), dtype=np.uint8))


def tile_rows(img):
    """[tile_row] -> the zlib streams of that row of 256 x 256 tiles, zero padded."""
    h, w = img.shape
    out = []
    for ty in range(0, h, 256):
        row = []
        for tx in range(0, w, 256):
            t = np.zeros((256, 256), np.uint8)
            part = img[ty:ty + 256, tx:tx + 256]
            t[:part.shape[0], :part.shape[1]] = part
            row.append(zlib.compress(t.tobytes(), 6))
        out.append(row)
    return out
