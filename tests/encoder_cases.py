"""Inputs for the exact-stream tests of the GPU tile encoders (tests/test_gpu_encoder_exact.py, tests/test_stream_ref.py):
lookup tables that put the library into each code regime, blocks in which every record occurs, and tiles with a
controlled number of new pixels."""
import numpy as np

from tests.cases import make_block

T = 256
HSG_CODES = np.array([0, 1, 2, 3, 4, 11, 12, 13, 14, 7, 255], np.uint8)    # every soil class, 9 twice
# the tuned code's shape for a number of values: (literal bits, longest literal/length code, bits of symbol 285)
SHAPES = {2: (3, 9, 2), 4: (4, 9, 2), 8: (5, 9, 2), 16: (6, 9, 2), 32: (7, 9, 2), 64: (8, 9, 2), 128: (8, 9, 3),
          192: (8, 10, 4), 224: (8, 11, 5), 240: (8, 12, 6)}


def _variants(mask):
    return sorted({k % 9 for k in range(18) if mask >> k & 1})


def tables_with_values(nvals, mask, seed=0):
    """Tables whose selected planes hold exactly ``nvals`` byte values (0 and nodata 255 included) in at most 255
    records: the values sit in the cells (variant, land cover, soil group) of a few land-cover classes, every other
    entry is 255.  A land cover holds values below 144 (8-bit fixed-code literals) or at and above it (9-bit), never
    both, so that under the fixed code all planes share one literal class."""
    rng = np.random.default_rng(seed)
    t = np.full((9, 256, 5), 255, np.int32)
    pool = [0] + sorted(rng.choice(np.arange(1, 255), size=nvals - 2, replace=False).tolist())
    var = _variants(mask)
    per_lc = 5 * len(var)
    free = list(rng.permutation(256))
    for half in ([v for v in pool if v < 144], [v for v in pool if v >= 144]):
        lcs = [free.pop() for _ in range(-(-len(half) // per_lc))]
        cells = [(v, lc, sg) for lc in lcs for v in var for sg in range(5)]
        for i, ci in enumerate(rng.permutation(len(cells))):
            v, lc, sg = cells[ci]
            t[v, lc, sg] = half[i % len(half)]
    return t


def tables_with_records(nrec, mask):
    """Tables with exactly ``nrec`` records over the selected planes: land covers 0 .. nrec-2 get a record of their own
    at soil code 0 (values below 144), everything else is nodata."""
    t = np.full((9, 256, 5), 255, np.int32)
    var = _variants(mask)
    for i in range(nrec - 1):
        for j, v in enumerate(var):
            t[v, i, 0] = i if len(var) == 1 else (i % 143 if j == 0 else (i // 143 + 7 * j) % 143)
    return t


def tables_with_classes(tables, ncls):
    """The shipped tables (all values below 144) with a 9-bit literal (>= 144) in ncls - 1 variants, at land cover
    10, 20, ... and soil group B: the drained plane of each such variant gets a 9-bit-literal pattern of its own."""
    t = tables.copy()
    for v in range(ncls - 1):
        t[v, 10 * (v + 1), 1] = 200 + v
    return t


def random_block(w, h, seed):
    """Land cover uniform over 0..255 and soil codes from every class, so that every record occurs."""
    rng = np.random.default_rng(seed)
    b = make_block(w=w, h=h, seed=seed, hsg_patch=1)
    b["esa"] = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    # patches of 8 x 8 pixels keep most tiles compressible; a few noisy rows break runs
    b["esa"] = np.kron(b["esa"][::8, ::8], np.ones((8, 8), np.uint8))[:h, :w].copy()
    b["esa"][::37] = rng.integers(0, 256, size=b["esa"][::37].shape, dtype=np.uint8)
    b["hsg"] = HSG_CODES[rng.integers(0, len(HSG_CODES), size=b["hsg"].shape)]
    return b


def noisy_tile(n, seed, pool):
    """A 256 x 256 land-cover tile: land cover 10 with the first n pixels of a fixed random order replaced by classes
    from ``pool``.  The stream grows with n."""
    rng = np.random.default_rng(seed)
    t = np.full(T * T, 10, np.uint8)
    order = rng.permutation(T * T)
    t[order[:n]] = rng.choice(pool, size=n)
    return t.reshape(T, T)
