"""The overview rule of include/gcn10_cuda.h (gcn10_overview_dim / _src / _levels) restated in numpy, for the tests."""
import numpy as np


def dim(n, k):
    return (n + (1 << k) - 1) >> k


def src(i, k, n):
    return np.minimum((np.asarray(i, dtype=np.int64) << k) + ((1 << k) >> 1), n - 1)


def levels(w, h, max_levels=16):
    k = 0
    while k < max_levels and (dim(w, k) > 256 or dim(h, k) > 256):
        k += 1
    return k


def decimate(a, k):
    """Level k of a 2-D raster (or of the last two axes of a stack): every level samples level 0."""
    h, w = a.shape[-2:]
    rows = src(np.arange(dim(h, k)), k, h)
    cols = src(np.arange(dim(w, k)), k, w)
    return a[..., rows[:, None], cols[None, :]]
