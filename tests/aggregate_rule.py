"""The mean-raster rule of include/gcn10_cuda.h (gcn10_aggregate_*), restated in numpy for the tests: the f x f mean of
a plane, cells aligned to pixel (0, 0), edge cells covering the pixels they have, 255 (nodata) left out of the mean,
rounded half up, and 255 only for a cell whose pixels are all 255."""
import numpy as np

NODATA = 255
MAX_FACTOR = 1024


def dim(n, f):
    return -(-n // f)


def sums(plane, f):
    """(sum, count) uint64 [ch, cw] of the pixels that are not 255, per f x f cell."""
    h, w = plane.shape
    ch, cw = dim(h, f), dim(w, f)
    p = np.zeros((ch * f, cw * f), np.uint64)
    valid = np.zeros((ch * f, cw * f), np.uint64)
    p[:h, :w] = plane
    valid[:h, :w] = plane != NODATA
    p *= valid
    s = p.reshape(ch, f, cw, f).sum(axis=(1, 3))
    n = valid.reshape(ch, f, cw, f).sum(axis=(1, 3))
    return s, n


def value(s, n):
    """gcn10_aggregate_value, elementwise."""
    s, n = np.asarray(s, np.uint64), np.asarray(n, np.uint64)
    safe = np.maximum(n, 1)
    return np.where(n > 0, (2 * s + n) // (2 * safe), NODATA).astype(np.uint8)


def mean(plane, f):
    """uint8 [ceil(h / f), ceil(w / f)]: the mean raster of a plane."""
    return value(*sums(plane, f))
