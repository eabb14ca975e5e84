"""TIFF LZW streams from libtiff itself (the library GDAL's GTiff driver links), driven through ctypes.

The encoder and decoder here are libtiff's own LZWEncode / LZWDecode (tif_lzw.c), taken from the copy Pillow bundles,
so streams made for tests and benchmarks are the ones `gdal_translate -co COMPRESS=LZW` writes, and a verdict on a
damaged stream is the one GDAL's read would give.  A tile's stream is made as a one-strip image of the tile's size:
the strip and tile codecs are the same code, and strips take any width (libtiff refuses tile widths that are not
multiples of 16).
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import tempfile

import numpy as np

_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        import PIL
        from PIL import Image  # noqa: F401  (loads the libraries libtiff depends on)
        paths = glob.glob(os.path.join(os.path.dirname(os.path.dirname(PIL.__file__)), "pillow.libs", "libtiff*.so*"))
        if not paths:
            raise RuntimeError("no libtiff found next to Pillow")
        L = C.CDLL(paths[0])
        L.TIFFOpen.restype = C.c_void_p
        L.TIFFOpen.argtypes = [C.c_char_p, C.c_char_p]
        L.TIFFClose.argtypes = [C.c_void_p]
        L.TIFFSetField.argtypes = [C.c_void_p, C.c_uint32]      # variadic: values passed as c_int
        L.TIFFWriteEncodedTile.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_ssize_t]
        L.TIFFWriteEncodedTile.restype = C.c_ssize_t
        L.TIFFWriteEncodedStrip.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_ssize_t]
        L.TIFFWriteEncodedStrip.restype = C.c_ssize_t
        L.TIFFWriteRawStrip.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_ssize_t]
        L.TIFFWriteRawStrip.restype = C.c_ssize_t
        L.TIFFReadEncodedStrip.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_ssize_t]
        L.TIFFReadEncodedStrip.restype = C.c_ssize_t
        L.TIFFReadRawStrip.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_ssize_t]
        L.TIFFReadRawStrip.restype = C.c_ssize_t
        L.TIFFRawStripSize64.argtypes = [C.c_void_p, C.c_uint32]
        L.TIFFRawStripSize64.restype = C.c_uint64
        L.TIFFSetErrorHandler.restype = C.c_void_p
        L.TIFFSetErrorHandler.argtypes = [C.c_void_p]
        L.TIFFSetWarningHandler.restype = C.c_void_p
        L.TIFFSetWarningHandler.argtypes = [C.c_void_p]
        L.TIFFSetErrorHandler(None)           # verdicts are return values; keep libtiff's messages off stderr
        L.TIFFSetWarningHandler(None)
        _LIB = L
    return _LIB


def _open_strips(path, w, rows, nstrips):
    L = _lib()
    t = L.TIFFOpen(os.fsencode(path), b"w")
    if not t:
        raise RuntimeError("TIFFOpen failed")
    for tag, v in [(256, w), (257, rows * nstrips), (258, 8), (277, 1), (262, 1), (284, 1), (259, 5), (278, rows)]:
        L.TIFFSetField(t, tag, C.c_int(v))
    return t


def encode(tiles, tile_w: int, tile_h: int, count: int | None = None) -> list[bytes]:
    """libtiff's LZW stream (no predictor) of every tile_h x tile_w uint8 array in ``tiles`` (an iterable of
    ``count`` arrays, or a sequence)."""
    L = _lib()
    if count is None:
        tiles = list(tiles)
        count = len(tiles)
    with tempfile.TemporaryDirectory(prefix="gcn10_lzw_") as d:
        path = os.path.join(d, "enc.tif")
        t = _open_strips(path, tile_w, tile_h, max(count, 1))
        for i, a in enumerate(tiles):
            a = np.ascontiguousarray(a, dtype=np.uint8)
            assert a.shape == (tile_h, tile_w)
            if L.TIFFWriteEncodedStrip(t, i, a.ctypes.data, a.size) < 0:
                L.TIFFClose(t)
                raise RuntimeError("TIFFWriteEncodedStrip failed")
        L.TIFFClose(t)
        t = L.TIFFOpen(os.fsencode(path), b"r")
        out = []
        for i in range(count):
            n = L.TIFFRawStripSize64(t, i)
            buf = C.create_string_buffer(max(int(n), 1))
            got = L.TIFFReadRawStrip(t, i, buf, n)
            assert got == n
            out.append(buf.raw[:n])
        L.TIFFClose(t)
    return out


def decode(stream: bytes, tile_w: int, tile_h: int):
    """libtiff's reading of one tile's stream: the tile_h x tile_w array, or None where libtiff reports an error."""
    L = _lib()
    with tempfile.TemporaryDirectory(prefix="gcn10_lzw_") as d:
        path = os.path.join(d, "dec.tif")
        t = _open_strips(path, tile_w, tile_h, 1)
        data = bytes(stream) if stream else b"\x00"
        if L.TIFFWriteRawStrip(t, 0, data, len(data)) < 0:
            L.TIFFClose(t)
            raise RuntimeError("TIFFWriteRawStrip failed")
        L.TIFFClose(t)
        t = L.TIFFOpen(os.fsencode(path), b"r")
        out = np.zeros((tile_h, tile_w), dtype=np.uint8)
        n = L.TIFFReadEncodedStrip(t, 0, out.ctypes.data, out.size)
        L.TIFFClose(t)
    return out if n == out.size else None


def write_file(path, a, tile: int | None = 256, predictor: int = 1):
    """An 8-bit LZW TIFF of ``a`` written by libtiff: tiled (tile x tile, a multiple of 16) or, with tile=None, in
    strips of 16 rows; ``predictor`` 1 (none) or 2 (horizontal differencing).  No georeferencing tags."""
    L = _lib()
    a = np.ascontiguousarray(a, dtype=np.uint8)
    h, w = a.shape
    t = L.TIFFOpen(os.fsencode(str(path)), b"w")
    if not t:
        raise RuntimeError("TIFFOpen failed")
    tags = [(256, w), (257, h), (258, 8), (277, 1), (262, 1), (284, 1), (259, 5), (317, predictor)]
    tags += [(322, tile), (323, tile)] if tile else [(278, 16)]
    for tag, v in tags:
        L.TIFFSetField(t, tag, C.c_int(v))
    if tile:
        i = 0
        for ty in range(0, h, tile):
            for tx in range(0, w, tile):
                buf = np.zeros((tile, tile), dtype=np.uint8)
                part = a[ty:ty + tile, tx:tx + tile]
                buf[:part.shape[0], :part.shape[1]] = part
                ok = L.TIFFWriteEncodedTile(t, i, buf.ctypes.data, buf.size) >= 0
                i += 1
                if not ok:
                    L.TIFFClose(t)
                    raise RuntimeError("TIFFWriteEncodedTile failed")
    else:
        for i, y in enumerate(range(0, h, 16)):
            rows = np.ascontiguousarray(a[y:y + 16])
            if L.TIFFWriteEncodedStrip(t, i, rows.ctypes.data, rows.size) < 0:
                L.TIFFClose(t)
                raise RuntimeError("TIFFWriteEncodedStrip failed")
    L.TIFFClose(t)
