"""ctypes binding of libgcn10cuda.so (C ABI: include/gcn10_cuda.h).

This is the thin Python mirror used by the tests and the benchmark harness; the product is the
shared library itself and the C host program in gcn10_b200/host/.  There is no fallback: if the
library is missing or no CUDA device is usable, loading / context creation raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GCN10_CUDA_LIB") or os.path.join(HERE, "libgcn10cuda.so")

NVARIANTS = 9
NPLANES = 18
MASK_DRAINED = 0x001FF
MASK_UNDRAINED = 0x3FE00
MASK_ALL = 0x3FFFF

# every symbol include/gcn10_cuda.h declares
EXPORTS = (
    "gcn10_cuda_version", "gcn10_cuda_last_error", "gcn10_cuda_device_count", "gcn10_cuda_create",
    "gcn10_cuda_destroy", "gcn10_cuda_set_luts", "gcn10_cuda_block", "gcn10_cuda_block_rows",
    "gcn10_cuda_block_deflate", "gcn10_cuda_block_deflate_rows", "gcn10_cuda_block_device",
    "gcn10_cuda_index_maps", "gcn10_cuda_synchronize", "gcn10_cuda_last_kernel_ms",
    "gcn10_cuda_launch_count", "gcn10_cuda_set_option", "gcn10_cuda_host_alloc", "gcn10_cuda_host_free",
    "gcn10_cuda_host_register", "gcn10_cuda_host_unregister", "gcn10_cuda_bind_host_thread",
    "gcn10_cuda_inflate_tiles", "gcn10_cuda_block_tiles_deflate", "gcn10_cuda_last_inflate_ms",
    "gcn10_cuda_tiles_prefetch", "gcn10_cuda_block_async", "gcn10_cuda_wait", "gcn10_cuda_event_query",
    "gcn10_cuda_pcie_probe", "gcn10_cuda_parts_prefetch", "gcn10_cuda_inflate_parts", "gcn10_cuda_block_parts_deflate",
    "gcn10_cuda_last_histograms",
)

_vp = C.c_void_p
_dp = C.POINTER(C.c_double)


class TileStrip(C.Structure):
    """gcn10_tile_strip of include/gcn10_cuda.h."""
    _fields_ = [("tile_row0", C.c_int), ("n_tile_rows", C.c_int), ("tiles_x", C.c_int), ("n_planes", C.c_int),
                ("plane_ids", C.POINTER(C.c_int)), ("offsets", C.POINTER(C.c_uint64)),
                ("sizes", C.POINTER(C.c_uint32)), ("blob", C.POINTER(C.c_uint8)), ("blob_bytes", C.c_size_t),
                ("level", C.c_int), ("level_w", C.c_int), ("level_h", C.c_int), ("aggregate", C.c_int),
                ("framed", C.c_int)]


TILE_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(TileStrip))


class TileSourceStruct(C.Structure):
    """gcn10_tile_source of include/gcn10_cuda.h."""
    _fields_ = [("tile_w", C.c_int), ("tile_h", C.c_int), ("tiles_x", C.c_int), ("tiles_y", C.c_int),
                ("x_off", C.c_int), ("y_off", C.c_int), ("blob", C.c_void_p), ("blob_bytes", C.c_size_t),
                ("offsets", C.c_void_p), ("sizes", C.c_void_p), ("compression", C.c_int)]


COMPRESSION = {"deflate": 8, "lzw": 5}          # TIFF Compression tag values of the codecs the GPU decodes


class TileSource:
    """Compressed tiles of a raster window as a tiled GeoTIFF holds them: one zlib stream per tile (``compression``
    0, 8 or 32946) or one LZW stream per tile (5).

    ``blob`` uint8 [n], ``offsets`` uint64 [tiles_y*tiles_x], ``sizes`` uint32 [tiles_y*tiles_x] (0 = sparse
    tile).  ``from_raster`` builds one from a decoded raster on the host (zlib, or libtiff's LZW encoder): a test /
    benchmark convenience standing in for "read the tile bytes from the file"."""

    def __init__(self, tile_w, tile_h, tiles_x, tiles_y, x_off, y_off, blob, offsets, sizes, compression=0):
        self.tile_w, self.tile_h, self.tiles_x, self.tiles_y = tile_w, tile_h, tiles_x, tiles_y
        self.x_off, self.y_off = x_off, y_off
        self.blob = blob
        self.offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self.sizes = np.ascontiguousarray(sizes, dtype=np.uint32)
        self.compression = compression

    @classmethod
    def from_raster(cls, raster, tile_w=1024, tile_h=1024, level=6, x_off=0, y_off=0, sparse=(), gap=0,
                    pad_value=0, blob_alloc=None, codec="deflate"):
        """Tile ``raster`` (the window occupies raster[y_off:, x_off:] of the grid's pixel space only in the
        sense that the CALLER passes x_off / y_off to say where its window starts).  ``codec`` "deflate" (zlib at
        ``level``; level < 0 stores the raw bytes) or "lzw" (libtiff's encoder, gcn10_b200.tiff_lzw)."""
        import zlib
        if codec not in COMPRESSION:
            raise ValueError(f"codec {codec!r}: expected one of {sorted(COMPRESSION)}")
        h, w = raster.shape
        tiles_x, tiles_y = (w + tile_w - 1) // tile_w, (h + tile_h - 1) // tile_h
        cells = [(ty, tx) for ty in range(tiles_y) for tx in range(tiles_x) if (ty, tx) not in sparse]

        def grid():
            for ty, tx in cells:
                t = np.full((tile_h, tile_w), pad_value, dtype=np.uint8)
                part = raster[ty * tile_h:(ty + 1) * tile_h, tx * tile_w:(tx + 1) * tile_w]
                t[:part.shape[0], :part.shape[1]] = part
                yield t
        if codec == "lzw":
            from . import tiff_lzw
            coded = iter(tiff_lzw.encode(grid(), tile_w, tile_h, len(cells)))
        else:
            coded = (zlib.compress(t.tobytes(), level) if level >= 0 else t.tobytes() for t in grid())
        streams, offsets, sizes = [], [], []
        pos = 0
        for ty in range(tiles_y):
            for tx in range(tiles_x):
                if (ty, tx) in sparse:
                    offsets.append(0)
                    sizes.append(0)
                    continue
                z = next(coded)
                pos += gap
                streams.append(b"\x00" * gap + z)
                offsets.append(pos)
                sizes.append(len(z))
                pos += len(z)
        data = b"".join(streams)
        if blob_alloc is not None:
            blob = blob_alloc(max(len(data), 1))
            blob[:len(data)] = np.frombuffer(data, dtype=np.uint8)
            blob = blob[:len(data)]
        else:
            blob = np.frombuffer(data, dtype=np.uint8).copy()
        return cls(tile_w, tile_h, tiles_x, tiles_y, x_off, y_off, blob, offsets, sizes, COMPRESSION[codec])

    def struct(self):
        return TileSourceStruct(self.tile_w, self.tile_h, self.tiles_x, self.tiles_y, self.x_off, self.y_off,
                                self.blob.ctypes.data, self.blob.size, self.offsets.ctypes.data,
                                self.sizes.ctypes.data, self.compression)


class TilePartStruct(C.Structure):
    """gcn10_tile_part of include/gcn10_cuda.h."""
    _fields_ = [("tiles", TileSourceStruct), ("dst_x", C.c_int), ("dst_y", C.c_int), ("w", C.c_int), ("h", C.c_int)]


def parts_array(parts):
    """[(TileSource, dst_x, dst_y, w, h), ...] -> ctypes array of gcn10_tile_part."""
    arr = (TilePartStruct * len(parts))()
    for i, (src, dx, dy, pw, ph) in enumerate(parts):
        arr[i] = TilePartStruct(src.struct(), dx, dy, pw, ph)
    return arr


class Gcn10Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gcn10cuda error {code}: {msg}")
        self.code = code


def load(path: str = LIB_PATH) -> C.CDLL:
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} not built: run `make cuda` (nvcc -gencode arch=compute_100a,code=sm_100a). "
            "There is no CPU fallback for the Curve Number path.")
    lib = C.CDLL(path)
    lib.gcn10_cuda_version.restype = C.c_char_p
    lib.gcn10_cuda_last_error.restype = C.c_char_p
    lib.gcn10_cuda_create.argtypes = [C.c_int, C.POINTER(_vp)]
    lib.gcn10_cuda_destroy.argtypes = [_vp]
    lib.gcn10_cuda_destroy.restype = None
    lib.gcn10_cuda_set_luts.argtypes = [_vp, _vp]
    blk = [_vp, _vp, C.c_int, C.c_int, C.c_size_t, _dp, _vp, C.c_int, C.c_int, C.c_size_t, _dp,
           C.c_uint, C.POINTER(_vp), C.c_size_t]
    lib.gcn10_cuda_block.argtypes = blk
    lib.gcn10_cuda_block_rows.argtypes = blk[:4] + [C.c_int, C.c_int] + blk[4:]
    lib.gcn10_cuda_block_device.argtypes = blk + [_vp]
    lib.gcn10_cuda_block_async.argtypes = blk + [C.POINTER(_vp)]
    lib.gcn10_cuda_wait.argtypes = [_vp]
    lib.gcn10_cuda_event_query.argtypes = [_vp]
    lib.gcn10_cuda_pcie_probe.argtypes = [_vp, C.c_size_t, C.c_int, _dp]
    lib.gcn10_cuda_block_deflate.argtypes = blk[:12] + [TILE_SINK, _vp]
    lib.gcn10_cuda_block_deflate_rows.argtypes = blk[:4] + [C.c_int, C.c_int] + blk[4:12] + [TILE_SINK, _vp]
    lib.gcn10_cuda_index_maps.argtypes = [_vp, C.c_int, C.c_int, _dp, C.c_int, C.c_int, _dp, _vp, _vp]
    lib.gcn10_cuda_synchronize.argtypes = [_vp]
    lib.gcn10_cuda_last_kernel_ms.argtypes = [_vp, C.POINTER(C.c_float)]
    lib.gcn10_cuda_launch_count.argtypes = [_vp, C.POINTER(C.c_uint64)]
    lib.gcn10_cuda_last_histograms.argtypes = [_vp, _vp]
    lib.gcn10_cuda_set_option.argtypes = [_vp, C.c_char_p, C.c_long]
    lib.gcn10_cuda_host_alloc.argtypes = [C.c_size_t]
    lib.gcn10_cuda_host_alloc.restype = _vp
    lib.gcn10_cuda_host_free.argtypes = [_vp]
    lib.gcn10_cuda_host_free.restype = None
    lib.gcn10_cuda_host_register.argtypes = [_vp, C.c_size_t]
    lib.gcn10_cuda_host_unregister.argtypes = [_vp]
    lib.gcn10_cuda_bind_host_thread.argtypes = [C.c_int]
    lib.gcn10_cuda_inflate_tiles.argtypes = [_vp, C.POINTER(TileSourceStruct), C.c_int, C.c_int, _vp, C.c_size_t, _vp]
    lib.gcn10_cuda_block_tiles_deflate.argtypes = [_vp, C.POINTER(TileSourceStruct), C.c_int, C.c_int, _dp,
                                                   _vp, C.c_int, C.c_int, C.c_size_t, _dp, C.c_uint, TILE_SINK, _vp]
    lib.gcn10_cuda_last_inflate_ms.argtypes = [_vp, C.POINTER(C.c_float)]
    lib.gcn10_cuda_tiles_prefetch.argtypes = [_vp, C.POINTER(TileSourceStruct), C.c_int, C.c_int]
    pp = C.POINTER(TilePartStruct)
    lib.gcn10_cuda_parts_prefetch.argtypes = [_vp, pp, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.gcn10_cuda_inflate_parts.argtypes = [_vp, pp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_size_t, _vp]
    lib.gcn10_cuda_block_parts_deflate.argtypes = [_vp, pp, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _vp, C.c_int, C.c_int,
                                                   C.c_size_t, _dp, C.c_uint, TILE_SINK, _vp]
    return lib


def _d6(a):
    return (C.c_double * 6)(*[float(v) for v in a])


def _rows(a):
    """(array, row pitch in bytes) for a 2-D uint8 array; row-strided views are passed through,
    anything else is copied to C order."""
    if a.ndim == 2 and a.shape[1] > 1 and a.strides[1] == 1 and a.strides[0] >= a.shape[1]:
        return a, a.strides[0]
    a = np.ascontiguousarray(a)
    return a, a.shape[1]


class PinnedArray:
    """uint8 numpy view over page-locked memory from gcn10_cuda_host_alloc."""

    def __init__(self, lib, shape):
        self.lib = lib
        n = int(np.prod(shape))
        self.ptr = lib.gcn10_cuda_host_alloc(n)
        if not self.ptr:
            raise Gcn10Error(-3, lib.gcn10_cuda_last_error().decode())
        buf = (C.c_uint8 * n).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=np.uint8).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            self.lib.gcn10_cuda_host_free(self.ptr)
            self.ptr = None


class Context:
    """One gcn10_ctx: a GPU worker (replaces one MPI rank of the reference)."""

    def __init__(self, device: int = 0, lib: C.CDLL | None = None):
        self.lib = lib or load()
        h = _vp()
        self._check(self.lib.gcn10_cuda_create(device, C.byref(h)))
        self.h = h
        self.device = device
        self._stats = False

    def _check(self, rc):
        if rc != 0:
            raise Gcn10Error(rc, self.lib.gcn10_cuda_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.gcn10_cuda_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_luts(self, tables):
        t = np.ascontiguousarray(tables, dtype=np.int32)
        assert t.shape == (NVARIANTS, 256, 5), t.shape
        self._check(self.lib.gcn10_cuda_set_luts(self.h, t.ctypes.data))

    def set_option(self, key: str, value: int):
        self._check(self.lib.gcn10_cuda_set_option(self.h, key.encode(), int(value)))
        if key == "stats":
            self._stats = bool(value)

    def last_histograms(self) -> np.ndarray:
        """uint64 [18, 256]: per plane, the pixels of each value in the last block a compressed-tile call completed
        with option "stats" on (gcn10_cuda_last_histograms)."""
        out = np.zeros((NPLANES, 256), dtype=np.uint64)
        self._check(self.lib.gcn10_cuda_last_histograms(self.h, out.ctypes.data))
        return out

    def _histograms(self):
        """The result dicts' ``histograms``: None while option "stats" is off, or no block has completed (a band
        that does not end its block)."""
        if not self._stats:
            return None
        out = np.zeros((NPLANES, 256), dtype=np.uint64)
        return out if self.lib.gcn10_cuda_last_histograms(self.h, out.ctypes.data) == 0 else None

    def index_maps(self, w, h, gt, hsx, hsy, soil_gt):
        ci = np.empty(w, dtype=np.int32)
        cj = np.empty(h, dtype=np.int32)
        self._check(self.lib.gcn10_cuda_index_maps(self.h, w, h, _d6(gt), hsx, hsy, _d6(soil_gt),
                                                   ci.ctypes.data, cj.ctypes.data))
        return ci, cj

    def block(self, esa, gt, hsg, soil_gt, plane_mask=MASK_ALL, out=None):
        """Host-buffer call.  esa [h,w] uint8, hsg [hsy,hsx] uint8 (numpy, any row stride).
        Returns uint8 [18,h,w]; planes not in the mask are left untouched (zeros if allocated here)."""
        assert esa.dtype == np.uint8 and hsg.dtype == np.uint8
        esa, esa_pitch = _rows(esa)
        hsg, hsg_pitch = _rows(hsg)
        h, w = esa.shape
        hsy, hsx = hsg.shape
        if out is None:
            out = np.zeros((NPLANES, h, w), dtype=np.uint8)
        ptrs = (_vp * NPLANES)()
        for k in range(NPLANES):
            ptrs[k] = out[k].ctypes.data if plane_mask & (1 << k) else None
        self._check(self.lib.gcn10_cuda_block(
            self.h, esa.ctypes.data, w, h, esa_pitch, _d6(gt), hsg.ctypes.data, hsx, hsy,
            hsg_pitch, _d6(soil_gt), plane_mask, ptrs, out.strides[1]))
        return out

    def block_async(self, esa, gt, hsg, soil_gt, plane_mask=MASK_ALL, out=None):
        """Queues a block and returns a handle; ``wait(handle)`` returns the uint8 [18,h,w] result.  The arrays
        are kept alive by the handle (use page-locked arrays for copies that really overlap)."""
        esa, esa_pitch = _rows(esa)
        hsg, hsg_pitch = _rows(hsg)
        h, w = esa.shape
        hsy, hsx = hsg.shape
        if out is None:
            out = np.zeros((NPLANES, h, w), dtype=np.uint8)
        ptrs = (_vp * NPLANES)()
        for k in range(NPLANES):
            ptrs[k] = out[k].ctypes.data if plane_mask & (1 << k) else None
        ev = _vp()
        self._check(self.lib.gcn10_cuda_block_async(
            self.h, esa.ctypes.data, w, h, esa_pitch, _d6(gt), hsg.ctypes.data, hsx, hsy,
            hsg_pitch, _d6(soil_gt), plane_mask, ptrs, out.strides[1], C.byref(ev)))
        return dict(event=ev, out=out, keep=(esa, hsg, ptrs))

    def query(self, handle) -> bool:
        rc = self.lib.gcn10_cuda_event_query(handle["event"])
        if rc < 0:
            self._check(rc)
        return rc == 1

    def wait(self, handle):
        ev, handle["event"] = handle["event"], None
        self._check(self.lib.gcn10_cuda_wait(ev))
        return handle["out"]

    def pcie_probe(self, nbytes=256 << 20, reps=4):
        g = (C.c_double * 3)()
        self._check(self.lib.gcn10_cuda_pcie_probe(self.h, nbytes, reps, g))
        return {"h2d_gbs": g[0], "d2h_gbs": g[1], "d2h_ship_kernel_gbs": g[2]}

    def block_rows(self, esa_rows, h, row0, gt, hsg, soil_gt, plane_mask=MASK_ALL):
        """Band call: esa_rows holds rows [row0, row0+len) of a block that is h rows tall."""
        esa_rows, esa_pitch = _rows(esa_rows)
        hsg, hsg_pitch = _rows(hsg)
        nrows, w = esa_rows.shape
        hsy, hsx = hsg.shape
        out = np.zeros((NPLANES, nrows, w), dtype=np.uint8)
        ptrs = (_vp * NPLANES)()
        for k in range(NPLANES):
            ptrs[k] = out[k].ctypes.data if plane_mask & (1 << k) else None
        self._check(self.lib.gcn10_cuda_block_rows(
            self.h, esa_rows.ctypes.data, w, h, row0, nrows, esa_pitch, _d6(gt), hsg.ctypes.data,
            hsx, hsy, hsg_pitch, _d6(soil_gt), plane_mask, ptrs, out.strides[1]))
        return out

    def _deflate_call(self, fn, on_strip, *args):
        """Runs the compressed-tile library call ``fn(ctx, *args, sink, NULL)`` with a sink that files every tile of a
        strip (level 0 under tiles, overview level k under overviews[k], the mean rasters under aggregate) unless
        ``on_strip(strip_struct)`` takes the strips instead; returns block_deflate's result dict."""
        tiles, overviews, aggregate, total = {}, {}, {}, [0]

        def sink(_user, sp):
            st = sp.contents
            total[0] += st.blob_bytes
            if on_strip is not None:
                return int(on_strip(st) or 0)
            blob = C.string_at(st.blob, st.blob_bytes)
            dest = aggregate if st.aggregate else tiles if st.level == 0 else overviews.setdefault(st.level, {})
            for k in range(st.n_planes):
                d = dest.setdefault(st.plane_ids[k], {})
                for tr in range(st.n_tile_rows):
                    for tx in range(st.tiles_x):
                        i = (k * st.n_tile_rows + tr) * st.tiles_x + tx
                        d[(st.tile_row0 + tr, tx)] = blob[st.offsets[i]: st.offsets[i] + st.sizes[i]]
            return 0

        cb = TILE_SINK(sink)
        self._check(fn(self.h, *args, cb, None))
        return dict(tiles=tiles, overviews=overviews, aggregate=aggregate, bytes=total[0], histograms=self._histograms())

    def block_deflate(self, esa, gt, hsg, soil_gt, plane_mask=MASK_ALL, on_strip=None):
        """Compressed-tile call.  Returns dict(tiles={plane: {(tile_row, tile_x): bytes}},
        overviews={level: {plane: {(tile_row, tile_x): bytes}}} (option "overviews"), bytes=total,
        histograms=uint64 [18, 256] (option "stats", else None), aggregate={plane: {(tile_row, tile_x): bytes}} (the f x f mean
        rasters of option "aggregate", else empty)); with ``on_strip(strip_struct)`` the tiles are not
        copied."""
        esa, esa_pitch = _rows(esa)
        hsg, hsg_pitch = _rows(hsg)
        h, w = esa.shape
        hsy, hsx = hsg.shape
        return self._deflate_call(self.lib.gcn10_cuda_block_deflate, on_strip, esa.ctypes.data, w, h, esa_pitch,
                                  _d6(gt), hsg.ctypes.data, hsx, hsy, hsg_pitch, _d6(soil_gt), plane_mask)

    def block_deflate_rows(self, esa_rows, h, row0, gt, hsg, soil_gt, plane_mask=MASK_ALL, on_strip=None):
        """Band form of block_deflate: esa_rows holds rows [row0, row0+len) of a block that is h rows tall; the
        result holds this band's tiles (and, for the band that ends the block, its overview levels and mean rasters)."""
        esa_rows, esa_pitch = _rows(esa_rows)
        hsg, hsg_pitch = _rows(hsg)
        nrows, w = esa_rows.shape
        hsy, hsx = hsg.shape
        return self._deflate_call(self.lib.gcn10_cuda_block_deflate_rows, on_strip, esa_rows.ctypes.data, w, h, row0,
                                  nrows, esa_pitch, _d6(gt), hsg.ctypes.data, hsx, hsy, hsg_pitch, _d6(soil_gt),
                                  plane_mask)

    def inflate_tiles(self, src: "TileSource", w, h, out=None, want_status=False):
        """GPU inflate of a tile source into a host raster uint8 [h, w]."""
        if out is None:
            out = np.zeros((h, w), dtype=np.uint8)
        status = np.full(src.tiles_x * src.tiles_y, -1, dtype=np.int32)
        st = src.struct()
        rc = self.lib.gcn10_cuda_inflate_tiles(self.h, C.byref(st), w, h, out.ctypes.data, out.strides[0],
                                               status.ctypes.data)
        if want_status:
            return rc, out, status
        self._check(rc)
        return out

    def block_tiles_deflate(self, src: "TileSource", w, h, gt, hsg, soil_gt, plane_mask=MASK_ALL, on_strip=None):
        """Compressed land-cover tiles in, compressed Curve Number tiles out (same result layout as
        block_deflate)."""
        hsg, hsg_pitch = _rows(hsg)
        hsy, hsx = hsg.shape
        st = src.struct()
        return self._deflate_call(self.lib.gcn10_cuda_block_tiles_deflate, on_strip, C.byref(st), w, h, _d6(gt),
                                  hsg.ctypes.data, hsx, hsy, hsg_pitch, _d6(soil_gt), plane_mask)

    def inflate_parts(self, parts, fill, w, h, want_status=False):
        """GPU inflate of a mosaic ([(TileSource, dst_x, dst_y, w, h), ...]) into a host raster uint8 [h, w]."""
        out = np.zeros((h, w), dtype=np.uint8)
        n = sum(p[0].tiles_x * p[0].tiles_y for p in parts)
        status = np.full(n, -1, dtype=np.int32)
        arr = parts_array(parts)
        rc = self.lib.gcn10_cuda_inflate_parts(self.h, arr, len(parts), fill, w, h, out.ctypes.data, out.strides[0],
                                               status.ctypes.data)
        if want_status:
            return rc, out, status
        self._check(rc)
        return out

    def block_parts_deflate(self, parts, fill, w, h, gt, hsg, soil_gt, plane_mask=MASK_ALL, on_strip=None):
        """Mosaic form of block_tiles_deflate; same result layout."""
        hsg, hsg_pitch = _rows(hsg)
        hsy, hsx = hsg.shape
        return self._deflate_call(self.lib.gcn10_cuda_block_parts_deflate, on_strip, parts_array(parts), len(parts), fill,
                                  w, h, _d6(gt), hsg.ctypes.data, hsx, hsy, hsg_pitch, _d6(soil_gt), plane_mask)

    def tiles_prefetch(self, src: "TileSource", w, h):
        """Start upload + GPU inflate of a block's tiles; the next block_tiles_deflate / inflate_tiles call with the
        same source picks the result up.  Keep ``src`` alive until then."""
        st = src.struct()
        self._check(self.lib.gcn10_cuda_tiles_prefetch(self.h, C.byref(st), w, h))

    def last_inflate_ms(self) -> float:
        v = C.c_float()
        self._check(self.lib.gcn10_cuda_last_inflate_ms(self.h, C.byref(v)))
        return v.value

    def block_device(self, d_esa, w, h, esa_pitch, gt, d_hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask,
                     d_out_ptrs, out_pitch, stream=None):
        """Device-buffer call; pointers are integers (e.g. torch.Tensor.data_ptr())."""
        ptrs = (_vp * NPLANES)()
        for k in range(NPLANES):
            ptrs[k] = d_out_ptrs[k] if (plane_mask & (1 << k)) and d_out_ptrs[k] else None
        self._check(self.lib.gcn10_cuda_block_device(
            self.h, d_esa, w, h, esa_pitch, _d6(gt), d_hsg, hsx, hsy, hsg_pitch, _d6(soil_gt),
            plane_mask, ptrs, out_pitch, stream))

    def synchronize(self):
        self._check(self.lib.gcn10_cuda_synchronize(self.h))

    def last_kernel_ms(self) -> float:
        v = C.c_float()
        self._check(self.lib.gcn10_cuda_last_kernel_ms(self.h, C.byref(v)))
        return v.value

    def launch_count(self) -> int:
        v = C.c_uint64()
        self._check(self.lib.gcn10_cuda_launch_count(self.h, C.byref(v)))
        return v.value
