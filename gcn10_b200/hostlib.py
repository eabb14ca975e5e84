"""ctypes binding of gcn10_b200/host/libgcn10host.so -- the CUDA-free part of the C host program
(config file, lookup CSVs, window arithmetic, block list, shapefile extents, GeoTIFF I/O).
Used by the tests and by bench.py to read lookup tables exactly as the gcn10 executable does."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "host", "libgcn10host.so")
EXE_PATH = os.path.join(HERE, "host", "gcn10")
ERRLEN = 512

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_vp = C.c_void_p


class Window(C.Structure):
    _fields_ = [("xoff", C.c_int), ("yoff", C.c_int), ("xcount", C.c_int), ("ycount", C.c_int),
                ("gt", C.c_double * 6)]


class Config(C.Structure):
    _fields_ = [(k, C.c_char_p) for k in ("hysogs_data_path", "esa_data_path", "blocks_shp_path",
                                           "lookup_table_path", "log_dir")]


class HostError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gcn10 host error {code}: {msg}")
        self.code = code
        self.msg = msg


_lib = None


def load(path: str | None = None) -> C.CDLL:
    """The host library (cached), or -- path given -- another build of it, e.g. one with the GDAL backend."""
    global _lib
    if path is None and _lib is not None:
        return _lib
    lib_path = path or LIB_PATH
    if not os.path.exists(lib_path):
        raise FileNotFoundError(f"{lib_path} not built: run `make host`")
    L = C.CDLL(lib_path)
    L.gh_load_lookup_tables.argtypes = [C.c_char_p, _vp, C.c_char_p, C.c_size_t]
    L.gh_load_lookup_table.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, _vp, C.c_char_p, C.c_size_t]
    L.gh_raster_window.argtypes = [C.c_int, C.c_int, _dp, _dp, C.POINTER(Window)]
    L.gh_config_parse.argtypes = [C.c_char_p, C.POINTER(Config), C.c_char_p, C.c_size_t]
    L.gh_config_free.argtypes = [C.POINTER(Config)]
    L.gh_read_block_list.argtypes = [C.c_char_p, C.POINTER(_ip), _ip]
    L.gh_blocks_open.argtypes = [C.c_char_p, C.POINTER(_vp), C.c_char_p, C.c_size_t]
    L.gh_blocks_count.argtypes = [_vp]
    L.gh_blocks_id.argtypes = [_vp, C.c_int]
    L.gh_blocks_bbox.argtypes = [_vp, C.c_int, _dp]
    L.gh_blocks_close.argtypes = [_vp]
    L.gh_blocks_close.restype = None
    L.gh_tiff_open.argtypes = [C.c_char_p, C.POINTER(_vp), C.c_char_p, C.c_size_t]
    L.gh_tiff_size.argtypes = [_vp, _ip, _ip]
    L.gh_tiff_geotransform.argtypes = [_vp, _dp]
    L.gh_tiff_read_window.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_size_t, C.c_int,
                                      C.c_char_p, C.c_size_t]
    L.gh_tiff_close.argtypes = [_vp]
    L.gh_tiff_close.restype = None
    L.gh_tiff_window_tiles_plan.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]
    L.gh_tiff_window_tiles_read.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_char_p, C.c_size_t]
    L.gh_tiff_write.argtypes = [C.c_char_p, _vp, C.c_int, C.c_int, C.c_size_t, _dp, C.c_int, C.c_char_p, C.c_size_t]
    L.gh_tiff_write_cog.argtypes = [C.c_char_p, _vp, C.c_int, C.c_int, C.c_size_t, _dp, C.c_int, C.c_int, C.c_char_p,
                                    C.c_size_t]
    L.gh_tiffw_open.argtypes = [C.c_char_p, C.c_int, C.c_int, _dp, C.POINTER(_vp), C.c_char_p, C.c_size_t]
    L.gh_tiffw_put_tile_row.argtypes = [_vp, C.c_int, _vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
    L.gh_tiffw_put_tile_rows.argtypes = [_vp, C.c_int, C.c_int, _vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
    L.gh_tiffw_write_rows.argtypes = [_vp, _vp, C.c_size_t, C.c_int, C.c_int, C.c_int]
    L.gh_tiffw_set_overviews.argtypes = [_vp, C.c_int]
    L.gh_tiffw_levels.argtypes = [_vp]
    L.gh_tiffw_set_stats.argtypes = [_vp, C.c_int]
    L.gh_tiffw_put_histogram.argtypes = [_vp, C.POINTER(C.c_uint64)]
    L.gh_tiffw_set_nodata.argtypes = [_vp, C.c_int]
    L.gh_tiffw_set_cog.argtypes = [_vp, C.c_int]
    L.gh_tiffw_put_framed_tile_rows.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, C.POINTER(C.c_uint64),
                                                C.POINTER(C.c_uint32)]
    L.gh_tiffw_put_level_tile_rows.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, C.POINTER(C.c_uint64),
                                               C.POINTER(C.c_uint32)]
    L.gh_tiffw_close.argtypes = [_vp]
    L.gh_tiffw_abort.argtypes = [_vp]
    L.gh_tiffw_abort.restype = None
    L.gh_raster_open.argtypes = [C.c_char_p, C.POINTER(_vp), C.c_char_p, C.c_size_t]
    L.gh_raster_size.argtypes = [_vp, _ip, _ip]
    L.gh_raster_geotransform.argtypes = [_vp, _dp]
    L.gh_raster_is_mosaic.argtypes = [_vp]
    L.gh_raster_source_count.argtypes = [_vp]
    L.gh_raster_fill.argtypes = [_vp]
    L.gh_raster_read_window.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_size_t, C.c_int,
                                        C.c_char_p, C.c_size_t]
    L.gh_raster_window_parts.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _ip, C.c_char_p, C.c_size_t]
    L.gh_raster_close.argtypes = [_vp]
    L.gh_raster_close.restype = None
    L.gh_raster_backend.argtypes = [_vp]
    L.gh_raster_backend.restype = C.c_char_p
    L.gh_raster_have_gdal.argtypes = []
    L.gh_log_open.argtypes = [C.c_char_p, C.c_int]
    L.gh_log_open.restype = _vp
    L.gh_log_message.argtypes = [_vp, C.c_char_p, C.c_char_p, C.c_int]
    L.gh_log_message.restype = None
    L.gh_log_close.argtypes = [_vp]
    L.gh_log_close.restype = None
    if path is None:
        _lib = L
    return L


def _err():
    return C.create_string_buffer(ERRLEN)


def load_lookup_tables(lookup_dir: str) -> np.ndarray:
    """int32 [9,256,5] in the reference's order p_i..g_iii (cn.c:146-147)."""
    L = load()
    t = np.empty((9, 256, 5), dtype=np.int32)
    e = _err()
    rc = L.gh_load_lookup_tables(os.fsencode(lookup_dir), t.ctypes.data, e, ERRLEN)
    if rc:
        raise HostError(rc, e.value.decode(errors="replace"))
    return t


def raster_window(rw, rh, t, bbox):
    L = load()
    w = Window()
    rc = L.gh_raster_window(rw, rh, (C.c_double * 6)(*t), (C.c_double * 4)(*bbox), C.byref(w))
    if rc:
        return None
    return w.xoff, w.yoff, w.xcount, w.ycount, tuple(w.gt)


def parse_config(path: str) -> dict:
    L = load()
    cfg = Config()
    e = _err()
    rc = L.gh_config_parse(os.fsencode(path), C.byref(cfg), e, ERRLEN)
    if rc:
        raise HostError(rc, e.value.decode(errors="replace"))
    out = {k: getattr(cfg, k).decode(errors="replace") for k, _ in Config._fields_}
    L.gh_config_free(C.byref(cfg))
    return out


def read_block_list(path: str):
    L = load()
    ids = _ip()
    n = C.c_int()
    rc = L.gh_read_block_list(os.fsencode(path), C.byref(ids), C.byref(n))
    if rc:
        raise HostError(rc, f"cannot open block list file {path}")
    out = [ids[i] for i in range(n.value)]
    C.CDLL(None).free(ids)
    return out


class Blocks:
    def __init__(self, shp_path: str):
        self.L = load()
        h = _vp()
        e = _err()
        rc = self.L.gh_blocks_open(os.fsencode(shp_path), C.byref(h), e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        self.h = h

    def __len__(self):
        return self.L.gh_blocks_count(self.h)

    def ids(self):
        return [self.L.gh_blocks_id(self.h, i) for i in range(len(self))]

    def bbox(self, block_id):
        b = (C.c_double * 4)()
        if self.L.gh_blocks_bbox(self.h, block_id, b):
            return None
        return tuple(b)

    def close(self):
        if self.h:
            self.L.gh_blocks_close(self.h)
            self.h = None


def tiff_write(path: str, data: np.ndarray, gt, threads: int = 4):
    L = load()
    data = np.ascontiguousarray(data, dtype=np.uint8)
    h, w = data.shape
    e = _err()
    rc = L.gh_tiff_write(os.fsencode(path), data.ctypes.data, w, h, w, (C.c_double * 6)(*gt), threads, e, ERRLEN)
    if rc:
        raise HostError(rc, e.value.decode(errors="replace"))


def tiff_write_cog(path: str, data: np.ndarray, gt, overviews: int = 16, threads: int = 4):
    """The whole raster as a Cloud Optimized GeoTIFF with up to ``overviews`` levels sampled on the host
    (gh_tiff_write_cog): the CPU reference of the COG layout."""
    L = load()
    data = np.ascontiguousarray(data, dtype=np.uint8)
    h, w = data.shape
    e = _err()
    rc = L.gh_tiff_write_cog(os.fsencode(path), data.ctypes.data, w, h, w, (C.c_double * 6)(*gt), overviews, threads, e,
                             ERRLEN)
    if rc:
        raise HostError(rc, e.value.decode(errors="replace"))


class GeoKeys(C.Structure):
    """gh_geokeys of gcn10_host.h."""
    _fields_ = [("keys", C.POINTER(C.c_uint16)), ("n_keys", C.c_size_t), ("doubles", _dp), ("n_doubles", C.c_size_t),
                ("ascii", C.c_char_p), ("n_ascii", C.c_size_t)]


class Tiff:
    def __init__(self, path: str):
        self.L = load()
        h = _vp()
        e = _err()
        rc = self.L.gh_tiff_open(os.fsencode(path), C.byref(h), e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        self.h = h
        w, hh = C.c_int(), C.c_int()
        self.L.gh_tiff_size(h, w, hh)
        self.width, self.height = w.value, hh.value
        gt = (C.c_double * 6)()
        self.georeferenced = self.L.gh_tiff_geotransform(h, gt) == 0
        self.gt = tuple(gt)

    def read(self, xoff=0, yoff=0, xcount=None, ycount=None, threads=4) -> np.ndarray:
        xcount = self.width - xoff if xcount is None else xcount
        ycount = self.height - yoff if ycount is None else ycount
        out = np.empty((ycount, xcount), dtype=np.uint8)
        e = _err()
        rc = self.L.gh_tiff_read_window(self.h, xoff, yoff, xcount, ycount, out.ctypes.data, xcount, threads, e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        return out

    def window_tiles(self, xoff=0, yoff=0, xcount=None, ycount=None, threads=4):
        """The compressed tiles of a window as they lie in the file (gh_tiff_window_tiles_plan / _read), or None when
        the dataset cannot be handed to the GPU decoder (not tiled, neither DEFLATE nor LZW, predictor 2).
        Returns dict(tile_w, tile_h, tiles_x, tiles_y, x_in, y_in, blob, offsets, sizes, compression)."""
        xcount = self.width - xoff if xcount is None else xcount
        ycount = self.height - yoff if ycount is None else ycount
        plan = TilePlan()
        if self.L.gh_tiff_window_tiles_plan(self.h, xoff, yoff, xcount, ycount, C.byref(plan)) != 0:
            return None
        n = plan.tiles_x * plan.tiles_y
        blob = np.zeros(max(plan.blob_bytes, 1), dtype=np.uint8)
        offsets = np.zeros(n, dtype=np.uint64)
        sizes = np.zeros(n, dtype=np.uint32)
        e = _err()
        rc = self.L.gh_tiff_window_tiles_read(self.h, C.byref(plan), blob.ctypes.data, offsets.ctypes.data,
                                              sizes.ctypes.data, threads, e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        return dict(tile_w=plan.tile_w, tile_h=plan.tile_h, tiles_x=plan.tiles_x, tiles_y=plan.tiles_y, x_in=plan.x_in,
                    y_in=plan.y_in, blob=blob[:plan.blob_bytes], offsets=offsets, sizes=sizes,
                    compression=plan.compression)

    def close(self):
        if self.h:
            self.L.gh_tiff_close(self.h)
            self.h = None


class TilePlan(C.Structure):
    """gh_tile_plan of gcn10_host.h."""
    _fields_ = [("tile_w", C.c_int), ("tile_h", C.c_int), ("tx0", C.c_int), ("ty0", C.c_int), ("tiles_x", C.c_int),
                ("tiles_y", C.c_int), ("x_in", C.c_int), ("y_in", C.c_int), ("blob_bytes", C.c_size_t),
                ("compression", C.c_int)]


class RasterPart(C.Structure):
    """gh_raster_part of gcn10_host.h."""
    _fields_ = [("ds", _vp), ("plan", TilePlan), ("dst_x", C.c_int), ("dst_y", C.c_int), ("w", C.c_int), ("h", C.c_int)]


class Raster:
    """gh_raster: a GeoTIFF or a VRT mosaic of GeoTIFFs, as GDALOpen() would present it (raster.c:119)."""

    def __init__(self, path: str, lib: C.CDLL | None = None):
        self.L = lib or load()
        h = _vp()
        e = _err()
        rc = self.L.gh_raster_open(os.fsencode(path), C.byref(h), e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        self.h = h
        w, hh = C.c_int(), C.c_int()
        self.L.gh_raster_size(h, w, hh)
        self.width, self.height = w.value, hh.value
        gt = (C.c_double * 6)()
        self.L.gh_raster_geotransform(h, gt)
        self.gt = tuple(gt)
        self.is_mosaic = bool(self.L.gh_raster_is_mosaic(h))
        self.source_count = self.L.gh_raster_source_count(h)
        self.fill = self.L.gh_raster_fill(h)
        self.backend = self.L.gh_raster_backend(h).decode()     # "geotiff", "vrt" or "gdal"

    def read(self, xoff, yoff, xcount, ycount, threads=4, pitch=None) -> np.ndarray:
        pitch = xcount if pitch is None else pitch
        out = np.zeros((max(ycount, 0), max(pitch, 1)), dtype=np.uint8)
        e = _err()
        rc = self.L.gh_raster_read_window(self.h, xoff, yoff, xcount, ycount, out.ctypes.data, pitch, threads, e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        return out[:, :xcount]

    def window_parts(self, xoff, yoff, xcount, ycount, max_parts=9, threads=4):
        """(rc, parts): rc 0 -> parts = [dict(dst_x, dst_y, w, h, tile_w, tile_h, tiles_x, tiles_y, x_in, y_in, blob,
        offsets, sizes, compression)] ready for capi.TileSource; rc 1 -> decode on the host; raises when a source is missing."""
        arr = (RasterPart * max_parts)()
        n = C.c_int()
        e = _err()
        rc = self.L.gh_raster_window_parts(self.h, xoff, yoff, xcount, ycount, arr, max_parts, C.byref(n), e, ERRLEN)
        if rc < 0:
            raise HostError(rc, e.value.decode(errors="replace"))
        parts = []
        for k in range(n.value if rc == 0 else 0):
            plan = arr[k].plan
            nt = plan.tiles_x * plan.tiles_y
            blob = np.zeros(max(plan.blob_bytes, 1), dtype=np.uint8)
            offsets = np.zeros(nt, dtype=np.uint64)
            sizes = np.zeros(nt, dtype=np.uint32)
            r2 = self.L.gh_tiff_window_tiles_read(arr[k].ds, C.byref(plan), blob.ctypes.data, offsets.ctypes.data,
                                                  sizes.ctypes.data, threads, e, ERRLEN)
            if r2:
                raise HostError(r2, e.value.decode(errors="replace"))
            parts.append(dict(dst_x=arr[k].dst_x, dst_y=arr[k].dst_y, w=arr[k].w, h=arr[k].h, tile_w=plan.tile_w,
                              tile_h=plan.tile_h, tiles_x=plan.tiles_x, tiles_y=plan.tiles_y, x_in=plan.x_in,
                              y_in=plan.y_in, blob=blob[:plan.blob_bytes], offsets=offsets, sizes=sizes,
                              compression=plan.compression))
        return rc, parts

    def close(self):
        if self.h:
            self.L.gh_raster_close(self.h)
            self.h = None


class TiffWriter:
    """Incremental tiled-DEFLATE GeoTIFF writer (gh_tiffw_*): raw row bands or pre-compressed tile rows.
    ``overviews=n`` adds up to n overview levels (gh_tiffw_set_overviews); ``levels`` is how many the file gets.
    ``stats=True`` adds the NoData tag and the band statistics (gh_tiffw_set_stats): write_rows counts the pixels itself,
    tiles put already compressed need ``put_histogram``.  ``nodata=True`` adds the NoData tag alone (gh_tiffw_set_nodata)."""

    def __init__(self, path: str, w: int, h: int, gt, overviews: int = 0, stats: bool = False, nodata: bool = False,
                 geokeys=None, cog: bool = False):
        self.L = load()
        h_ = _vp()
        e = _err()
        rc = self.L.gh_tiffw_open(os.fsencode(path), w, h, (C.c_double * 6)(*gt), C.byref(h_), e, ERRLEN)
        if rc:
            raise HostError(rc, e.value.decode(errors="replace"))
        self.h = h_
        self.tiles_x = (w + 255) // 256
        if overviews and self.L.gh_tiffw_set_overviews(h_, overviews):
            self.L.gh_tiffw_abort(h_)
            self.h = None
            raise HostError(-1, f"gh_tiffw_set_overviews({overviews}) failed")
        if stats and self.L.gh_tiffw_set_stats(h_, 1):
            self.L.gh_tiffw_abort(h_)
            self.h = None
            raise HostError(-1, "gh_tiffw_set_stats(1) failed")
        if nodata and self.L.gh_tiffw_set_nodata(h_, 1):
            self.L.gh_tiffw_abort(h_)
            self.h = None
            raise HostError(-1, "gh_tiffw_set_nodata(1) failed")
        if geokeys is not None:
            keys, doubles, ascii = geokeys
            k = (C.c_uint16 * len(keys))(*keys)
            d = (C.c_double * max(len(doubles), 1))(*doubles)
            a = ascii.encode() if ascii else None
            gk = GeoKeys(k, len(keys), d if doubles else None, len(doubles), a, len(a) if a else 0)
            fn = self.L["gh_tiffw_set_geokeys"]     # (a function object of its own: tests bind the symbol their way)
            fn.argtypes = [_vp, C.POINTER(GeoKeys)]
            if fn(h_, C.byref(gk)):
                self.L.gh_tiffw_abort(h_)
                self.h = None
                raise HostError(-1, "gh_tiffw_set_geokeys failed")
        if cog and self.L.gh_tiffw_set_cog(h_, 1):
            self.L.gh_tiffw_abort(h_)
            self.h = None
            raise HostError(-1, "gh_tiffw_set_cog(1) failed")
        self.levels = self.L.gh_tiffw_levels(h_)

    def put_histogram(self, hist):
        """hist: 256 pixel counts of the full-resolution raster (added to what the writer has counted)."""
        a = np.ascontiguousarray(hist, dtype=np.uint64)
        assert a.shape == (256,), a.shape
        return self.L.gh_tiffw_put_histogram(self.h, a.ctypes.data_as(C.POINTER(C.c_uint64)))

    def put_tile_row(self, tile_row: int, streams, level: int = 0):
        """streams: the zlib streams (bytes) of one tile row of ``level`` (0 = full resolution)."""
        if level == 0:
            assert len(streams) == self.tiles_x
        blob = b"".join(streams)
        offs = (C.c_uint64 * len(streams))()
        sizes = (C.c_uint32 * len(streams))()
        pos = 0
        for i, z in enumerate(streams):
            offs[i], sizes[i] = pos, len(z)
            pos += len(z)
        buf = C.create_string_buffer(blob, max(len(blob), 1))
        if level == 0:
            return self.L.gh_tiffw_put_tile_row(self.h, tile_row, buf, offs, sizes)
        return self.L.gh_tiffw_put_level_tile_rows(self.h, level, tile_row, 1, buf, offs, sizes)

    def put_tile_rows(self, level: int, tile_row0: int, nrows: int, blob, offsets, sizes, framed: bool = False):
        """``nrows`` tile rows of ``level`` at once, [nrows][tiles_x] tiles: tile i is blob[offsets[i] : offsets[i] +
        sizes[i]] (gh_tiffw_put_level_tile_rows; ``framed``: the tiles carry their COG leader and trailer in blob,
        gh_tiffw_put_framed_tile_rows)."""
        n = len(sizes)
        buf = C.create_string_buffer(bytes(blob), max(len(blob), 1))
        offs = (C.c_uint64 * n)(*[int(v) for v in offsets])
        sz = (C.c_uint32 * n)(*[int(v) for v in sizes])
        f = self.L.gh_tiffw_put_framed_tile_rows if framed else self.L.gh_tiffw_put_level_tile_rows
        return f(self.h, level, tile_row0, nrows, buf, offs, sz)

    def write_rows(self, data: np.ndarray, y0: int, threads: int = 2):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        return self.L.gh_tiffw_write_rows(self.h, data.ctypes.data, data.shape[1], y0, data.shape[0], threads)

    def close(self):
        rc = self.L.gh_tiffw_close(self.h)
        self.h = None
        return rc


def write_tiled_deflate_tiff(path: str, w: int, h: int, tile_w: int, tile_h: int, blob, offsets, sizes, gt):
    """Assembles a tiled DEFLATE GeoTIFF (classic TIFF, Compression = 8, no predictor) from zlib streams that are
    already compressed: blob[offsets[i] : offsets[i] + sizes[i]] is tile i, row-major over the ceil(w / tile_w) x
    ceil(h / tile_h) grid.  Used by bench.py / tools to turn the benchmark's compressed land-cover tiles (1024 x
    1024, the layout of the ESA WorldCover files) into the file the gcn10 executable reads, without re-encoding."""
    import struct
    tx, ty = (w + tile_w - 1) // tile_w, (h + tile_h - 1) // tile_h
    n = tx * ty
    assert len(offsets) == n and len(sizes) == n
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    pos = 8
    file_off = []
    for i in range(n):
        file_off.append(pos)
        pos += int(sizes[i])
    pos += pos & 1
    data_off = pos                                  # TileOffsets | TileByteCounts | scale | tiepoint | geokeys
    off_offsets, off_counts = data_off, data_off + 4 * n
    off_scale = off_counts + 4 * n
    off_tie = off_scale + 24
    off_keys = off_tie + 48
    geokeys = [1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2048, 0, 1, 4326]
    off_ifd = off_keys + 2 * len(geokeys)
    off_ifd += off_ifd & 1
    assert off_ifd + 512 < 2**32, "classic TIFF only"
    entries = [(256, 4, 1, w), (257, 4, 1, h), (258, 3, 1, 8), (259, 3, 1, 8), (262, 3, 1, 1), (277, 3, 1, 1),
               (284, 3, 1, 1), (322, 3, 1, tile_w), (323, 3, 1, tile_h),
               (324, 4, n, file_off[0] if n == 1 else off_offsets), (325, 4, n, int(sizes[0]) if n == 1 else off_counts),
               (339, 3, 1, 1), (33550, 12, 3, off_scale), (33922, 12, 6, off_tie), (34735, 3, len(geokeys), off_keys)]
    with open(path, "wb") as f:
        f.write(struct.pack("<2sHI", b"II", 42, off_ifd))
        for i in range(n):
            o, s_ = int(offsets[i]), int(sizes[i])
            f.write(blob[o:o + s_].tobytes())
        f.write(b"\0" * (data_off - f.tell()))
        f.write(struct.pack(f"<{n}I", *file_off))
        f.write(struct.pack(f"<{n}I", *[int(v) for v in sizes]))
        f.write(struct.pack("<3d", gt[1], -gt[5], 0.0))
        f.write(struct.pack("<6d", 0.0, 0.0, 0.0, gt[0], gt[3], 0.0))
        f.write(struct.pack(f"<{len(geokeys)}H", *geokeys))
        f.write(b"\0" * (off_ifd - f.tell()))
        f.write(struct.pack("<H", len(entries)))
        for tag, typ, cnt, val in entries:
            if typ == 3 and cnt == 1:
                f.write(struct.pack("<HHIHH", tag, typ, cnt, val, 0))
            else:
                f.write(struct.pack("<HHII", tag, typ, cnt, val))
        f.write(struct.pack("<I", 0))
    return path
