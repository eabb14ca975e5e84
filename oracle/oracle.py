"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY.

Python front-end of the parity checker for the GCN10 Curve Number hot path:

* ``Port``  -- ctypes binding of ``oracle/libcn_oracle.so`` (the plain-C restatement,
  ``oracle/cn_oracle.c``),
* ``Ref``   -- ctypes binding of ``oracle/_ref/libgcn10_ref.so`` (the reference's own
  ``src/cn.c`` + ``src/raster.c`` compiled unmodified over RAM GDAL/OGR/MPI stand-ins),
* ``numpy_block`` -- a vectorised numpy restatement for small cases.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  Nothing under ``gcn10_b200/`` does.
Parity status: PINNED (see ``cn_oracle.h``).  Citations are relative to /root/reference/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "libcn_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libgcn10_ref.so")

NPLANES = 18
HCS = ("p", "f", "g")          # cn.c:146
ARCS = ("i", "ii", "iii")      # cn.c:147
CONDS = ("drained", "undrained")  # cn.c:145

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_ip = C.POINTER(C.c_int)


def plane_names():
    """Names of the 18 planes in the reference's save order (cn.c:236,258-259,308)."""
    return [f"{c}/{h}_{a}" for c in CONDS for h in HCS for a in ARCS]


def build(ref: bool = True) -> None:
    """Compile the restatement and, when /root/reference is present, the _ref library."""
    subprocess.check_call(["make", "-s", "-C", HERE, "port"])
    if ref:
        subprocess.check_call(["make", "-s", "-C", HERE, "ref"])


def _d6(a):
    return (C.c_double * 6)(*[float(v) for v in a])


def _d4(a):
    return (C.c_double * 4)(*[float(v) for v in a])


def _u8(a):
    return a.ctypes.data_as(_u8p)


class Port:
    """The plain-C restatement (oracle/cn_oracle.c)."""

    def __init__(self, path: str = PORT_SO):
        if not os.path.exists(path):
            build(ref=False)
        self.lib = C.CDLL(path)
        L = self.lib
        L.cn_oracle_parse_lookup.argtypes = [C.c_char_p, C.c_void_p]
        L.cn_oracle_load_tables.argtypes = [C.c_char_p, C.c_void_p]
        L.cn_oracle_window.argtypes = [C.c_int, C.c_int, _dp, _dp, _ip, _ip, _ip, _ip, _dp]
        L.cn_oracle_col_index.argtypes = [C.c_int, _dp, _dp, C.c_int, C.c_void_p]
        L.cn_oracle_row_index.argtypes = [C.c_int, _dp, _dp, C.c_int, C.c_void_p]
        L.cn_oracle_block_rows.argtypes = [_u8p, C.c_int, C.c_int, _dp, _u8p, C.c_int, C.c_int, _dp,
                                           C.c_void_p, C.c_int, C.c_int, _u8p, C.c_size_t]
        L.cn_oracle_col_index.restype = None
        L.cn_oracle_row_index.restype = None

    def parse_lookup(self, csv_path: str) -> np.ndarray:
        t = np.empty((256, 5), dtype=np.int32)
        rc = self.lib.cn_oracle_parse_lookup(csv_path.encode(), t.ctypes.data)
        if rc:
            raise OSError(f"cn_oracle_parse_lookup({csv_path}) -> {rc}")
        return t

    def load_tables(self, lookup_dir: str) -> np.ndarray:
        t = np.empty((9, 256, 5), dtype=np.int32)
        rc = self.lib.cn_oracle_load_tables(lookup_dir.encode(), t.ctypes.data)
        if rc:
            raise OSError(f"cn_oracle_load_tables({lookup_dir}) -> {rc}")
        return t

    def window(self, rw, rh, t, bbox):
        xo, yo, xc, yc = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        gt = (C.c_double * 6)()
        rc = self.lib.cn_oracle_window(rw, rh, _d6(t), _d4(bbox), xo, yo, xc, yc, gt)
        if rc:
            return None
        return xo.value, yo.value, xc.value, yc.value, tuple(gt)

    def col_index(self, w, gt, soil_gt, hsx) -> np.ndarray:
        out = np.empty(max(w, 0), dtype=np.int32)
        self.lib.cn_oracle_col_index(w, _d6(gt), _d6(soil_gt), hsx, out.ctypes.data)
        return out

    def row_index(self, h, gt, soil_gt, hsy) -> np.ndarray:
        out = np.empty(max(h, 0), dtype=np.int32)
        self.lib.cn_oracle_row_index(h, _d6(gt), _d6(soil_gt), hsy, out.ctypes.data)
        return out

    def block_rows(self, esa, gt, hsg, soil_gt, tables, y0=0, y1=None, h=None) -> np.ndarray:
        """18 planes for rows [y0,y1) of a block; returns uint8 [18, y1-y0, w].

        ``esa`` is either the whole window [h, w] (default) or, when ``h`` (the block's row
        count) is given, just the rows [y0,y1) -- for spot checks of very large blocks."""
        esa = np.ascontiguousarray(esa, dtype=np.uint8)
        hsg = np.ascontiguousarray(hsg, dtype=np.uint8)
        tables = np.ascontiguousarray(tables, dtype=np.int32)
        w = esa.shape[1]
        hh, hw = hsg.shape
        if h is None:
            h = esa.shape[0]
            y1 = h if y1 is None else y1
            rows = esa[y0:y1]
        else:
            assert y1 is not None and esa.shape[0] == y1 - y0
            rows = esa
        rows = np.ascontiguousarray(rows)
        out = np.empty((NPLANES, y1 - y0, w), dtype=np.uint8)
        rc = self.lib.cn_oracle_block_rows(_u8(rows), w, h, _d6(gt), _u8(hsg), hw, hh, _d6(soil_gt),
                                           tables.ctypes.data, y0, y1, _u8(out), (y1 - y0) * w)
        if rc:
            raise MemoryError("cn_oracle_block_rows")
        return out

    def run_block(self, esa_raster, esa_t, hsg_raster, hsg_t, bbox, lookup_dir, *, block_id=1):
        """What ``Ref.run_block`` returns for the rasters process_block() saves (nplanes, w, h, gt, paths,
        planes), restated: both windows cut from ``bbox``, a block whose window is invalid in either raster is
        skipped (nplanes == 0, cn.c:188-192), else the 18 planes in the save order (cn.c:236,258-259,308)."""
        esa_raster = np.ascontiguousarray(esa_raster, dtype=np.uint8)
        hsg_raster = np.ascontiguousarray(hsg_raster, dtype=np.uint8)
        we = self.window(esa_raster.shape[1], esa_raster.shape[0], esa_t, bbox)
        wh = self.window(hsg_raster.shape[1], hsg_raster.shape[0], hsg_t, bbox)
        if we is None or wh is None:
            return dict(nplanes=0, w=0, h=0, gt=(0.0,) * 6, paths=[], planes=None)
        xo, yo, xc, yc, gt = we
        hxo, hyo, hxc, hyc, sgt = wh
        planes = self.block_rows(esa_raster[yo:yo + yc, xo:xo + xc], gt, hsg_raster[hyo:hyo + hyc, hxo:hxo + hxc], sgt,
                                 self.load_tables(lookup_dir))
        paths = [f"cn_rasters_{c}/cn_{h}_{a}_{block_id}.tif" for c in CONDS for h in HCS for a in ARCS]
        return dict(nplanes=NPLANES, w=xc, h=yc, gt=gt, paths=paths, planes=planes)


class Ref:
    """The reference's own object code (oracle/_ref/libgcn10_ref.so)."""

    def __init__(self, path: str = REF_SO):
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} missing: build it in the container that has /root/reference (make -C oracle ref)")
        self.lib = C.CDLL(path)
        L = self.lib
        L.refshim_run_block.argtypes = [_u8p, C.c_int, C.c_int, _dp, _u8p, C.c_int, C.c_int, _dp, _dp,
                                        C.c_char_p, C.c_char_p, C.c_int, C.c_int, _u8p, C.c_size_t,
                                        _ip, _ip, _dp]
        L.refshim_window.argtypes = [C.c_int, C.c_int, _dp, _dp, _ip, _ip, _ip, _ip, _dp]
        L.refshim_log.restype = C.c_char_p
        L.refshim_plane_path.restype = C.c_char_p
        L.refshim_plane_path.argtypes = [C.c_int]
        L.refshim_create_option.restype = C.c_char_p
        L.refshim_create_option.argtypes = [C.c_int]
        L.refshim_plane_time.restype = C.c_double
        L.refshim_plane_time.argtypes = [C.c_int]

    @staticmethod
    def available(path: str = REF_SO) -> bool:
        return os.path.exists(path)

    def log(self) -> str:
        return self.lib.refshim_log().decode(errors="replace")

    def window(self, rw, rh, t, bbox):
        xo, yo, xc, yc = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        gt = (C.c_double * 6)()
        rc = self.lib.refshim_window(rw, rh, _d6(t), _d4(bbox), xo, yo, xc, yc, gt)
        if rc:
            return None
        return xo.value, yo.value, xc.value, yc.value, tuple(gt)

    def run_block(self, esa_raster, esa_t, hsg_raster, hsg_t, bbox, lookup_dir, *, block_id=1,
                  overwrite=True, keep=True, scratch_dir=None):
        """process_block() on one bbox of two in-memory rasters.

        Returns dict(planes=uint8[18,h,w] or None, w, h, gt, paths, times, nplanes, log).
        ``planes`` is None when keep=False (timing only) or when the reference skipped
        the block (nplanes == 0, see ``log``).
        """
        esa_raster = np.ascontiguousarray(esa_raster, dtype=np.uint8)
        hsg_raster = np.ascontiguousarray(hsg_raster, dtype=np.uint8)
        eh, ew = esa_raster.shape
        hh, hw = hsg_raster.shape
        # capacity: the window can never exceed the raster itself
        cap = ew * eh
        out = np.empty((NPLANES, cap), dtype=np.uint8) if keep else None
        ow, oh = C.c_int(), C.c_int()
        ogt = (C.c_double * 6)()
        tmp = None
        if scratch_dir is None:
            tmp = tempfile.TemporaryDirectory(prefix="gcn10_ref_")
            scratch_dir = tmp.name
        try:
            n = self.lib.refshim_run_block(
                _u8(esa_raster), ew, eh, _d6(esa_t), _u8(hsg_raster), hw, hh, _d6(hsg_t), _d4(bbox),
                os.fsencode(lookup_dir), os.fsencode(scratch_dir), int(block_id), int(bool(overwrite)),
                _u8(out) if keep else None, cap, ow, oh, ogt)
        finally:
            if tmp is not None:
                tmp.cleanup()
        res = dict(nplanes=n, w=ow.value, h=oh.value, gt=tuple(ogt), log=self.log(),
                   paths=[self.lib.refshim_plane_path(k).decode() for k in range(max(n, 0))],
                   times=[self.lib.refshim_plane_time(k) for k in range(max(n, 0))],
                   options=[self.lib.refshim_create_option(k).decode() for k in range(2)],
                   planes=None)
        if keep and n > 0:
            w, h = ow.value, oh.value
            res["planes"] = np.ascontiguousarray(out[:n, : w * h].reshape(n, h, w))
        return res


# --------------------------------------------------------------------------- numpy restatement


def c_round(x: np.ndarray) -> np.ndarray:
    """C99 round(): half away from zero, evaluated without an inexact x+0.5 (cn.c:225-226)."""
    t = np.trunc(x)
    frac = np.abs(x - t)                      # exact for doubles
    return np.where(frac >= 0.5, t + np.copysign(1.0, x), t)


def _to_int_x86(v: np.ndarray) -> np.ndarray:
    ok = (v > -2147483649.0) & (v < 2147483648.0)
    out = np.full(v.shape, -2**31, dtype=np.int64)
    out[ok] = v[ok].astype(np.int64)
    return out


def numpy_index_maps(w, h, gt, soil_gt, hsx, hsy):
    """cn.c:219-229 as separate IEEE operations (numpy never fuses multiply-add)."""
    with np.errstate(all="ignore"):
        x = np.arange(w, dtype=np.float64)
        y = np.arange(h, dtype=np.float64)
        px = np.float64(gt[0]) + (x + 0.5) * np.float64(gt[1])
        py = np.float64(gt[3]) + (y + 0.5) * np.float64(gt[5])
        dc = (px - np.float64(soil_gt[0])) / np.float64(soil_gt[1])
        dr = (np.float64(soil_gt[3]) - py) / np.abs(np.float64(soil_gt[5]))
        ci = np.clip(_to_int_x86(c_round(dc)), 0, hsx - 1).astype(np.int32)
        cj = np.clip(_to_int_x86(c_round(dr)), 0, hsy - 1).astype(np.int32)
    return ci, cj


def numpy_block(esa, gt, hsg, soil_gt, tables) -> np.ndarray:
    """All 18 planes of a block, vectorised; for small cases (cn.c:218-290)."""
    esa = np.asarray(esa, dtype=np.uint8)
    hsg = np.asarray(hsg, dtype=np.uint8)
    h, w = esa.shape
    hh, hw = hsg.shape
    ci, cj = numpy_index_maps(w, h, gt, soil_gt, hw, hh)
    res = hsg[cj[:, None], ci[None, :]]                                   # cn.c:230
    out = np.empty((NPLANES, h, w), dtype=np.uint8)
    for c in range(2):
        adj = res.copy()
        dual = (adj >= 11) & (adj <= 14)
        if c == 0:
            adj[dual] = 4                                                  # cn.c:92-98
        else:
            adj[dual] = adj[dual] - 10                                     # cn.c:99-110
        valid = adj < 5                                                    # cn.c:123-124
        sg = np.where(valid, adj, 0).astype(np.intp)
        for t in range(9):
            v = np.asarray(tables[t])[esa.astype(np.intp), sg]
            keep = valid & (v < 255)                                       # cn.c:126
            out[c * 9 + t] = np.where(keep, v.astype(np.int64) & 0xFF, 255).astype(np.uint8)
    return out
