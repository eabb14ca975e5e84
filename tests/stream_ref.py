"""The exact bytes the GPU tile encoders write, predicted on the CPU.

tests/harness/tile_code_host.cpp holds a scalar reference of both encoders (cn_deflate_fused_kernel and
deflate_tiles_kernel); this module picks the encoder and the code the library picks for a set of lookup tables and a
plane mask (``regime``, the rules of build_fused_tables in gcn10_cuda.cu) and encodes planes tile by tile with it.
The planes are the oracle's: a pixel's record is the tuple of its values over the selected planes, so the oracle's
planes carry everything the fused kernel's parse sees.  DESIGN.md section 4.5 lists the rules; this module and the
harness define the stream format the tests hold the kernels to.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from dataclasses import dataclass, field

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "harness", "tile_code_host.cpp")
T = 256
STORED_BYTES = 2 + 2 * 5 + T * T + 4
NPLANES = 18
MODE_FIELDS = ("stored", "stored_mask", "template", "rounds", "fine", "pieces", "classes", "maxp")

_lib = None


def lib() -> C.CDLL:
    """The harness, compiled once per process into a temporary directory."""
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="gcn10_stream_ref_"), "libtile_code_host.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", "-o", out, SRC])
        L = C.CDLL(out)
        L.gcn10_ref_fused_new.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.gcn10_ref_fused_new.restype = C.c_void_p
        L.gcn10_ref_fused_free.argtypes = [C.c_void_p]
        L.gcn10_ref_fused_tile.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p]
        L.gcn10_ref_fused_tile.restype = C.c_int
        L.gcn10_ref_plain_tile.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]
        L.gcn10_ref_plain_tile.restype = C.c_uint32
        L.gcn10_test_tile_tokens.argtypes = [C.c_void_p, C.c_void_p]
        L.gcn10_test_tile_code_lengths.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def cn_byte(v: int) -> int:
    """A table entry as a plane byte: below 255 it wraps to 8 bits (negatives too), 255 and above are nodata."""
    return v & 255 if v < 255 else 255


def soil_code(sc: int) -> int:
    """Soil class 0..9 of the fused kernel -> a raw HYSOGs code: 0, 1..4 (A..D), 11..14 (dual groups), other."""
    return sc if sc <= 4 else 11 + sc - 5 if sc <= 8 else 255


def records(tables, mask: int) -> list[tuple]:
    """The distinct value records of the selected planes, in the order build_fused_tables numbers them: land cover
    0..255, soil class 0..9 (9 = any code that is not 0..4 or 11..14: nodata in every plane).  A dual group 11..14
    is soil group D (4) under drained conditions (planes 0..8) and A..D under undrained ones (planes 9..17)."""
    planes = [k for k in range(NPLANES) if mask >> k & 1]
    t = np.asarray(tables, dtype=np.int64)
    seen, out = set(), []
    for lc in range(256):
        for sc in range(10):
            code = soil_code(sc)
            rec = []
            for k in planes:
                cond, v = divmod(k, 9)
                sg = code
                if 11 <= code <= 14:
                    sg = 4 if cond == 0 else code - 10
                rec.append(cn_byte(int(t[v, lc, sg])) if sg < 5 else 255)
            rec = tuple(rec)
            if rec not in seen:
                seen.add(rec)
                out.append(rec)
    return out


@dataclass
class Regime:
    """Which encoder and code the library uses: path "tuned" / "fixed" (cn_deflate_fused_kernel with the tuned code of
    tile_code.h or RFC 1951's fixed code) or "two_kernel" (cn_block_kernel + deflate_tiles_kernel)."""
    path: str
    mask: int
    n_records: int
    n_values: int
    present: np.ndarray
    cls: list = field(default_factory=list)       # 9-bit-literal class per selected plane (fixed code)
    shape: tuple | None = None                    # tuned code: (lit_bits, longest code, bits of symbol 285)

    @property
    def planes(self):
        return [k for k in range(NPLANES) if self.mask >> k & 1]

    @property
    def fused(self):
        return self.path != "two_kernel"


def code_shape(present) -> tuple | None:
    """(literal bits, longest literal/length code, bits of symbol 285) of the tuned code for these values, None when
    there is none (more than 240 values)."""
    p = np.ascontiguousarray(present, dtype=np.uint8)
    bits = (C.c_int * 29)()
    eob, lit, hdr = C.c_int(), C.c_int(), C.c_int()
    if lib().gcn10_test_tile_code_lengths(p.ctypes.data, bits, C.byref(eob), C.byref(lit), C.byref(hdr)):
        return None
    return lit.value, max(list(bits) + [eob.value]), bits[28]


def regime(tables, mask: int, fused: int = 1, tuned_code: int = 1) -> Regime:
    """build_fused_tables (gcn10_cuda.cu) restated.  It depends on the tables and the mask, not on a block's pixels:
      * more than 255 records (id 255 is the padding's): two-kernel path;
      * the values the planes can hold -- every record value, and 0 for the padding -- make the tuned code when they
        are at most 240 (and option tuned_code is on);
      * else the fixed code, whose 8- and 9-bit literals (values >= 144) must fall in at most 3 patterns ("classes")
        over the records across the planes, else the two-kernel path."""
    recs = records(tables, mask)
    present = np.zeros(256, np.uint8)
    present[0] = 1
    for r in recs:
        present[list(r)] = 1
    nv = int(present.sum())
    base = dict(mask=mask, n_records=len(recs), n_values=nv, present=present)
    if not fused or len(recs) > 255:
        return Regime("two_kernel", **base)
    shape = code_shape(present)
    if tuned_code and shape is not None:
        return Regime("tuned", cls=[0] * bin(mask).count("1"), shape=shape, **base)
    patterns, cls = [], []
    for j in range(bin(mask).count("1")):
        pat = tuple(r[j] >= 144 for r in recs)
        if pat not in patterns:
            if len(patterns) >= 3:
                return Regime("two_kernel", **base)
            patterns.append(pat)
        cls.append(patterns.index(pat))
    return Regime("fixed", cls=cls, **base)


def _tiles_of(h, w):
    return [(r, c) for r in range((h + T - 1) // T) for c in range((w + T - 1) // T)]


def fused_tiles(planes: dict, reg: Regime, tile_rows=None):
    """cn_deflate_fused_kernel's streams of the selected planes.  planes: {plane: uint8 [h, w]}.  Returns
    ({plane: {(tile_row, tile_x): bytes}}, modes int [tiles, 8] (MODE_FIELDS), token counts)."""
    L = lib()
    sel = reg.planes
    arrs = [np.ascontiguousarray(planes[k], dtype=np.uint8) for k in sel]
    h, w = arrs[0].shape
    cls = np.asarray(reg.cls, np.uint8)
    hd = L.gcn10_ref_fused_new(reg.present.ctypes.data, int(reg.path == "tuned"), len(sel), cls.ctypes.data)
    assert hd, "no tuned code for this value set"
    out = np.zeros(len(sel) * STORED_BYTES, np.uint8)
    sizes = np.zeros(len(sel), np.uint32)
    mode = np.zeros(8, np.int32)
    ptrs = (C.c_void_p * len(sel))()
    tiles = {k: {} for k in sel}
    modes, ntok = [], []
    try:
        for (r, c) in _tiles_of(h, w):
            if tile_rows is not None and r not in tile_rows:
                continue
            for j, a in enumerate(arrs):
                ptrs[j] = a.ctypes.data + r * T * w + c * T
            n = L.gcn10_ref_fused_tile(hd, ptrs, w, min(T, w - c * T), min(T, h - r * T), out.ctypes.data,
                                       sizes.ctypes.data, mode.ctypes.data)
            for j, k in enumerate(sel):
                tiles[k][(r, c)] = out[j * STORED_BYTES: j * STORED_BYTES + int(sizes[j])].tobytes()
            modes.append(mode.copy())
            ntok.append(n)
    finally:
        L.gcn10_ref_fused_free(hd)
    return tiles, np.array(modes, np.int32).reshape(-1, 8), ntok


def plain_tiles(plane) -> dict:
    """deflate_tiles_kernel's streams of one plane: {(tile_row, tile_x): bytes}."""
    L = lib()
    a = np.ascontiguousarray(plane, dtype=np.uint8)
    h, w = a.shape
    out = np.zeros(STORED_BYTES, np.uint8)
    res = {}
    for (r, c) in _tiles_of(h, w):
        n = L.gcn10_ref_plain_tile(a.ctypes.data + r * T * w + c * T, w, min(T, w - c * T), min(T, h - r * T),
                                   out.ctypes.data)
        res[(r, c)] = out[:n].tobytes()
    return res


def expected_tiles(planes: dict, reg: Regime) -> dict:
    """The streams the library emits for these planes under this regime: {plane: {(tile_row, tile_x): bytes}}."""
    if reg.fused:
        return fused_tiles(planes, reg)[0]
    return {k: plain_tiles(planes[k]) for k in reg.planes}


def check_tiles(got: dict, planes: dict, reg: Regime, what=""):
    """Every stream of ``got`` ({plane: {(tile_row, tile_x): bytes}}) equals the reference's, byte for byte."""
    want = expected_tiles(planes, reg)
    assert sorted(got) == sorted(want), (what, sorted(got))
    for k in want:
        assert sorted(got[k]) == sorted(want[k]), (what, k)
        for key, z in want[k].items():
            g = got[k][key]
            if g != z:
                i = next((i for i in range(min(len(g), len(z))) if g[i] != z[i]), min(len(g), len(z)))
                raise AssertionError(f"{what} {reg.path}: plane {k} tile {key}: {len(g)} bytes, reference {len(z)}, "
                                     f"first difference at byte {i}")
