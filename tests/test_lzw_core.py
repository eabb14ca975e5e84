"""CPU checks of the decode-lane half of the GPU LZW tile decoder (gcn10_b200/csrc/lzw_core.h).

GDAL reads an LZW GeoTIFF tile through libtiff's LZWDecode, so libtiff is the judge: the streams come from libtiff's
own encoder (gcn10_b200/tiff_lzw.py drives the copy Pillow bundles), and every output and every ok / error verdict is
compared with libtiff's reading of the same stream.  tests/harness/lzw_host.cpp compiles the header the CUDA kernel
includes and emulates the writer warp in scalar code.  The GPU kernel itself is checked in tests/test_gpu_lzw.py.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import pytest

from gcn10_b200 import synth, tiff_lzw

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "harness", "lzw_host.cpp")
GUARD = 64


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("lzw_harness") / "liblzw_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", "-o", out, SRC])
    lib = ctypes.CDLL(out)
    lib.gcn10_test_lzw.restype = ctypes.c_int
    lib.gcn10_test_lzw.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p,
                                   ctypes.c_uint32, ctypes.c_void_p]
    return lib


def run(lib, stream: bytes, out_len: int, misalign: int = 0):
    out = np.full(out_len + GUARD, 0xEE, dtype=np.uint8)
    stats = np.zeros(2, dtype=np.uint64)
    rc = lib.gcn10_test_lzw(stream, len(stream), misalign, out.ctypes.data, out_len, stats.ctypes.data)
    assert (out[out_len:] == 0xEE).all(), "harness wrote past the tile"
    assert rc >= 0, f"harness invariant broken ({rc})"
    return rc, out[:out_len], stats


def pack(codes):
    """MSB-first code packing: [(code, width), ...] -> bytes (a stream made code by code, for damaged cases)."""
    acc = nbits = 0
    buf = bytearray()
    for c, w in codes:
        acc = (acc << w) | c
        nbits += w
        while nbits >= 8:
            nbits -= 8
            buf.append((acc >> nbits) & 255)
        acc &= (1 << nbits) - 1
    if nbits:
        buf.append((acc << (8 - nbits)) & 255)
    return bytes(buf)


def tiles():
    rng = np.random.default_rng(11)
    return {
        "worldcover1024": np.asarray(synth.esa_tile(1024, 1024, 2234)),
        "coastal512": np.asarray(synth.esa_tile(512, 512, 77, profile="coastal")),
        "noise512": rng.integers(0, 256, (512, 512), dtype=np.uint8),          # table refills, every width step
        "flat1024": np.full((1024, 1024), 80, dtype=np.uint8),                  # strings up to the longest
        "stripes256": np.tile(np.arange(256, dtype=np.uint8), (256, 1)),
        "nonsquare1000x700": np.asarray(synth.esa_tile(1000, 700, 5)),
        "odd3x5": rng.integers(0, 4, (5, 3), dtype=np.uint8),
        "one1x1": np.array([[42]], dtype=np.uint8),
        "row4097x1": rng.integers(0, 2, (1, 4097), dtype=np.uint8),
    }


TILES = tiles()


@pytest.mark.parametrize("name", sorted(TILES))
def test_matches_libtiff(harness, name):
    a = TILES[name]
    h, w = a.shape
    stream = tiff_lzw.encode([a], w, h)[0]
    assert np.array_equal(tiff_lzw.decode(stream, w, h), a)
    rc, out, stats = run(harness, stream, a.size)
    assert rc == 0, f"lzw error {rc}"
    assert np.array_equal(out.reshape(h, w), a)
    assert stats[0] > 0


@pytest.mark.parametrize("misalign", range(16))
def test_every_alignment(harness, misalign):
    a = TILES["coastal512"]
    stream = tiff_lzw.encode([a], 512, 512)[0]
    rc, out, _ = run(harness, stream, a.size, misalign)
    assert rc == 0 and np.array_equal(out.reshape(512, 512), a)
    # the old-style signature sits in the first two bytes, which may straddle a ring word
    rc, _, _ = run(harness, bytes([0x00, 0x01, 0x00, 0x00, 0x40]), 4, misalign)
    assert rc == 11


def test_kwkwk_and_table_refill(harness):
    # a run makes KwKwK codes (the code being defined is used at once); noise makes libtiff's encoder emit Clear
    # codes at every table refill: both are in one stream here
    rng = np.random.default_rng(3)
    a = np.concatenate([np.full(70000, 9, np.uint8), rng.integers(0, 256, 60000, dtype=np.uint8),
                        np.full(5000, 200, np.uint8)]).reshape(1, -1)
    stream = tiff_lzw.encode([a], a.shape[1], 1)[0]
    rc, out, _ = run(harness, stream, a.size)
    assert rc == 0 and np.array_equal(out, a[0])
    kw = pack([(256, 9), (65, 9), (258, 9), (259, 9), (257, 9)])     # A, AA (KwKwK), AAA (KwKwK)
    assert tiff_lzw.decode(kw, 6, 1).tolist() == [[65] * 6]
    rc, out, _ = run(harness, kw, 6)
    assert rc == 0 and out.tolist() == [65] * 6


def verdicts_agree(harness, stream, w, h):
    want = tiff_lzw.decode(stream, w, h)
    rc, out, _ = run(harness, stream, w * h)
    if want is None:
        assert rc != 0, f"libtiff refuses the stream, the decoder returned ok ({len(stream)} bytes)"
    else:
        assert rc == 0, f"libtiff reads the stream, the decoder returned {rc} ({len(stream)} bytes)"
        assert np.array_equal(out.reshape(h, w), want)
    return rc


def test_truncated_at_every_byte(harness):
    rng = np.random.default_rng(5)
    a = rng.integers(0, 7, (40, 48), dtype=np.uint8)
    stream = tiff_lzw.encode([a], 48, 40)[0]
    codes = set()
    for n in range(len(stream) + 1):
        codes.add(verdicts_agree(harness, stream[:n], 48, 40))
    assert 0 in codes and 8 in codes          # the last bytes hold EOI only: the tile is full without them


def test_damaged_codes(harness):
    cases = {
        "no Clear first": (pack([(65, 9), (66, 9), (67, 9), (68, 9), (257, 9)]), 12),
        "EOI first": (pack([(257, 9)]), 9),
        "first code after Clear above 257": (pack([(256, 9), (258, 9), (66, 9), (257, 9)]), 12),
        "code beyond the next free entry": (pack([(256, 9), (65, 9), (259, 9), (257, 9)]), 12),
        "EOI before the tile is full": (pack([(256, 9), (65, 9), (66, 9), (257, 9)]), 9),
        "Clear, Clear, literal": (pack([(256, 9), (256, 9), (65, 9), (66, 9), (67, 9), (68, 9)]), 0),
        "codes after the tile is full": (pack([(256, 9), (65, 9), (66, 9), (67, 9), (68, 9), (300, 9), (5, 9)]), 0),
        "string cut at the end of the tile": (pack([(256, 9), (65, 9), (66, 9), (258, 9), (258, 9)]), 0),
        "old style (LSB first)": (bytes([0x00, 0x01, 0x00, 0x00]), 11),
        # far more input than one batch stages: Clear codes count toward a batch like any other code
        "3000 Clear codes, then ABCD": (pack([(256, 9)] * 3000 + [(65, 9), (66, 9), (67, 9), (68, 9), (257, 9)]), 0),
    }
    for name, (stream, want) in cases.items():
        rc = verdicts_agree(harness, stream, 2, 2)
        assert rc == want, f"{name}: status {rc}, expected {want}"


def test_table_without_clear(harness):
    # literal codes only, never a Clear: libtiff makes entries up to 5118 (its table has 1023 spare entries) and
    # refuses the code that would make the next one
    def stream(n):
        codes, free, width = [(256, 9), (1, 9)], 258, 9
        for i in range(n):
            codes.append((i & 1, width))
            free += 1
            if free >= (1 << width) - 1 and width < 12:
                width += 1
        return pack(codes), n + 1
    ok, n_ok = stream(4096 + 1023 - 258)
    assert verdicts_agree(harness, ok, n_ok, 1) == 0
    bad, n_bad = stream(4096 + 1023 - 258 + 1)
    assert verdicts_agree(harness, bad, n_bad, 1) == 12


def test_random_damage(harness):
    rng = np.random.default_rng(8)
    a = np.asarray(synth.esa_tile(64, 48, 9, patch=6))
    stream = bytearray(tiff_lzw.encode([a], 64, 48)[0])
    for _ in range(300):
        s = bytearray(stream)
        for _ in range(int(rng.integers(1, 4))):
            s[int(rng.integers(0, len(s)))] ^= 1 << int(rng.integers(0, 8))
        verdicts_agree(harness, bytes(s), 64, 48)
