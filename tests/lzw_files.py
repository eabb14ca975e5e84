"""LZW GeoTIFFs for the tests: a tiled DEFLATE GeoTIFF (hostlib.tiff_write) re-coded tile by tile with libtiff's LZW
encoder (gcn10_b200/tiff_lzw.py), georeferencing tags and tile grid kept.  Classic little-endian TIFF only."""
import struct
import zlib

import numpy as np

from gcn10_b200 import tiff_lzw


def recode_to_lzw(src, dst):
    b = bytearray(open(src, "rb").read())
    assert b[:4] == b"II*\x00", "classic little-endian TIFF expected"
    ifd = struct.unpack_from("<I", b, 4)[0]
    ent = {}
    for i in range(struct.unpack_from("<H", b, ifd)[0]):
        at = ifd + 2 + 12 * i
        tag, typ, cnt, val = struct.unpack_from("<HHII", b, at)
        ent[tag] = (at, typ, cnt, val)
    tw, th = ent[322][3], ent[323][3]
    n = ent[324][2]

    def array(tag):
        at, typ, cnt, val = ent[tag]
        assert typ == 4
        return list(struct.unpack_from(f"<{cnt}I", b, at + 8 if cnt == 1 else val))
    offs, counts = array(324), array(325)
    tiles = (np.frombuffer(zlib.decompress(bytes(b[o:o + c])), np.uint8).reshape(th, tw) for o, c in zip(offs, counts))
    streams = tiff_lzw.encode(tiles, tw, th, n)
    new_offs, new_counts = [], []
    for s in streams:
        if len(b) & 1:
            b.append(0)
        new_offs.append(len(b))
        new_counts.append(len(s))
        b += s
    for tag, vals in ((324, new_offs), (325, new_counts)):
        at = ent[tag][0]
        if n == 1:
            struct.pack_into("<I", b, at + 8, vals[0])
        else:
            struct.pack_into("<I", b, at + 8, len(b))
            b += struct.pack(f"<{n}I", *vals)
    struct.pack_into("<H", b, ent[259][0] + 8, 5)
    open(dst, "wb").write(bytes(b))
