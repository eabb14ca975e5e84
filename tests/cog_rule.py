"""The Cloud Optimized GeoTIFF layout rules, restated from GDAL's COG driver and its validate_cloud_optimized_geotiff.py,
checked on a file's bytes with `struct` alone (independently of the project's writer and reader):

1. classic little-endian TIFF; GDAL's ghost area at offset 8, exactly; IFD0 at the next even offset;
2. IFD0, then the overview IFDs from the largest to the smallest, chained, and every array any IFD points to (tile
   tables, GeoTIFF tags, GDAL_METADATA) before the first tile byte;
3. the smallest level's tiles first, then each larger level, the full resolution last; within an IFD row-major order
   with strictly increasing offsets (padding between tiles allowed);
4. every tile framed: its byte count as a uint32 LE in the 4 bytes before it, its last 4 bytes repeated after it; the
   TileByteCounts do not include the framing.
"""
import struct

GHOST = ("LAYOUT=IFDS_BEFORE_DATA\n"
         "BLOCK_ORDER=ROW_MAJOR\n"
         "BLOCK_LEADER=SIZE_AS_UINT4\n"
         "BLOCK_TRAILER=LAST_4_BYTES_REPEATED\n"
         "KNOWN_INCOMPATIBLE_EDITION=NO\n ")
TYPE_SIZE = {1: 1, 2: 1, 3: 2, 4: 4, 5: 8, 6: 1, 7: 1, 8: 2, 9: 4, 10: 8, 11: 4, 12: 8, 16: 8, 17: 8, 18: 8}
_FMT = {3: "H", 4: "I", 16: "Q"}


def ghost_area():
    """The bytes at offset 8: the size line (the size computed, not written down) and the layout text."""
    return (f"GDAL_STRUCTURAL_METADATA_SIZE={len(GHOST):06d} bytes\n" + GHOST).encode()


def _ifd(data, off):
    """(entries {tag: (type, count, inline field bytes, extent or None)}, extent of the IFD, next IFD offset)."""
    n, = struct.unpack_from("<H", data, off)
    ents = {}
    for i in range(n):
        tag, typ, cnt = struct.unpack_from("<HHI", data, off + 2 + 12 * i)
        field = data[off + 2 + 12 * i + 8: off + 2 + 12 * i + 12]
        size = TYPE_SIZE[typ] * cnt
        ext = None
        if size > 4:
            at, = struct.unpack("<I", field)
            assert at + size <= len(data), f"tag {tag} points past the end of the file"
            ext = (at, at + size)
        ents[tag] = (typ, cnt, field, ext)
    nxt, = struct.unpack_from("<I", data, off + 2 + 12 * n)
    return ents, (off, off + 2 + 12 * n + 4), nxt


def _values(data, ent):
    typ, cnt, field, ext = ent
    raw = field if ext is None else data[ext[0]:ext[1]]
    return list(struct.unpack_from(f"<{cnt}{_FMT[typ]}", raw))


def check(path):
    """Asserts rules 1-4 on the file at `path`; returns [per IFD: dict(offset, w, h, offsets, counts)], IFD0 first."""
    with open(path, "rb") as f:
        data = f.read()
    # 1. header and ghost area
    assert data[:4] == b"II*\0", "not a classic little-endian TIFF"
    g = ghost_area()
    assert data[8:8 + len(g)] == g, "no GDAL ghost area at offset 8"
    ifd0, = struct.unpack_from("<I", data, 4)
    assert ifd0 == (8 + len(g) + 1) & ~1, f"IFD0 at {ifd0}, not right behind the ghost area"
    # 2. the IFD chain and everything it points to
    ifds, extents, off = [], [], ifd0
    while off:
        assert not ifds or off > ifds[-1]["offset"], "IFDs not in file order"
        ents, ext, nxt = _ifd(data, off)
        extents.append(ext)
        extents += [e[3] for e in ents.values() if e[3] is not None]
        w, h = _values(data, ents[256])[0], _values(data, ents[257])[0]
        assert _values(data, ents[322]) == [256] and _values(data, ents[323]) == [256], "tiles must be 256 x 256"
        ifds.append(dict(offset=off, w=w, h=h, offsets=_values(data, ents[324]), counts=_values(data, ents[325])))
        assert len(ifds[-1]["offsets"]) == ((w + 255) // 256) * ((h + 255) // 256)
        off = nxt
    for a, b in zip(ifds, ifds[1:]):
        assert b["w"] < a["w"] or b["h"] < a["h"], "overview IFDs not from the largest to the smallest"
    first_data = min(o for d in ifds for o in d["offsets"]) - 4
    header_end = max(e[1] for e in extents)
    assert header_end <= first_data, f"header region ends at {header_end}, after the first tile byte {first_data}"
    # 3. data order: smallest level first, full resolution last, row-major within each, 4. framing
    prev_end = header_end
    for d in reversed(ifds):
        for o, n in zip(d["offsets"], d["counts"]):
            assert n >= 4, "tile too short to carry a trailer"
            assert o - 4 >= prev_end, f"tile at {o} out of order or overlapping the previous one"
            lead, = struct.unpack_from("<I", data, o - 4)
            assert lead == n, f"tile at {o}: leader {lead} != byte count {n}"
            assert o + n + 4 <= len(data)
            assert data[o + n:o + n + 4] == data[o + n - 4:o + n], f"tile at {o}: trailer does not repeat its last 4 bytes"
            prev_end = o + n + 4
    return ifds
