"""Fixture writers for the host-program tests: a block shapefile (.shp/.shx/.dbf, PolygonZ records with
an integer ID attribute, like /root/reference/blocks/esa_extent_blocks.*) and GeoTIFF rasters; and the runner of the
gcn10 executable on such a world."""
import os
import struct
import subprocess

import numpy as np

from gcn10_b200 import hostlib


def run_program(root, config="config.txt", *extra, host_inflate=False):
    """gcn10 on one GPU with the config <root>/<config> and the block list <root>/blocks.txt, run from root; the land
    cover is decoded on the host with host_inflate (GCN10_HOST_INFLATE=1).  Returns the CompletedProcess."""
    assert os.path.exists(hostlib.EXE_PATH), "gcn10 executable not built (make host)"
    env = dict(os.environ, GCN10_HOST_INFLATE="1" if host_inflate else "0")
    return subprocess.run([hostlib.EXE_PATH, "-c", os.path.join(root, config), "-l", os.path.join(root, "blocks.txt"),
                           "--gpus", "1", "--io-threads", "4", *extra], cwd=str(root), capture_output=True, text=True,
                          timeout=300, env=env)


def write_block_shapefile(path_shp, blocks):
    """blocks: list of (id, minx, miny, maxx, maxy).  Writes PolygonZ (type 15) records."""
    recs = []
    for bid, x0, y0, x1, y1 in blocks:
        pts = [(x0, y0), (x0, y1), (x1, y1), (x1, y0), (x0, y0)]
        body = struct.pack("<i4d2i", 15, x0, y0, x1, y1, 1, 5) + struct.pack("<i", 0)
        body += b"".join(struct.pack("<2d", *p) for p in pts)
        body += struct.pack("<2d", 0.0, 0.0) + struct.pack("<5d", *([0.0] * 5))      # Z range + Z
        body += struct.pack("<2d", 0.0, 0.0) + struct.pack("<5d", *([0.0] * 5))      # M range + M
        recs.append(body)
    xs0 = min(b[1] for b in blocks); ys0 = min(b[2] for b in blocks)
    xs1 = max(b[3] for b in blocks); ys1 = max(b[4] for b in blocks)
    total = 100 + sum(8 + len(r) for r in recs)

    def header(length_bytes):
        return (struct.pack(">i5i", 9994, 0, 0, 0, 0, 0) + struct.pack(">i", length_bytes // 2) +
                struct.pack("<2i", 1000, 15) + struct.pack("<8d", xs0, ys0, xs1, ys1, 0, 0, 0, 0))

    with open(path_shp, "wb") as f:
        f.write(header(total))
        for i, r in enumerate(recs):
            f.write(struct.pack(">2i", i + 1, len(r) // 2) + r)
    base = path_shp[:-4]
    with open(base + ".shx", "wb") as f:
        f.write(header(100 + 8 * len(recs)))
        off = 100
        for r in recs:
            f.write(struct.pack(">2i", off // 2, len(r) // 2))
            off += 8 + len(r)
    # dBASE III: fields fid N(20), ID N(10) -- same layout as the reference's .dbf
    fields = [(b"fid", 20), (b"ID", 10)]
    hlen = 32 + 32 * len(fields) + 1
    rlen = 1 + sum(n for _, n in fields)
    with open(base + ".dbf", "wb") as f:
        f.write(struct.pack("<4BIHH20x", 3, 124, 8, 25, len(blocks), hlen, rlen))
        for name, n in fields:
            f.write(name.ljust(11, b"\0") + b"N" + b"\0" * 4 + bytes([n, 0]) + b"\0" * 14)
        f.write(b"\r")
        for i, b in enumerate(blocks):
            f.write(b" " + str(i + 1).rjust(20).encode() + str(b[0]).rjust(10).encode())
        f.write(b"\x1a")
    return path_shp


def write_config(path, esa, hsg, shp, lookups, log_dir):
    with open(path, "w") as f:
        f.write("# gcn10 test config\n\n"
                f"hysogs_data_path = {hsg}\n"
                f"esa_data_path={esa}\n"
                f"  blocks_shp_path=  {shp}  \n"
                f"lookup_table_path={lookups}\n"
                f"log_dir={log_dir}\n")
    return path


def write_vrt(path, w, h, gt, sources, kind="ComplexSource", nodata=0, remote_prefix=None):
    """A VRT with the structure of /root/reference/landcover/esa_worldcover_2021.vrt: one Byte band, one
    <ComplexSource> per file with SrcRect / DstRect, NODATA 0.  sources: (filename, src_x, src_y, dst_x, dst_y, w, h)."""
    gts = ", ".join(f"{v:.16e}" for v in gt)
    out = [f'<VRTDataset rasterXSize="{w}" rasterYSize="{h}">',
           '  <SRS dataAxisToSRSAxisMapping="2,1">GEOGCS["WGS 84",AUTHORITY["EPSG","4326"]]</SRS>',
           f'  <GeoTransform> {gts}</GeoTransform>',
           '  <VRTRasterBand dataType="Byte" band="1">',
           f'    <NoDataValue>{nodata}</NoDataValue>',
           '    <ColorInterp>Palette</ColorInterp>']
    for name, sx, sy, dx, dy, sw, sh in sources:
        fn = (remote_prefix + os.path.basename(name)) if remote_prefix else name
        rel = 0 if (remote_prefix or os.path.isabs(name)) else 1
        out += [f'    <{kind} resampling="nearest">',
                f'      <SourceFilename relativeToVRT="{rel}">{fn.replace("&", "&amp;")}</SourceFilename>',
                '      <SourceBand>1</SourceBand>',
                f'      <SourceProperties RasterXSize="{sw}" RasterYSize="{sh}" DataType="Byte" BlockXSize="256" BlockYSize="256" />',
                f'      <SrcRect xOff="{sx}" yOff="{sy}" xSize="{sw}" ySize="{sh}" />',
                f'      <DstRect xOff="{dx}" yOff="{dy}" xSize="{sw}" ySize="{sh}" />',
                f'      <NODATA>{nodata}</NODATA>',
                f'    </{kind}>']
    out += ['  </VRTRasterBand>', '  <OverviewList resampling="nearest">2 4</OverviewList>', '</VRTDataset>']
    with open(path, "w") as f:
        f.write("\n".join(out) + "\n")
    return path
