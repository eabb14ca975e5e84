#!/usr/bin/env python
"""LZW land cover on one GPU: a 36000 x 36000 worldcover block in 1024 x 1024 tiles, as libtiff LZW tiles (no
predictor, GDAL's COMPRESS=LZW) next to the same pixels as zlib-6 tiles.

Measured in one process, with the card's name and power limit read in the same run:
  - ms per block through gcn10_cuda_block_tiles_deflate with the next block prefetched, 9 and 18 planes, zlib and LZW
    input alternated block by block, and each block's decode kernel time (gcn10_cuda_last_inflate_ms);
  - the host-decode path for the same LZW file, which the program takes without GPU decoding: gh_tiff_read_window
    (16 threads) + gcn10_cuda_block_deflate, 9 and 18 planes alternated (after the GPU blocks: a host block in between
    would break the prefetch chain).
Prints one JSON line of medians; --out DIR writes it to DIR/r09_lzw.json."""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gcn10_b200 import capi, hostlib, synth, tiff_lzw  # noqa: E402
from tests import lookups  # noqa: E402
from tools.overview_bench import N, T_IN, gpu_info, tile_source  # noqa: E402


def lzw_source(ctx, esa):
    n = (N + T_IN - 1) // T_IN

    def tiles():
        for i in range(n * n):
            ty, tx = divmod(i, n)
            t = np.zeros((T_IN, T_IN), dtype=np.uint8)
            part = esa[ty * T_IN:(ty + 1) * T_IN, tx * T_IN:(tx + 1) * T_IN]
            t[:part.shape[0], :part.shape[1]] = part
            yield t
    streams = tiff_lzw.encode(tiles(), T_IN, T_IN, n * n)
    sizes = np.array([len(z) for z in streams], dtype=np.uint32)
    offsets = np.concatenate([[0], np.cumsum(sizes[:-1], dtype=np.uint64)]).astype(np.uint64)
    pin = capi.PinnedArray(ctx.lib, (int(sizes.sum()),))
    pin.array[:] = np.frombuffer(b"".join(streams), dtype=np.uint8)
    return pin, capi.TileSource(T_IN, T_IN, n, n, 0, 0, pin.array, offsets, sizes, compression=5)


def med(v):
    return round(statistics.median(v), 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per setting")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    info = gpu_info()
    ctx = capi.Context(0)
    ctx.set_luts(hostlib.load_lookup_tables(lookups.write_default_lookups(tempfile.mkdtemp())))
    gt, sgt, hsx, hsy = synth.block_geometry(-114.0, 42.0, N, N)
    hsg = synth.hsg_tile(hsx, hsy, 3234)
    esa = synth.esa_tile(N, N, 2234, device=torch.device("cuda:0")).cpu().numpy()
    t0 = time.perf_counter()
    pin_z, src_z = tile_source(ctx, esa)
    pin_l, src_l = lzw_source(ctx, esa)
    t_encode = time.perf_counter() - t0
    masks = {9: capi.MASK_DRAINED, 18: capi.MASK_ALL}

    # GPU decode: zlib and LZW alternated block by block, the next block always prefetched
    settings = [(codec, planes) for planes in (9, 18) for codec in ("zlib", "lzw")]
    src = {"zlib": src_z, "lzw": src_l}
    res = {f"{c}_{p}planes": dict(block_ms=[], decode_ms=[]) for c, p in settings}
    seq = [settings[i % len(settings)] for i in range(a.warmup + a.blocks * len(settings))]
    ctx.tiles_prefetch(src[seq[0][0]], N, N)
    for i, (codec, planes) in enumerate(seq):
        if i + 1 < len(seq):
            ctx.tiles_prefetch(src[seq[i + 1][0]], N, N)
        t0 = time.perf_counter()
        ctx.block_tiles_deflate(src[codec], N, N, gt, hsg, sgt, plane_mask=masks[planes], on_strip=lambda st: 0)
        dt = (time.perf_counter() - t0) * 1e3
        if i >= a.warmup:
            r = res[f"{codec}_{planes}planes"]
            r["block_ms"].append(dt)
            r["decode_ms"].append(ctx.last_inflate_ms())

    # host decode of the same LZW tiles: the path the program takes without GPU decoding
    fd, path = tempfile.mkstemp(suffix=".tif", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    os.close(fd)
    host = {f"host_lzw_{p}planes": dict(block_ms=[], read_ms=[]) for p in (9, 18)}
    try:
        tiff_lzw.write_file(path, esa, tile=T_IN)
        t = hostlib.Tiff(path)
        for i in range(2 + 2 * a.blocks):
            planes = (9, 18)[i % 2]
            t0 = time.perf_counter()
            raster = t.read(threads=16)
            t1 = time.perf_counter()
            ctx.block_deflate(raster, gt, hsg, sgt, plane_mask=masks[planes], on_strip=lambda st: 0)
            t2 = time.perf_counter()
            if i >= 2:
                r = host[f"host_lzw_{planes}planes"]
                r["block_ms"].append((t2 - t0) * 1e3)
                r["read_ms"].append((t1 - t0) * 1e3)
            del raster
        t.close()
    finally:
        os.unlink(path)

    out = {k: dict(block_ms_median=med(r["block_ms"]), block_ms_min=round(min(r["block_ms"]), 2),
                   block_ms_max=round(max(r["block_ms"]), 2), decode_kernel_ms_median=med(r["decode_ms"]),
                   blocks=len(r["block_ms"])) for k, r in res.items()}
    for k, r in host.items():
        out[k] = dict(block_ms_median=med(r["block_ms"]), read_window_ms_median=med(r["read_ms"]),
                      blocks=len(r["block_ms"]))
    line = dict(gpu=info, block=f"{N}x{N} worldcover, {T_IN}x{T_IN} tiles",
                input_mb=dict(zlib6=round(src_z.blob.size / 1e6, 1), lzw=round(src_l.blob.size / 1e6, 1)),
                host_encode_s=round(t_encode, 1), settings=out, gpu_after=gpu_info())
    ctx.close()
    pin_z.free()
    pin_l.free()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r09_lzw.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
