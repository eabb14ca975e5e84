#!/usr/bin/env python
"""Cost of option "overviews" on one GPU: 36000 x 36000 worldcover blocks through gcn10_cuda_block_tiles_deflate with
the next block prefetched (the setting of bench.py's e2e leg), 9 and 18 planes, overviews 0 and automatic alternated
block by block in one process.  Prints one JSON line: per setting the median ms per block, MB out per block, the level
pass (host clock from the hand-over of the last full-resolution strip to the end of the call; and the growth of the
library's summed encoder time), and tiles per level; the card's name and power limit are read in the same run.
With --program it also times the gcn10 executable file -> file (on /dev/shm when it exists) with and without
--overviews.  --out DIR writes the line to DIR/overview_bench.json as well."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from gcn10_b200 import capi, hostlib, synth  # noqa: E402
from tests import fixtures, lookups  # noqa: E402

N = 36000
T_IN = 1024


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def tile_source(ctx, esa):
    tx_n = ty_n = (N + T_IN - 1) // T_IN

    def one(i):
        ty, tx = divmod(i, tx_n)
        t = np.zeros((T_IN, T_IN), dtype=np.uint8)
        part = esa[ty * T_IN:(ty + 1) * T_IN, tx * T_IN:(tx + 1) * T_IN]
        t[:part.shape[0], :part.shape[1]] = part
        return zlib.compress(t.tobytes(), 6)

    with ThreadPoolExecutor(16) as ex:
        streams = list(ex.map(one, range(tx_n * ty_n)))
    sizes = np.array([len(z) for z in streams], dtype=np.uint32)
    offsets = np.concatenate([[0], np.cumsum(sizes[:-1], dtype=np.uint64)]).astype(np.uint64)
    pin = capi.PinnedArray(ctx.lib, (int(sizes.sum()),))
    pin.array[:] = np.frombuffer(b"".join(streams), dtype=np.uint8)
    return pin, capi.TileSource(T_IN, T_IN, tx_n, ty_n, 0, 0, pin.array, offsets, sizes)


def run_blocks(a):
    import torch
    dev = torch.device("cuda:0")
    ctx = capi.Context(0)
    ctx.set_luts(hostlib.load_lookup_tables(lookups.write_default_lookups(tempfile.mkdtemp())))
    gt, sgt, hsx, hsy = synth.block_geometry(-114.0, 42.0, N, N)
    hsg = synth.hsg_tile(hsx, hsy, 3234)
    pins, srcs = [], []
    for b in range(a.distinct):
        esa = synth.esa_tile(N, N, 2234 + b, device=dev).cpu().numpy()
        pin, src = tile_source(ctx, esa)
        pins.append(pin)
        srcs.append(src)
        del esa
    settings = [(planes, ov) for planes in (9, 18) for ov in (0, 16)]
    res = {f"{p}planes_ov{'auto' if ov else 0}": dict(block_ms=[], mb_out=[], level_tail_ms=[], kernel_ms=[], tiles={})
           for p, ov in settings}
    seq = [srcs[i % len(srcs)] for i in range(a.blocks * len(settings) + a.warmup)]
    ctx.tiles_prefetch(seq[0], N, N)
    for i in range(len(seq)):
        planes, ov = settings[i % len(settings)]      # alternate the settings block by block
        ctx.set_option("overviews", ov)
        if i + 1 < len(seq):
            ctx.tiles_prefetch(seq[i + 1], N, N)
        nb, tiles, t_last0 = [0], {}, [None]

        def on_strip(st):
            nb[0] += st.blob_bytes
            tiles[st.level] = tiles.get(st.level, 0) + st.n_tile_rows * st.tiles_x
            if st.level == 0 and (st.tile_row0 + st.n_tile_rows) * 256 >= N:
                t_last0[0] = time.perf_counter()
            return 0

        t0 = time.perf_counter()
        ctx.block_tiles_deflate(seq[i], N, N, gt, hsg, sgt, plane_mask=capi.MASK_DRAINED if planes == 9 else capi.MASK_ALL,
                                on_strip=on_strip)
        t1 = time.perf_counter()
        if i < a.warmup:
            continue
        r = res[f"{planes}planes_ov{'auto' if ov else 0}"]
        r["block_ms"].append((t1 - t0) * 1e3)
        r["mb_out"].append(nb[0] / 1e6)
        r["level_tail_ms"].append((t1 - t_last0[0]) * 1e3)
        r["kernel_ms"].append(ctx.last_kernel_ms())
        r["tiles"] = {str(k): v for k, v in sorted(tiles.items())}              # (a strip's tiles of one plane)
    ctx.set_option("overviews", 0)
    out = {}
    for k, r in res.items():
        out[k] = dict(block_ms_median=round(statistics.median(r["block_ms"]), 2),
                      block_ms_min=round(min(r["block_ms"]), 2), block_ms_max=round(max(r["block_ms"]), 2),
                      mb_out_per_block=round(statistics.median(r["mb_out"]), 2),
                      tail_after_last_level0_strip_ms=round(statistics.median(r["level_tail_ms"]), 2),
                      encoder_ms_sum_over_strips=round(statistics.median(r["kernel_ms"]), 2),
                      tiles_per_plane_by_level=r["tiles"], blocks=len(r["block_ms"]))
    ctx.close()
    for p in pins:
        p.free()
    return out


def run_program(a):
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    root = tempfile.mkdtemp(prefix="gcn10_ovprog_", dir=base)
    px, hpx, n, s = 1.0 / 12000.0, 1.0 / 480.0, a.program_blocks, a.program_size
    import torch
    esa = synth.esa_tile(s * n, s, 2234, device=torch.device("cuda:0")).cpu().numpy()
    hsg = synth.hsg_tile(s * n // 25 + 2, s // 25 + 2, 3234)
    hostlib.tiff_write(os.path.join(root, "esa.tif"), esa, (-114.0, px, 0, 42.0, 0, -px), threads=16)
    hostlib.tiff_write(os.path.join(root, "hsg.tif"), hsg, (-114.0, hpx, 0, 42.0, 0, -hpx))
    del esa
    blocks = [(100 + i, -114.0 + i * s * px, 42.0 - (s - 0.25) * px, -114.0 + ((i + 1) * s - 0.25) * px, 42.0)
              for i in range(n)]
    fixtures.write_block_shapefile(os.path.join(root, "blocks.shp"), blocks)
    lookups.write_default_lookups(os.path.join(root, "lookups"))
    fixtures.write_config(os.path.join(root, "config.txt"), os.path.join(root, "esa.tif"), os.path.join(root, "hsg.tif"),
                          os.path.join(root, "blocks.shp"), os.path.join(root, "lookups"), os.path.join(root, "logs"))
    with open(os.path.join(root, "blocks.txt"), "w") as f:
        f.write("\n".join(str(b[0]) for b in blocks) + "\n")
    out = {}
    try:
        for rep in range(a.program_reps):
            for ov in (False, True):
                cmd = [hostlib.EXE_PATH, "-c", os.path.join(root, "config.txt"), "-l", os.path.join(root, "blocks.txt"),
                       "-o", "--gpus", "1"] + (["--overviews"] if ov else [])
                subprocess.run(["rm", "-rf", os.path.join(root, "cn_rasters_drained"),
                                os.path.join(root, "cn_rasters_undrained")])
                t0 = time.perf_counter()
                r = subprocess.run(cmd, cwd=root, capture_output=True, text=True)
                dt = time.perf_counter() - t0
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-2000:])
                mb = sum(os.path.getsize(os.path.join(dp, f)) for d in ("cn_rasters_drained", "cn_rasters_undrained")
                         for dp, _, fs in os.walk(os.path.join(root, d)) for f in fs) / 1e6
                key = "overviews" if ov else "plain"
                out.setdefault(key, dict(wall_s=[], mb_written=mb))["wall_s"].append(round(dt, 3))
    finally:
        subprocess.run(["rm", "-rf", root])
    return dict(blocks=n, block_edge=s, dir=base or "tmp", runs=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=6, help="timed blocks per setting")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--distinct", type=int, default=2, help="different land-cover blocks cycled through")
    ap.add_argument("--program", action="store_true")
    ap.add_argument("--program-blocks", type=int, default=2)
    ap.add_argument("--program-size", type=int, default=36000)
    ap.add_argument("--program-reps", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    line = dict(gpu=gpu_info(), block=f"{N}x{N} worldcover", call="block_tiles_deflate + prefetch", settings=run_blocks(a))
    if a.program:
        line["program_file_to_file"] = run_program(a)
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "overview_bench.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
