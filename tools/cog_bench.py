#!/usr/bin/env python
"""Cost of option "cog" on one GPU: 36000 x 36000 worldcover blocks through gcn10_cuda_block_tiles_deflate with the next
block prefetched, 9 and 18 planes, overviews automatic and "ordered" on (the program's setting), cog 0 and 1 alternated
block by block in one process.  Prints one JSON line: per setting the median ms per block, MB out per block (with cog
the 8 framing bytes per tile included), the time to the first strip in hand, and whether every strip left framed; the
card's name and power limit are read in the same run.  With --program it also times the gcn10 executable file -> file
(on /dev/shm when it exists) with --overviews against --cog.  --out DIR writes the line to DIR/cog_bench.json."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gcn10_b200 import capi, hostlib, synth  # noqa: E402
from tests import fixtures, lookups  # noqa: E402
from tools.overview_bench import N, gpu_info, tile_source  # noqa: E402


def run_blocks(a):
    import torch
    dev = torch.device("cuda:0")
    ctx = capi.Context(0)
    ctx.set_luts(hostlib.load_lookup_tables(lookups.write_default_lookups(tempfile.mkdtemp())))
    ctx.set_option("overviews", 16)
    ctx.set_option("ordered", 1)
    gt, sgt, hsx, hsy = synth.block_geometry(-114.0, 42.0, N, N)
    hsg = synth.hsg_tile(hsx, hsy, 3234)
    pins, srcs = [], []
    for b in range(a.distinct):
        esa = synth.esa_tile(N, N, 2234 + b, device=dev).cpu().numpy()
        pin, src = tile_source(ctx, esa)
        pins.append(pin)
        srcs.append(src)
        del esa
    settings = [(planes, cog) for planes in (9, 18) for cog in (0, 1)]
    res = {f"{p}planes_ovauto_cog{cog}": dict(block_ms=[], mb_out=[], first_strip_ms=[], framed=True)
           for p, cog in settings}
    seq = [srcs[i % len(srcs)] for i in range(a.blocks * len(settings) + a.warmup)]
    ctx.tiles_prefetch(seq[0], N, N)
    for i in range(len(seq)):
        planes, cog = settings[i % len(settings)]      # alternate the settings block by block
        ctx.set_option("cog", cog)
        if i + 1 < len(seq):
            ctx.tiles_prefetch(seq[i + 1], N, N)
        nb, t_first, framed = [0], [None], [True]

        def on_strip(st):
            nb[0] += st.blob_bytes
            framed[0] = framed[0] and st.framed == cog
            if t_first[0] is None:
                t_first[0] = time.perf_counter()
            return 0

        t0 = time.perf_counter()
        ctx.block_tiles_deflate(seq[i], N, N, gt, hsg, sgt, plane_mask=capi.MASK_DRAINED if planes == 9 else capi.MASK_ALL,
                                on_strip=on_strip)
        t1 = time.perf_counter()
        if i < a.warmup:
            continue
        r = res[f"{planes}planes_ovauto_cog{cog}"]
        r["block_ms"].append((t1 - t0) * 1e3)
        r["mb_out"].append(nb[0] / 1e6)
        r["first_strip_ms"].append((t_first[0] - t0) * 1e3)
        r["framed"] = r["framed"] and framed[0]
    ctx.set_option("cog", 0)
    out = {}
    for k, r in res.items():
        out[k] = dict(block_ms_median=round(statistics.median(r["block_ms"]), 2),
                      block_ms_min=round(min(r["block_ms"]), 2), block_ms_max=round(max(r["block_ms"]), 2),
                      mb_out_per_block=round(statistics.median(r["mb_out"]), 2),
                      first_strip_in_hand_ms=round(statistics.median(r["first_strip_ms"]), 2),
                      every_strip_framed_as_set=r["framed"], blocks=len(r["block_ms"]))
    ctx.close()
    for p in pins:
        p.free()
    return out


def run_program(a):
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    root = tempfile.mkdtemp(prefix="gcn10_cogprog_", dir=base)
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
            for flag in ("--overviews", "--cog"):
                cmd = [hostlib.EXE_PATH, "-c", os.path.join(root, "config.txt"), "-l", os.path.join(root, "blocks.txt"),
                       "-o", "--gpus", "1", flag]
                subprocess.run(["rm", "-rf", os.path.join(root, "cn_rasters_drained"),
                                os.path.join(root, "cn_rasters_undrained")])
                t0 = time.perf_counter()
                r = subprocess.run(cmd, cwd=root, capture_output=True, text=True)
                dt = time.perf_counter() - t0
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-2000:])
                mb = sum(os.path.getsize(os.path.join(dp, f)) for d in ("cn_rasters_drained", "cn_rasters_undrained")
                         for dp, _, fs in os.walk(os.path.join(root, d)) for f in fs) / 1e6
                out.setdefault(flag[2:], dict(wall_s=[], mb_written=mb))["wall_s"].append(round(dt, 3))
    finally:
        subprocess.run(["rm", "-rf", root])
    return dict(blocks=n, block_edge=s, dir=base or "tmp", runs=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per setting")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--distinct", type=int, default=2, help="different land-cover blocks cycled through")
    ap.add_argument("--program", action="store_true")
    ap.add_argument("--program-blocks", type=int, default=2)
    ap.add_argument("--program-size", type=int, default=36000)
    ap.add_argument("--program-reps", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    line = dict(gpu=gpu_info(), block=f"{N}x{N} worldcover", call="block_tiles_deflate + prefetch, overviews auto, ordered",
                settings=run_blocks(a))
    if a.program:
        line["program_file_to_file"] = run_program(a)
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "cog_bench.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
