#!/usr/bin/env python
"""Cost of option "aggregate" on one GPU: 36000 x 36000 worldcover blocks through gcn10_cuda_block_tiles_deflate with the
next block prefetched (the setting of bench.py's e2e leg), 9 and 18 planes, aggregate off, 25 and 100 alternated block by
block in one process (each block behind one of another setting, in a fixed rotation).  Prints one JSON line: per setting
the median ms per block, the library's summed encoder time and the bytes of the mean tiles; the card's name and power
limit are read in the same run.  --out DIR writes the line to DIR/aggregate_bench.json as well."""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gcn10_b200 import capi, hostlib, synth  # noqa: E402
from tests import lookups  # noqa: E402
from tools.overview_bench import N, gpu_info, tile_source  # noqa: E402

FACTORS = (0, 25, 100)


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
    out = {}
    for planes in (9, 18):
        mask = capi.MASK_DRAINED if planes == 9 else capi.MASK_ALL
        res = {f: dict(block_ms=[], kernel_ms=[], mean_bytes=[]) for f in FACTORS}
        seq = [srcs[i % len(srcs)] for i in range(a.blocks * len(FACTORS) + a.warmup)]
        ctx.tiles_prefetch(seq[0], N, N)
        for i in range(len(seq)):
            f = FACTORS[i % len(FACTORS)]
            ctx.set_option("aggregate", f)
            if i + 1 < len(seq):
                ctx.tiles_prefetch(seq[i + 1], N, N)
            mean_bytes = [0]

            def on_strip(st, mb=mean_bytes):
                if st.aggregate:
                    mb[0] += st.blob_bytes
                return 0

            t0 = time.perf_counter()
            ctx.block_tiles_deflate(seq[i], N, N, gt, hsg, sgt, plane_mask=mask, on_strip=on_strip)
            t1 = time.perf_counter()
            assert (mean_bytes[0] > 0) == (f > 0)
            if i < a.warmup:
                continue
            res[f]["block_ms"].append((t1 - t0) * 1e3)
            res[f]["kernel_ms"].append(ctx.last_kernel_ms())
            res[f]["mean_bytes"].append(mean_bytes[0])
        for f, r in res.items():
            out[f"{planes}planes_aggregate{f}"] = dict(
                block_ms_median=round(statistics.median(r["block_ms"]), 2), block_ms_min=round(min(r["block_ms"]), 2),
                block_ms_max=round(max(r["block_ms"]), 2),
                encoder_ms_sum_over_strips=round(statistics.median(r["kernel_ms"]), 2),
                mean_tile_bytes=int(statistics.median(r["mean_bytes"])), blocks=len(r["block_ms"]))
    ctx.set_option("aggregate", 0)
    ctx.close()
    for p in pins:
        p.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per setting")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--distinct", type=int, default=2, help="different land-cover blocks cycled through")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    line = dict(gpu=gpu_info(), block=f"{N}x{N} worldcover", call="block_tiles_deflate + prefetch",
                settings=run_blocks(a))
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "aggregate_bench.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
