#!/usr/bin/env python
"""Cost of one block option (overviews, stats, aggregate or cog) on one GPU: 36000 x 36000 worldcover blocks through
gcn10_cuda_block_tiles_deflate with the next block prefetched (the setting of bench.py's e2e leg), 9 and 18 planes, the
option's settings alternated block by block in one process.  What runs before a block decides how much of the
prefetched inflate overlaps it, so every setting of one alternation sequence follows the same rotation:

  overviews  overviews 0 and automatic, 9 and 18 planes, in one sequence;
  stats      stats off and on, one sequence per (fused, planes): each block behind one of the same size, on the fused
             path and with option "fused" 0 (the two-kernel path, where a histogram kernel reads every strip's planes
             once more);
  aggregate  aggregate off, 25 and 100, one sequence per plane count;
  cog        cog 0 and 1, 9 and 18 planes, in one sequence, with overviews automatic and "ordered" on (the program's
             setting).

Prints one JSON line: per setting the median, min and max ms per block and the option's own fields (MB out, the level
pass after the last full-resolution strip, the library's summed encoder time, tiles per level, mean tile bytes, the
time to the first strip in hand, whether every strip left framed as set); the card's name and power limit are read in
the same run.  With --program (overviews, cog) it also times the gcn10 executable file -> file (on /dev/shm when it
exists) with the option's two flag sets.  --out DIR writes the line to DIR/<option>_bench.json as well."""
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


def _median(v):
    return round(statistics.median(v), 2)


# per option: the call's description, the default of --blocks, the context options held for the whole run, the
# alternation sequences as (options set before the sequence's first prefetch, [(setting, planes, options set before
# each block)]), the per-setting fields as (field, per-block sample, summary), and the program's two flag sets
OPTIONS = {
    "overviews": dict(
        call="block_tiles_deflate + prefetch", blocks=6, held={},
        sequences=[({}, [(f"{p}planes_ov{'auto' if v else 0}", p, dict(overviews=v)) for p in (9, 18) for v in (0, 16)])],
        fields=[("mb_out_per_block", "mb_out", _median),
                ("tail_after_last_level0_strip_ms", "tail_ms", _median),
                ("encoder_ms_sum_over_strips", "kernel_ms", _median),
                ("tiles_per_plane_by_level", "tiles", lambda v: v[-1])],
        program=((), ("--overviews",))),
    "stats": dict(
        call="block_tiles_deflate + prefetch", blocks=8, held={},
        sequences=[(dict(fused=f), [(f"fused{f}_{p}planes_stats{v}", p, dict(stats=v)) for v in (0, 1)])
                   for f in (1, 0) for p in (9, 18)],
        fields=[("encoder_ms_sum_over_strips", "kernel_ms", _median)],
        program=None),
    "aggregate": dict(
        call="block_tiles_deflate + prefetch", blocks=8, held={},
        sequences=[({}, [(f"{p}planes_aggregate{v}", p, dict(aggregate=v)) for v in (0, 25, 100)]) for p in (9, 18)],
        fields=[("encoder_ms_sum_over_strips", "kernel_ms", _median),
                ("mean_tile_bytes", "mean_bytes", lambda v: int(statistics.median(v)))],
        program=None),
    "cog": dict(
        call="block_tiles_deflate + prefetch, overviews auto, ordered", blocks=8, held=dict(overviews=16, ordered=1),
        sequences=[({}, [(f"{p}planes_ovauto_cog{v}", p, dict(cog=v)) for p in (9, 18) for v in (0, 1)])],
        fields=[("mb_out_per_block", "mb_out", _median),
                ("first_strip_in_hand_ms", "first_ms", _median),
                ("every_strip_framed_as_set", "framed", all)],
        program=(("--overviews",), ("--cog",))),
}


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


def run_block(ctx, src, gt, hsg, sgt, planes, opts, want_kernel_ms):
    """One block; returns its sample: every per-strip counter the options report."""
    mask = capi.MASK_DRAINED if planes == 9 else capi.MASK_ALL
    s = dict(bytes=0, mean_bytes=0, tiles={}, t_first=None, t_last0=None, framed=True)

    def on_strip(st):
        now = time.perf_counter()
        s["bytes"] += st.blob_bytes
        if st.aggregate:
            s["mean_bytes"] += st.blob_bytes
        s["tiles"][st.level] = s["tiles"].get(st.level, 0) + st.n_tile_rows * st.tiles_x   # (of one plane)
        s["framed"] = s["framed"] and st.framed == opts.get("cog", 0)
        if s["t_first"] is None:
            s["t_first"] = now
        if st.level == 0 and (st.tile_row0 + st.n_tile_rows) * 256 >= N:
            s["t_last0"] = now
        return 0

    t0 = time.perf_counter()
    r = ctx.block_tiles_deflate(src, N, N, gt, hsg, sgt, plane_mask=mask, on_strip=on_strip)
    t1 = time.perf_counter()
    if opts.get("stats"):
        assert all(int(r["histograms"][p].sum()) == N * N for p in range(18) if mask >> p & 1)
    assert (s["mean_bytes"] > 0) == (opts.get("aggregate", 0) > 0)
    return dict(block_ms=(t1 - t0) * 1e3, mb_out=s["bytes"] / 1e6, tail_ms=(t1 - s["t_last0"]) * 1e3,
                first_ms=(s["t_first"] - t0) * 1e3, mean_bytes=s["mean_bytes"], framed=s["framed"],
                tiles={str(k): v for k, v in sorted(s["tiles"].items())},
                kernel_ms=ctx.last_kernel_ms() if want_kernel_ms else None)


def run_blocks(a, spec):
    import torch
    dev = torch.device("cuda:0")
    ctx = capi.Context(0)
    ctx.set_luts(hostlib.load_lookup_tables(lookups.write_default_lookups(tempfile.mkdtemp())))
    for k, v in spec["held"].items():
        ctx.set_option(k, v)
    gt, sgt, hsx, hsy = synth.block_geometry(-114.0, 42.0, N, N)
    hsg = synth.hsg_tile(hsx, hsy, 3234)
    pins, srcs = [], []
    for b in range(a.distinct):
        esa = synth.esa_tile(N, N, 2234 + b, device=dev).cpu().numpy()
        pin, src = tile_source(ctx, esa)
        pins.append(pin)
        srcs.append(src)
        del esa
    want_kernel_ms = any(key == "kernel_ms" for _, key, _ in spec["fields"])
    blocks = a.blocks or spec["blocks"]
    out = {}
    for seq_opts, settings in spec["sequences"]:
        for k, v in seq_opts.items():
            ctx.set_option(k, v)
        samples = {name: [] for name, _, _ in settings}
        seq = [srcs[i % len(srcs)] for i in range(blocks * len(settings) + a.warmup)]
        ctx.tiles_prefetch(seq[0], N, N)
        for i in range(len(seq)):
            name, planes, opts = settings[i % len(settings)]      # alternate the settings block by block
            for k, v in opts.items():
                ctx.set_option(k, v)
            if i + 1 < len(seq):
                ctx.tiles_prefetch(seq[i + 1], N, N)
            sample = run_block(ctx, seq[i], gt, hsg, sgt, planes, opts, want_kernel_ms and i >= a.warmup)
            if i >= a.warmup:
                samples[name].append(sample)
        for name, ss in samples.items():
            ms = [x["block_ms"] for x in ss]
            out[name] = dict(block_ms_median=_median(ms), block_ms_min=round(min(ms), 2), block_ms_max=round(max(ms), 2),
                             **{field: summary([x[key] for x in ss]) for field, key, summary in spec["fields"]},
                             blocks=len(ss))
    ctx.close()
    for p in pins:
        p.free()
    return out


def run_program(a, option, flags_a, flags_b):
    """The gcn10 executable file -> file on program_blocks blocks of program_size², alternately with each flag set;
    runs are keyed by the last flag without its dashes ("plain" for none)."""
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    root = tempfile.mkdtemp(prefix=f"gcn10_{option}_prog_", dir=base)
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
            for flags in (flags_a, flags_b):
                cmd = [hostlib.EXE_PATH, "-c", os.path.join(root, "config.txt"), "-l", os.path.join(root, "blocks.txt"),
                       "-o", "--gpus", "1", *flags]
                subprocess.run(["rm", "-rf", os.path.join(root, "cn_rasters_drained"),
                                os.path.join(root, "cn_rasters_undrained")])
                t0 = time.perf_counter()
                r = subprocess.run(cmd, cwd=root, capture_output=True, text=True)
                dt = time.perf_counter() - t0
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-2000:])
                mb = sum(os.path.getsize(os.path.join(dp, f)) for d in ("cn_rasters_drained", "cn_rasters_undrained")
                         for dp, _, fs in os.walk(os.path.join(root, d)) for f in fs) / 1e6
                key = flags[-1][2:] if flags else "plain"
                out.setdefault(key, dict(wall_s=[], mb_written=mb))["wall_s"].append(round(dt, 3))
    finally:
        subprocess.run(["rm", "-rf", root])
    return dict(blocks=n, block_edge=s, dir=base or "tmp", runs=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--option", required=True, choices=sorted(OPTIONS))
    ap.add_argument("--blocks", type=int, default=0, help="timed blocks per setting (default: overviews 6, others 8)")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--distinct", type=int, default=2, help="different land-cover blocks cycled through")
    ap.add_argument("--program", action="store_true", help="overviews and cog only")
    ap.add_argument("--program-blocks", type=int, default=2)
    ap.add_argument("--program-size", type=int, default=36000)
    ap.add_argument("--program-reps", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    spec = OPTIONS[a.option]
    if a.program and spec["program"] is None:
        ap.error(f"--program: option {a.option} has no program comparison")
    line = dict(gpu=gpu_info(), block=f"{N}x{N} worldcover", call=spec["call"], settings=run_blocks(a, spec))
    if a.program:
        line["program_file_to_file"] = run_program(a, a.option, *spec["program"])
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, f"{a.option}_bench.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
