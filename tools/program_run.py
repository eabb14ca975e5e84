#!/usr/bin/env python
"""Drive the gcn10 executable on synthetic rasters: builds a small 'world' (one land-cover GeoTIFF, one
HSG GeoTIFF, a block shapefile, config, lookups), runs the program on N GPUs and reports wall time,
end-to-end Mpx/s and which worker processed which block (from the per-worker logs)."""
import argparse
import glob
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gcn10_b200 import hostlib, synth
from tests import lookups  # noqa: E402
from tests import fixtures  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--size", type=int, default=9000, help="block edge in pixels")
    ap.add_argument("--io-threads", type=int, default=0)
    ap.add_argument("--workers-per-gpu", type=int, default=1)
    ap.add_argument("--keep", action="store_true")
    ap.add_argument("--host-inflate", action="store_true", help="decode the land cover on the host (zlib threads)")
    a = ap.parse_args()
    px = 1.0 / 12000.0
    hpx = 1.0 / 480.0
    n, s = a.blocks, a.size
    root = tempfile.mkdtemp(prefix="gcn10_world_")
    W, H = s * n, s                                     # blocks side by side in one row
    t0 = time.time()
    try:                                                # full-size tiles take minutes in numpy: use the GPU when there is one
        import torch
        esa = synth.esa_tile(W, H, 2234, device=torch.device("cuda:0")).cpu().numpy() if torch.cuda.is_available() \
            else synth.esa_tile(W, H, 2234)
    except ImportError:
        esa = synth.esa_tile(W, H, 2234)
    hsg = synth.hsg_tile(W // 25 + 2, H // 25 + 2, 3234)
    hostlib.tiff_write(os.path.join(root, "esa.tif"), esa, (-114.0, px, 0, 42.0, 0, -px), threads=16)
    hostlib.tiff_write(os.path.join(root, "hsg.tif"), hsg, (-114.0, hpx, 0, 42.0, 0, -hpx))
    blocks = [(100 + i, -114.0 + i * s * px, 42.0 - (s - 0.25) * px, -114.0 + ((i + 1) * s - 0.25) * px, 42.0)
              for i in range(n)]
    fixtures.write_block_shapefile(os.path.join(root, "blocks.shp"), blocks)
    lookups.write_default_lookups(os.path.join(root, "lookups"))
    fixtures.write_config(os.path.join(root, "config.txt"), os.path.join(root, "esa.tif"), os.path.join(root, "hsg.tif"),
                          os.path.join(root, "blocks.shp"), os.path.join(root, "lookups"), os.path.join(root, "logs"))
    with open(os.path.join(root, "blocks.txt"), "w") as f:
        f.write("\n".join(str(b[0]) for b in blocks) + "\n")
    print(f"world built in {time.time() - t0:.1f} s: {n} blocks of {s}x{s}")
    cmd = [hostlib.EXE_PATH, "-c", os.path.join(root, "config.txt"), "-l", os.path.join(root, "blocks.txt"), "-o",
           "--gpus", str(a.gpus)]
    if a.io_threads:
        cmd += ["--io-threads", str(a.io_threads)]
    if a.workers_per_gpu > 1:
        cmd += ["--workers-per-gpu", str(a.workers_per_gpu)]
    t0 = time.time()
    env = dict(os.environ, GCN10_HOST_INFLATE="1" if a.host_inflate else "0")
    r = subprocess.run(cmd, cwd=root, capture_output=True, text=True, env=env)
    dt = time.time() - t0
    print(f"gcn10 rc={r.returncode} wall {dt:.2f} s -> {n * s * s / dt / 1e6:.1f} Mpx/s end to end "
          f"({18 * n} GeoTIFFs, {sum(os.path.getsize(p) for p in glob.glob(root + '/cn_rasters_*/*.tif')) / 1e6:.1f} MB)")
    for lp in sorted(glob.glob(os.path.join(root, "logs", "rank_*.log"))):
        txt = open(lp).read()
        ids = re.findall(r"processing block (\d+)", txt)
        per = re.findall(r"block (\d+): .* in ([\d.]+) s \(([\d.]+) Mpx/s; decode ([\d.]+) s, gpu\+copies ([\d.]+) s; (\w+) deflate\)", txt)
        print(os.path.basename(lp), "blocks", ids, per[:3])
    if r.returncode != 0:
        print(r.stderr[-2000:])
    if not a.keep:
        subprocess.run(["rm", "-rf", root])
    return r.returncode


if __name__ == "__main__":
    sys.exit(main())
