#!/usr/bin/env python
"""bench.py -- GCN10 Curve Number hot path on B200: CN Gpixel/s (9 LUT variants).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes, after the K timed kernel-resident steps, what the last of them computed: the nine
drained Curve Number planes of rank 0, as float32 DIR/cn_drained.npy [9, n] at n seeded pixel positions
(DIR/cn_drained_index.npy, float64 flat indices y * W + x; every pixel when the tile has at most 2**20).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.

One "step" = one pass of the hot path over one synthetic 3x3 degree block: a 36000 x 36000 uint8
WorldCover-like tile plus its 1440 x 1440 HSG window, all nine lookup variants (p/f/g x ARC
I/II/III) of one drainage condition written in a single fused pass (BASELINE.json configs[1]).
1 pixel = one land-cover pixel for which all nine CN values were written.

  value      whole-job Gpixel/s with inputs resident in HBM (device-side entry point
             gcn10_cuda_block_device), CUDA events on the launching stream, max over ranks
  e2e        the same metric through the host-buffer C-ABI call the gcn10 host program makes,
             gcn10_cuda_block_deflate: pinned host rasters in, H2D + Curve Number kernel + GPU DEFLATE of
             the 256x256 GeoTIFF tiles (the encode step of the reference's save_raster) + D2H of the
             compressed tiles inside the timed region; e2e.raw_planes = gcn10_cuda_block (nine raw
             planes back over PCIe) for comparison
  roofline   HBM: algorithmic bytes (W*H*(1+9) + HSG window) / mean step duration vs the measured
             copy peak in MEASURED_PEAKS.json
  cpu_baseline  the reference's own object code (oracle/_ref) on one host core, bounded sample

`--impl reference` times the reference's CPU implementation (oracle/_ref = src/cn.c + src/raster.c
compiled unmodified; falls back to the C restatement if that library is absent) on all host cores,
one independent process per core exactly like the reference's MPI ranks (main.c:171), each step a
bounded row-slab sample of the same tile.

Multi-GPU: blocks are independent (no collective on the data path); every rank runs its own tile
per step (weak scaling), value = N * pixels / max-over-ranks time.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TILE = 36000
HSG = 1440
NVAR = 9
METRIC = "CN Gpixel/s (9 LUT variants)"
UNIT = "Gpixel/s"
BLOCK_ID = 2234                 # first id of /root/reference/src/test/blocks.txt: NW corner (-114, 42)
LON0, LAT0 = -114.0, 42.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the kernel-resident leg (the headline value)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--profile", default="worldcover", choices=["worldcover", "random", "coastal"])
    ap.add_argument("--tile", type=int, default=TILE, help="tile edge in pixels (default 36000)")
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed end-to-end steps (default min(steps, 5))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-rows", type=int, default=1800)
    ap.add_argument("--ref-sample-rows", type=int, default=600)
    ap.add_argument("--ship", type=int, default=None, choices=[0, 1], help="override the library's strip hand-over path")
    ap.add_argument("--queue-blocks", type=int, default=64, help="blocks of the e2e.queue64 leg (0 = skip)")
    ap.add_argument("--program-blocks", type=int, default=4, help="blocks of the e2e.program leg per GPU (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's output planes to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm keeps no outputs)")
    return args


DUMP_SAMPLE = 1 << 20           # pixels per plane in --dump-outputs: 9 x 4 MB of float32 + 8 MB of indices
DUMP_SEED = 20240601


def dump_outputs(directory, d_out, w, h):
    """The drained planes of the last timed step at DUMP_SAMPLE seeded pixel positions (all pixels of a small tile)."""
    import numpy as np
    import torch
    n = w * h
    if n <= DUMP_SAMPLE:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, DUMP_SAMPLE, dtype=np.int64))
    vals = d_out.view(NVAR, n)[:, torch.from_numpy(idx).to(d_out.device)]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "cn_drained.npy"), vals.to(torch.float32).cpu().numpy())
    np.save(os.path.join(directory, "cn_drained_index.npy"), idx.astype(np.float64))


def workload_config(args, extra=None):
    t = args.tile
    hs = (t * HSG + TILE - 1) // TILE
    cfg = {
        "workload": (f"BASELINE configs[1]: synthetic 3x3 deg WorldCover tile {t}x{t} uint8 + {hs}x{hs} "
                     f"250 m HSG window, all 9 lookups (f/g/p x ARC I/II/III, drained) in one pass"),
        "tile": [t, t], "hsg_window": [hs, hs], "planes": NVAR, "profile": args.profile,
        "block_id": BLOCK_ID,
        "l2": "per-step working set (1.3 GB in + 11.7 GB out) >> 126 MB L2, so no flush between iterations",
        "parallelism": "one block per GPU per step, no collective (blocks are independent)",
    }
    if extra:
        cfg.update(extra)
    return cfg


# --------------------------------------------------------------------------- CPU reference legs


def _cpu_sample_inputs(tile, rows, profile, seed):
    """A bounded sample of the benchmark workload: the first `rows` rows of the tile (full width)."""
    from gcn10_b200 import synth
    gt, sgt, hsx, hsy = synth.block_geometry(LON0, LAT0, tile, rows)
    esa = synth.esa_tile(tile, rows, seed, profile)
    hsg = synth.hsg_tile(hsx, hsy, seed + 1000, profile)
    return esa, gt, hsg, sgt


_INPUT_CACHE = {}


def _ref_worker(task):
    """One 'MPI rank': run process_block() of the reference object code on its own slab."""
    tile, rows, profile, seed, lookup_dir, reps = task
    from oracle import oracle as O
    key = (tile, rows, profile, seed)
    if key not in _INPUT_CACHE:                 # pool processes keep their slab between steps
        _INPUT_CACHE.clear()
        _INPUT_CACHE[key] = _cpu_sample_inputs(tile, rows, profile, seed)
    esa, gt, hsg, sgt = _INPUT_CACHE[key]
    # far edges pulled in by 1/4 pixel so that ceil() in raster.c:129-130 yields exactly tile x rows
    bbox = (gt[0], gt[3] + (rows - 0.25) * gt[5], gt[0] + (tile - 0.25) * gt[1], gt[3])
    out = []
    if O.Ref.available():
        ref = O.Ref()
        for _ in range(reps):
            r = ref.run_block(esa, gt, hsg, sgt, bbox, lookup_dir, block_id=BLOCK_ID, keep=False)
            if r["nplanes"] != 18 or (r["w"], r["h"]) != (tile, rows):
                raise RuntimeError(f"reference run failed: {r['nplanes']} planes, {r['w']}x{r['h']}\n{r['log']}")
            out.append((r["times"][8], r["times"][17]))      # time to the 9th / 18th saved plane
        kind = "reference"
    else:
        port = O.Port()
        tables = port.load_tables(lookup_dir)
        for _ in range(reps):
            t0 = time.perf_counter()
            port.block_rows(esa, gt, hsg, sgt, tables)
            t = time.perf_counter() - t0
            out.append((t / 2, t))
        kind = "port"
    return kind, out


def cpu_baseline_one_core(args, lookup_dir):
    rows = min(args.cpu_sample_rows, args.tile)
    kind, times = _ref_worker((args.tile, rows, args.profile, BLOCK_ID, lookup_dir, 1))
    t9, t18 = times[0]
    px = args.tile * rows
    return {
        "value": px / t9 / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
        "sample": (f"first {rows} rows x {args.tile} px of the same tile ({px / 1e6:.1f} Mpx): "
                   f"process_block() time to the 9th saved plane {t9:.2f} s (all 18 planes: {t18:.2f} s)"),
        "value_18_planes": px / t18 / 1e9,
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    from tests import lookups
    lookup_dir = lookups.write_default_lookups(tempfile.mkdtemp(prefix="gcn10_lookups_"))
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    rows = min(args.ref_sample_rows, args.tile)
    px_per_proc = args.tile * rows
    # the reference's object code is loaded here, in the process the driver watches, before the ranks fork from it
    from oracle import oracle as O
    ref_loaded = None
    if O.Ref.available():
        ref_loaded = O.Ref()
    ctx = mp.get_context("fork")
    step_times = []
    kind = "reference"
    with ctx.Pool(cores) as pool:
        def one_step():
            nonlocal kind
            tasks = [(args.tile, rows, args.profile, BLOCK_ID + i, lookup_dir, 1) for i in range(cores)]
            t0 = time.perf_counter()
            res = pool.map(_ref_worker, tasks)
            wall = time.perf_counter() - t0
            kind = res[0][0]
            t9 = max(r[1][0][0] for r in res)       # slowest rank, time to its 9th plane
            t18 = max(r[1][0][1] for r in res)
            return t9, t18, wall
        for _ in range(args.warmup):
            one_step()
        for _ in range(args.steps):
            step_times.append(one_step())
    t9 = sum(s[0] for s in step_times) / len(step_times)
    t18 = sum(s[1] for s in step_times) / len(step_times)
    value = cores * px_per_proc / t9 / 1e9
    sample = (f"{cores} independent processes (= MPI ranks, main.c:171), each process_block() on a "
              f"{rows}-row x {args.tile}-px slab of the tile ({px_per_proc / 1e6:.1f} Mpx); rate = pixels / time to "
              f"the 9th saved plane of the slowest rank ({t9:.2f} s; all 18 planes {t18:.2f} s)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t9 * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args),
        "sample_rows_per_process": rows, "processes": cores,
        "reference_library": O.REF_SO if ref_loaded is not None else None,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print_json(line)
    return 0


# --------------------------------------------------------------------------- clocks sampler


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- our arm


def run_ours(args):
    import numpy as np
    import torch

    from gcn10_b200 import capi, synth
    from tests import lookups

    from gcn10_b200 import dist as gdist
    rank, local_rank, world = gdist.env_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the Curve Number path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    group = gdist.Group("nccl", device=dev)      # barrier + max-over-ranks only; no data-path collective
    barrier = group.barrier
    max_over_ranks = group.max

    # lookup tables through the product's own CSV reader when the host library is built,
    # else parsed here with the same rules (cn.c:13-85)
    lookup_dir = lookups.write_default_lookups(tempfile.mkdtemp(prefix="gcn10_lookups_"))
    tables = load_tables_host(lookup_dir)

    ctx = capi.Context(local_rank)
    ctx.set_luts(tables)
    # strip hand-over: the copy engine (size read-back + cudaMemcpyAsync) is faster when a GPU has the host link to
    # itself; from four GPUs on one host fabric the ship kernel's posted writes are (DESIGN.md 4.6, 6)
    ship = args.ship if args.ship is not None else (1 if world >= 4 else 0)
    ctx.set_option("ship", ship)
    # host thread -> NUMA node of this GPU, before any pinned allocation (matters at N > 1: see DESIGN.md 6)
    numa_node = ctx.lib.gcn10_cuda_bind_host_thread(local_rank)

    w = h = args.tile
    # every rank (GPU worker) takes its own block of the id list, round-robin like main.c:171
    seed = gdist.shard_blocks([BLOCK_ID + i for i in range(world)], rank, world)[0]
    gt, sgt, hsx, hsy = synth.block_geometry(LON0, LAT0, w, h)
    d_esa = synth.esa_tile(w, h, seed, args.profile, device=dev)
    hsg_np = synth.hsg_tile(hsx, hsy, seed + 1000, args.profile)
    d_hsg = torch.from_numpy(hsg_np).to(dev)
    d_out = torch.empty((NVAR, h, w), dtype=torch.uint8, device=dev)
    out_ptrs = [d_out[k].data_ptr() for k in range(NVAR)] + [0] * 9
    # a dedicated (non-default) torch stream: the library launches on the stream handle it is given,
    # and the CUDA events below are recorded on that same stream
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def step():
        ctx.block_device(d_esa.data_ptr(), w, h, w, gt, d_hsg.data_ptr(), hsx, hsy, hsx, sgt,
                         capi.MASK_DRAINED, out_ptrs, w, stream=stream.cuda_stream)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- kernel-resident timing: K steps, per-step events for the roofline average
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    l0 = ctx.launch_count()
    barrier()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record(stream)
    for a, b in ev:
        a.record(stream)
        step()
        b.record(stream)
    t_end.record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    total_ms = max_over_ranks(t_start.elapsed_time(t_end))
    step_ms = sorted(a.elapsed_time(b) for a, b in ev)
    mean_step_ms = sum(step_ms) / len(step_ms)
    px = float(w) * h
    value = world * px * args.steps / (total_ms * 1e-3) / 1e9
    # before the legs below write into d_out
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out, w, h)

    # ---- the drop-in pass: both drainage conditions, all 18 rasters of a block in one launch (19 B/px)
    all18 = None
    try:
        d_out18 = torch.empty((9, h, w), dtype=torch.uint8, device=dev)       # undrained planes; drained reuse d_out
        ptrs18 = [d_out[k].data_ptr() for k in range(NVAR)] + [d_out18[k].data_ptr() for k in range(9)]

        def step18():
            ctx.block_device(d_esa.data_ptr(), w, h, w, gt, d_hsg.data_ptr(), hsx, hsy, hsx, sgt,
                             capi.MASK_ALL, ptrs18, w, stream=stream.cuda_stream)
        for _ in range(3):
            step18()
        barrier()
        n18 = max(3, args.steps // 2)
        a18 = torch.cuda.Event(enable_timing=True)
        b18 = torch.cuda.Event(enable_timing=True)
        a18.record(stream)
        for _ in range(n18):
            step18()
        b18.record(stream)
        barrier()
        ms18 = max_over_ranks(a18.elapsed_time(b18)) / n18
        bytes18 = px * 19 + hsx * hsy
        all18 = {"planes": 18, "value": world * px / (ms18 * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms18,
                 "achieved_gbs": bytes18 / (ms18 * 1e-3) / 1e9, "frac": bytes18 / (ms18 * 1e-3) / 1e9 / measured_peak()[0],
                 "note": "all 18 rasters of a block (2 drainage conditions x 9 lookups) in one fused pass"}
        del d_out18
    except Exception as e:  # extra information only
        all18 = {"error": repr(e)}

    # ---- BASELINE configs[0]: lookup g_ii only (one plane: 1 B read + 1 B written per pixel)
    config0 = None
    try:
        ptr0 = [0] * 18
        ptr0[7] = d_out[0].data_ptr()

        def step0():
            ctx.block_device(d_esa.data_ptr(), w, h, w, gt, d_hsg.data_ptr(), hsx, hsy, hsx, sgt,
                             1 << 7, ptr0, w, stream=stream.cuda_stream)
        for _ in range(3):
            step0()
        barrier()
        n0 = max(5, args.steps)
        a0 = torch.cuda.Event(enable_timing=True)
        b0 = torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(n0):
            step0()
        b0.record(stream)
        barrier()
        ms0 = max_over_ranks(a0.elapsed_time(b0)) / n0
        bytes0 = px * 2 + hsx * hsy
        config0 = {"workload": "BASELINE configs[0]: same tile, lookup g_ii only (drained), one plane", "planes": 1,
                   "value": world * px / (ms0 * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms0,
                   "achieved_gbs": bytes0 / (ms0 * 1e-3) / 1e9, "frac": bytes0 / (ms0 * 1e-3) / 1e9 / measured_peak()[0],
                   "algorithmic_bytes_per_launch": bytes0, "kernel": "gcn10::cn_block_kernel<1,1>"}
        step()      # leave the nine-plane result in d_out for the spot check below
    except Exception as e:  # extra information only
        config0 = {"error": repr(e)}

    # ---- end to end through the host-buffer C ABI (pinned host memory both ways)
    e2e = None
    e2e_steps = args.e2e_steps if args.e2e_steps is not None else min(args.steps, 5)
    if e2e_steps > 0:
        e2e = run_e2e(args, ctx, capi, d_esa, hsg_np, gt, sgt, w, h, world, barrier, max_over_ranks, e2e_steps, group)

    clocks = sampler.stop() if rank == 0 else None

    # spot check on rank 0: one sampled row of the device result against itself through the host path
    # (full parity lives in tests/; this only guards against timing a kernel that writes nothing)
    chk = int(d_out[:, h // 2, : min(w, 4096)].to(torch.int64).sum().item())
    if chk == 0 or chk == 255 * NVAR * min(w, 4096):
        raise SystemExit("bench.py: output plane looks unwritten")

    algo_bytes = px * (1 + NVAR) + hsx * hsy
    achieved = algo_bytes / (mean_step_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak()
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": profiled_traffic(), "peak_source": peak_src,
            # SURVEY 8(d): also against the nominal 8 TB/s of the north star (target: >= 0.70 of it)
            "frac_of_nominal_8000_gbs": achieved / 8000.0,
            "algorithmic_bytes_per_launch": algo_bytes, "mean_launch_ms": mean_step_ms,
            "kernel": "gcn10::cn_block_kernel<9,1> (+ index_map_kernel, O(W+H))"}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu = cpu_baseline_one_core(args, lookup_dir)
            except Exception as e:  # the baseline leg must never take the benchmark down
                cpu = {"value": None, "unit": UNIT, "cores": 1, "kind": "unavailable", "sample": repr(e)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
            "cpu_baseline": cpu,
            "output_gpixel_per_s": value * NVAR, "numa_node_rank0": numa_node, "all_18_planes": all18,
            "config0": config0, "strip_hand_over": "ship kernel" if ship else "size read-back + copy engine",
        }
        print_json(line)
    ctx.close()
    group.close()
    return 0


def pcie_probe(ctx, group, barrier):
    """The host link this end-to-end number sits under: copy bandwidth of one GPU alone (rank 0, the others idle) and
    of all ranks at once (what the shared host fabric gives each GPU when N blocks' tile streams leave together)."""
    # 1 GiB per copy, so that eight ranks' buffers do not sit in the host's last-level cache: with a reused 256 MB
    # buffer the concurrent figure came out 3x above what the raw-plane and tile-stream legs sustain on the same box
    nbytes, reps = 1 << 30, 3
    alone = None
    barrier()
    if group.rank == 0:
        alone = ctx.pcie_probe(nbytes, reps)
    barrier()
    mine = ctx.pcie_probe(nbytes, reps)
    barrier()
    out = {"bytes": nbytes, "alone": alone}
    conc = {}
    for k, v in mine.items():
        conc[k + "_min"] = -group.max(-v)
        conc[k + "_sum"] = group.sum(v)
    out["concurrent"] = conc
    if alone:
        out["d2h_gbs_alone"] = alone["d2h_gbs"]
        out["d2h_gbs_concurrent"] = conc["d2h_gbs_min"]
        out["frac"] = conc["d2h_gbs_min"] / alone["d2h_gbs"]
    return out


def run_e2e(args, ctx, capi, d_esa, hsg_np, gt, sgt, w, h, world, barrier, max_over_ranks, steps, group):
    import numpy as np
    import psutil

    need = (1 + NVAR) * w * h
    avail = psutil.virtual_memory().available
    rows = h
    note = None
    if need * world * 1.3 > avail:
        # not enough host RAM to pin a full tile's planes on every rank: use a row slab
        rows = max(256, int(h * avail / (need * world * 1.3)) // 256 * 256)
        note = f"host RAM limited: e2e measured on a {rows}-row slab"
    lib = ctx.lib
    esa_pin = capi.PinnedArray(lib, (rows, w))
    out_pin = capi.PinnedArray(lib, (NVAR, rows, w))
    try:
        esa_pin.array[:] = d_esa[:rows].cpu().numpy()
        planes = out_pin.array
        # capi.Context.block wants an [18,h,w] array; build the pointer list by hand instead
        import ctypes as C
        ptrs = (C.c_void_p * capi.NPLANES)()
        for k in range(NVAR):
            ptrs[k] = planes[k].ctypes.data
        gt6 = (C.c_double * 6)(*gt)
        sgt6 = (C.c_double * 6)(*sgt)
        hsy, hsx = hsg_np.shape

        def step():
            rc = lib.gcn10_cuda_block(ctx.h, esa_pin.array.ctypes.data, w, rows, w, gt6, hsg_np.ctypes.data, hsx, hsy,
                                      hsx, sgt6, capi.MASK_DRAINED, ptrs, w)
            if rc:
                raise RuntimeError(lib.gcn10_cuda_last_error().decode())
            # the device->host read of the result is part of the call; touch it like a consumer would
            return int(planes[NVAR - 1, rows - 1, w - 1])

        for _ in range(2):
            step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        # ---- same call with the reference's save_raster() encode step fused in: DEFLATE tiles come back
        nbytes = [0, 0]

        def _sink(_user, sp):
            st = sp.contents
            nbytes[0] += st.blob_bytes
            nbytes[1] += st.n_planes * st.n_tile_rows * st.tiles_x * 12 + 16
            return 0

        cb = capi.TILE_SINK(_sink)

        def step_deflate():
            rc = lib.gcn10_cuda_block_deflate(ctx.h, esa_pin.array.ctypes.data, w, rows, w, gt6, hsg_np.ctypes.data, hsx,
                                              hsy, hsx, sgt6, capi.MASK_DRAINED, cb, None)
            if rc:
                raise RuntimeError(lib.gcn10_cuda_last_error().decode())

        for _ in range(2):
            step_deflate()
        barrier()
        nbytes[0] = nbytes[1] = 0
        t0 = time.perf_counter()
        for _ in range(steps):
            step_deflate()
        barrier()
        dt_z = max_over_ranks(time.perf_counter() - t0)
        deflate = {"value": world * float(w) * rows * steps / dt_z / 1e9, "unit": UNIT,
                   "h2d_bytes_per_step": int(w * rows + hsg_np.size),
                   "d2h_bytes_per_step": int((nbytes[0] + nbytes[1]) / steps),
                   "steps": steps, "ms_per_step": dt_z / steps * 1e3, "kernel_ms_per_step": ctx.last_kernel_ms(),
                   "compression_ratio": NVAR * float(w) * rows * steps / max(nbytes[0], 1),
                   "path": "gcn10_cuda_block_deflate: pinned host raster (decoded land cover) -> H2D / fused Curve "
                           "Number + tile DEFLATE kernel / D2H of zlib tile streams (the payload of save_raster's GTiff "
                           "tiles) -> pinned host (PCIe H2D bound: 1 byte per pixel)"}

        # ---- the whole load_raster -> cn.c -> save_raster chain: the land cover arrives as the DEFLATE tiles of
        # the GeoTIFF (1024 x 1024, zlib level 6: the layout of the ESA WorldCover files the reference's VRT
        # points at), is inflated on the GPU, and the Curve Number tiles leave compressed
        tiles_in = None
        try:
            tiles_in = run_e2e_tiles(args, ctx, capi, esa_pin.array, rows, w, gt6, sgt6, hsg_np, cb, nbytes, world,
                                     barrier, max_over_ranks, steps, group)
        except Exception as e:  # extra leg: never take the benchmark down
            tiles_in = {"error": repr(e)}

        raw = {"value": world * float(w) * rows * steps / dt / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int(w * rows + hsg_np.size), "d2h_bytes_per_step": int(NVAR * w * rows),
               "steps": steps, "ms_per_step": dt / steps * 1e3,
               "path": "gcn10_cuda_block: pinned host rasters -> strip-pipelined H2D / fused kernel / D2H of the nine raw "
                       "planes -> pinned host (PCIe D2H bound)"}
        # headline: the call the gcn10 host program makes by default (compressed tiles); the raw-plane call is
        # reported beside it
        if tiles_in and "value" in tiles_in:
            res = dict(tiles_in)
            res["raster_in"] = deflate
        else:
            res = dict(deflate)
            res["tiles_in"] = tiles_in
        res["raw_planes"] = raw
        try:
            res["pcie"] = pcie_probe(ctx, group, barrier)
            if res["pcie"].get("d2h_gbs_concurrent") and "d2h_bytes_per_step" in res and "ms_per_step" in res:
                # share of the probed device->host ceiling that the tile streams of a step use
                res["pcie"]["e2e_d2h_gbs_per_gpu"] = res["d2h_bytes_per_step"] / (res["ms_per_step"] * 1e-3) / 1e9
                res["pcie"]["e2e_frac_of_concurrent_d2h"] = (res["pcie"]["e2e_d2h_gbs_per_gpu"] /
                                                             res["pcie"]["d2h_gbs_concurrent"])
        except Exception as e:
            res["pcie"] = {"error": repr(e)}
        if note:
            res["note"] = note
        return res
    finally:
        esa_pin.free()
        out_pin.free()


def run_e2e_tiles(args, ctx, capi, esa, rows, w, gt6, sgt6, hsg_np, cb, nbytes, world, barrier, max_over_ranks, steps,
                  group, in_tile=1024, level=6):
    """Compressed tiles in, compressed tiles out (gcn10_cuda_block_tiles_deflate).  The tile bytes are produced
    once, outside the timed region, with zlib on the host: they stand for the bytes of the input GeoTIFF."""
    import ctypes as C
    import zlib
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np

    lib = ctx.lib
    tiles_x, tiles_y = (w + in_tile - 1) // in_tile, (rows + in_tile - 1) // in_tile

    def one(i):
        ty, tx = divmod(i, tiles_x)
        t = np.zeros((in_tile, in_tile), dtype=np.uint8)
        part = esa[ty * in_tile:(ty + 1) * in_tile, tx * in_tile:(tx + 1) * in_tile]
        t[:part.shape[0], :part.shape[1]] = part
        return zlib.compress(t.tobytes(), level)

    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 8)) as ex:
        streams = list(ex.map(one, range(tiles_x * tiles_y)))
    sizes = np.array([len(z) for z in streams], dtype=np.uint32)
    offsets = np.concatenate([[0], np.cumsum(sizes[:-1], dtype=np.uint64)]).astype(np.uint64)
    total = int(sizes.sum())
    blob_pin = capi.PinnedArray(lib, (max(total, 1),))
    try:
        pos = 0
        for z in streams:
            blob_pin.array[pos:pos + len(z)] = np.frombuffer(z, dtype=np.uint8)
            pos += len(z)
        del streams
        src = capi.TileSource(in_tile, in_tile, tiles_x, tiles_y, 0, 0, blob_pin.array[:total], offsets, sizes)
        st = src.struct()
        hsy, hsx = hsg_np.shape

        def step():
            # the next block's tiles start their way to the GPU (H2D + inflate) beside this block's strips, as a
            # worker that knows its next block would do; every step still uploads and inflates exactly one block
            rc = lib.gcn10_cuda_tiles_prefetch(ctx.h, C.byref(st), w, rows)
            if rc:
                raise RuntimeError(lib.gcn10_cuda_last_error().decode())
            rc = lib.gcn10_cuda_block_tiles_deflate(ctx.h, C.byref(st), w, rows, gt6, hsg_np.ctypes.data, hsx, hsy, hsx,
                                                    sgt6, capi.MASK_DRAINED, cb, None)
            if rc:
                raise RuntimeError(lib.gcn10_cuda_last_error().decode())

        if lib.gcn10_cuda_tiles_prefetch(ctx.h, C.byref(st), w, rows):
            raise RuntimeError(lib.gcn10_cuda_last_error().decode())
        for _ in range(2):
            step()
        barrier()
        nbytes[0] = nbytes[1] = 0
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        kernel_ms_step, inflate_ms_step = ctx.last_kernel_ms(), ctx.last_inflate_ms()
        # the same call for all 18 rasters of a block (both drainage conditions): what the gcn10 program asks for
        # (pipelined like the 9-plane steps: the slot prefetched by the last of those is this leg's first block)
        def step18():
            rc = lib.gcn10_cuda_tiles_prefetch(ctx.h, C.byref(st), w, rows)
            if rc:
                raise RuntimeError(lib.gcn10_cuda_last_error().decode())
            rc = lib.gcn10_cuda_block_tiles_deflate(ctx.h, C.byref(st), w, rows, gt6, hsg_np.ctypes.data, hsx, hsy, hsx,
                                                    sgt6, capi.MASK_ALL, cb, None)
            if rc:
                raise RuntimeError(lib.gcn10_cuda_last_error().decode())

        saved = list(nbytes)
        for _ in range(2):
            step18()
        barrier()
        nbytes[0] = nbytes[1] = 0
        t0 = time.perf_counter()
        for _ in range(steps):
            step18()
        barrier()
        dt18 = max_over_ranks(time.perf_counter() - t0) / steps
        bytes18 = nbytes[0] + nbytes[1]          # of the timed steps only (the call below is one more block)
        # (the block the last step prefetched is still waiting: run it, untimed, so that the next leg starts clean)
        rc = lib.gcn10_cuda_block_tiles_deflate(ctx.h, C.byref(st), w, rows, gt6, hsg_np.ctypes.data, hsx, hsy, hsx, sgt6,
                                                capi.MASK_ALL, cb, None)
        if rc:
            raise RuntimeError(lib.gcn10_cuda_last_error().decode())
        all18 = {"planes": 18, "value": world * float(w) * rows / dt18 / 1e9, "unit": UNIT, "ms_per_step": dt18 * 1e3,
                 "d2h_bytes_per_step": int(bytes18 / steps)}
        nbytes[0], nbytes[1] = saved
        d2h_step = int((nbytes[0] + nbytes[1]) / steps)
        out_ratio = NVAR * float(w) * rows * steps / max(nbytes[0], 1)
        queue64 = program = None
        if args.queue_blocks > 0:
            try:
                queue64 = run_queue64(args, ctx, capi, blob_pin.array[:total], offsets, sizes, tiles_x, tiles_y, in_tile,
                                      w, rows, cb, nbytes, group, barrier, max_over_ranks)
            except Exception as e:
                queue64 = {"error": repr(e)}
        if args.program_blocks > 0:
            try:
                program = run_program_leg(args, blob_pin.array[:total], offsets, sizes, in_tile, w, rows, hsg_np, group,
                                          barrier)
            except Exception as e:
                program = {"error": repr(e)}
        return {"value": world * float(w) * rows * steps / dt / 1e9, "unit": UNIT, "all_18_planes": all18,
                "queue64": queue64, "program": program,
                "h2d_bytes_per_step": int(total + offsets.nbytes + sizes.nbytes + hsg_np.size),
                "d2h_bytes_per_step": d2h_step,
                "steps": steps, "ms_per_step": dt / steps * 1e3, "kernel_ms_per_step": kernel_ms_step,
                "inflate_kernel_ms": inflate_ms_step,
                "input_compression_ratio": float(w) * rows / max(total, 1),
                "output_compression_ratio": out_ratio,
                "input_tiles": [in_tile, in_tile, int(tiles_x * tiles_y)],
                "path": "gcn10_cuda_block_tiles_deflate: pinned host DEFLATE tiles of the land-cover GeoTIFF (zlib "
                        f"level {level}, {in_tile} x {in_tile}) -> H2D / GPU inflate / fused Curve Number + tile DEFLATE "
                        "kernel / D2H of the nine rasters' zlib tile streams -> pinned host (load_raster + cn.c + "
                        "save_raster of process_block with compressed bytes on PCIe both ways); each step also issues "
                        "gcn10_cuda_tiles_prefetch for the following block, so one block's upload + inflate overlaps "
                        "the previous block's strips"}
    finally:
        blob_pin.free()


def queue_blocks(n):
    """The 8 x 8 grid of 3-degree blocks with SW corner (-114, 30) (SURVEY 8d config 4: lon -114..-90, lat 30..54;
    it contains all 16 ids of the reference's src/test/blocks.txt): [(id, west, north)], row-major from the NW."""
    with open(os.path.join(ROOT, "tests", "golden", "block_extents.json")) as f:
        ext = {(int(w_), int(n_)): int(i) for i, w_, n_ in json.load(f)["blocks"]}
    out = []
    for north in range(54, 30, -3):
        for west in range(-114, -90, 3):
            out.append((ext[(west, north)], float(west), float(north)))
    return out[:n]


def run_queue64(args, ctx, capi, blob, offsets, sizes, tiles_x, tiles_y, in_tile, w, rows, cb, nbytes, group, barrier,
                max_over_ranks, nvariants=8):
    """BASELINE configs[3]: 64 blocks (8 x 8) handed out by the per-GPU block work queue -- every rank (GPU worker)
    claims its next block with an atomic fetch-and-add on the job's store (dist.BlockQueue, the cross-process twin of
    the atomic counter in host_pipeline.c; the reference's static round-robin is main.c:171), prefetches it (upload +
    GPU inflate) beside the block it is working on and runs gcn10_cuda_block_tiles_deflate on it.  Strong scaling: the
    64 blocks are the whole job at every N.  Each block has its own geotransform (so its own fp64 index maps), one of 8
    HSG windows and one of 8 arrangements of the compressed land-cover tiles (the tile grid of the benchmark block
    rotated by whole tiles: distinct rasters without compressing 64 x 1.3 GB on the host)."""
    import ctypes as C

    import numpy as np

    from gcn10_b200 import dist as gdist
    from gcn10_b200 import synth
    lib = ctx.lib
    blocks = queue_blocks(args.queue_blocks)
    off2, size2 = offsets.reshape(tiles_y, tiles_x), sizes.reshape(tiles_y, tiles_x)
    srcs = []
    for v in range(nvariants):
        dy, dx = (5 * v) % tiles_y, (11 * v) % tiles_x
        o = np.ascontiguousarray(np.roll(off2, (dy, dx), axis=(0, 1))).reshape(-1)
        z = np.ascontiguousarray(np.roll(size2, (dy, dx), axis=(0, 1))).reshape(-1)
        src = capi.TileSource(in_tile, in_tile, tiles_x, tiles_y, 0, 0, blob, o, z)
        srcs.append((src, src.struct()))
    hsgs = []
    for v in range(nvariants):
        gt_, sgt_, hsx, hsy = synth.block_geometry(0.0, 0.0, w, rows)
        hsgs.append(np.ascontiguousarray(synth.hsg_tile(hsx, hsy, 5000 + v, args.profile)))
    geo = []
    for bid, west, north in blocks:
        gt_, sgt_, hsx, hsy = synth.block_geometry(west, north, w, rows)
        geo.append(((C.c_double * 6)(*gt_), (C.c_double * 6)(*sgt_), hsx, hsy))

    def prefetch(k):
        if lib.gcn10_cuda_tiles_prefetch(ctx.h, C.byref(srcs[k % nvariants][1]), w, rows):
            raise RuntimeError(lib.gcn10_cuda_last_error().decode())

    def process(k):
        gt6, sgt6, hsx, hsy = geo[k]
        hs = hsgs[(k // nvariants) % nvariants]
        rc = lib.gcn10_cuda_block_tiles_deflate(ctx.h, C.byref(srcs[k % nvariants][1]), w, rows, gt6, hs.ctypes.data, hsx,
                                                hsy, hsx, sgt6, capi.MASK_DRAINED, cb, None)
        if rc:
            raise RuntimeError(lib.gcn10_cuda_last_error().decode())

    def run(name, n):
        q = gdist.BlockQueue(group, n, name)
        mine = []
        cur = q.claim()
        if cur is not None:
            prefetch(cur)
        while cur is not None:
            nxt = q.claim()
            if nxt is not None:
                prefetch(nxt)
            process(cur)
            mine.append(cur)
            cur = nxt
        return mine

    run("warm", min(len(blocks), 2 * group.world))
    barrier()
    nbytes[0] = nbytes[1] = 0
    t0 = time.perf_counter()
    mine = run("timed", len(blocks))
    barrier()
    dt = max_over_ranks(time.perf_counter() - t0)
    counts = group.gather_ints(len(mine))
    d2h = group.sum(nbytes[0] + nbytes[1])
    assert sum(counts) == len(blocks), counts
    return {"workload": (f"BASELINE configs[3]: {len(blocks)} blocks (8 x 8 grid, SW corner -114/30, ids "
                         f"{blocks[0][0]}..{blocks[-1][0]}) of {w} x {rows} px over the dynamic per-GPU block queue"),
            "value": len(blocks) * float(w) * rows / dt / 1e9, "unit": UNIT, "scaling": "strong",
            "blocks": len(blocks), "blocks_per_rank": counts, "seconds": dt, "ms_per_block": dt / len(blocks) * 1e3,
            "distinct_land_cover_arrangements": nvariants, "distinct_hsg_windows": nvariants,
            "d2h_bytes_total": int(d2h),
            "claim": "atomic fetch-and-add on the rendezvous store (TCPStore.add), one block ahead for the prefetch"}


def run_program_leg(args, blob, offsets, sizes, in_tile, w, rows, hsg_np, group, barrier):
    """File to file: the gcn10 executable (C host program + libgcn10cuda) on a RAM disk.  One tiled DEFLATE GeoTIFF
    holds the benchmark's compressed land-cover tiles; a GDAL VRT places it B times side by side (the structure of
    the reference's landcover/esa_worldcover_2021.vrt), a shapefile holds the B block extents, and the program writes
    all 18 GeoTIFFs of every block.  Per-block times are the program's own log lines (time between consecutive
    blocks of a worker: read, GPU inflate, Curve Numbers, tile DEFLATE and the 18 file writes overlapped), the first
    block of every worker (CUDA start-up) excluded.  Rank 0 launches it on all N GPUs; the other ranks wait."""
    import re
    import shutil

    import numpy as np

    from gcn10_b200 import hostlib
    from tests import fixtures, lookups
    barrier()
    res = None
    if group.rank == 0 and os.path.exists(hostlib.EXE_PATH):
        nb = args.program_blocks * group.world
        # 18 rasters of ~22 MB per block + the inputs; a RAM disk that cannot hold them must not take the run down
        need = nb * 450e6 + 200e6
        bases = [d for d in ("/dev/shm", tempfile.gettempdir()) if os.path.isdir(d) and shutil.disk_usage(d).free > need]
        if not bases:
            barrier()
            return {"skipped": f"no scratch directory with {need / 1e9:.1f} GB free for {nb} blocks"}
        base = bases[0]
        root = tempfile.mkdtemp(prefix="gcn10_program_", dir=base)
        try:
            px = 1.0 / 12000.0
            lon0, lat0 = -114.0, 42.0
            gt = (lon0, px, 0.0, lat0, 0.0, -px)
            hostlib.write_tiled_deflate_tiff(os.path.join(root, "lc.tif"), w, rows, in_tile, in_tile, blob, offsets, sizes, gt)
            from tests.fixtures import write_vrt
            srcs = [("lc.tif", 0, 0, k * w, 0, w, rows) for k in range(nb)]
            write_vrt(os.path.join(root, "lc.vrt"), nb * w, rows, gt, srcs)
            hsy, hsx = hsg_np.shape
            hostlib.tiff_write(os.path.join(root, "hsg.tif"), np.tile(hsg_np, (1, nb)), (lon0, 1.0 / 480.0, 0.0, lat0, 0.0, -1.0 / 480.0))
            deg_w, deg_h = w * px, rows * px
            blocks = [(100 + k, lon0 + k * deg_w, lat0 - deg_h, lon0 + (k + 1) * deg_w, lat0) for k in range(nb)]
            fixtures.write_block_shapefile(os.path.join(root, "blocks.shp"), blocks)
            lookups.write_default_lookups(os.path.join(root, "lookups"))
            fixtures.write_config(os.path.join(root, "config.txt"), os.path.join(root, "lc.vrt"), os.path.join(root, "hsg.tif"),
                                  os.path.join(root, "blocks.shp"), os.path.join(root, "lookups"), os.path.join(root, "logs"))
            with open(os.path.join(root, "blocks.txt"), "w") as f:
                f.write("\n".join(str(b[0]) for b in blocks) + "\n")
            os.makedirs(os.path.join(root, "out"), exist_ok=True)
            t0 = time.perf_counter()
            r = subprocess.run([hostlib.EXE_PATH, "-c", os.path.join(root, "config.txt"), "-l", os.path.join(root, "blocks.txt"),
                                "-o", "--gpus", str(group.world), "--outdir", os.path.join(root, "out")],
                               cwd=root, capture_output=True, text=True, timeout=900,
                               env=dict(os.environ, GCN10_HOST_INFLATE="0", GCN10_HOST_DEFLATE="0"))
            wall = time.perf_counter() - t0
            per_worker = {}
            last_line = None
            logs = os.path.join(root, "logs")
            for fn in sorted(os.listdir(logs)) if os.path.isdir(logs) else []:
                for ln in open(os.path.join(root, "logs", fn)):
                    m = re.search(r"block (\d+): (\d+) x (\d+) px, 18 rasters in ([0-9.]+) s", ln)
                    if m:
                        per_worker.setdefault(fn, []).append(float(m.group(4)))
                        last_line = ln.strip()
            warm = [t for ts in per_worker.values() for t in ts[1:]]
            files = sum(len(fs) for _, _, fs in os.walk(os.path.join(root, "out")))
            out_bytes = sum(os.path.getsize(os.path.join(d, f)) for d, _, fs in os.walk(os.path.join(root, "out")) for f in fs)
            res = {"returncode": r.returncode, "blocks": nb, "gpus": group.world, "rasters_written": files,
                   "output_bytes": out_bytes, "wall_s_incl_startup": wall,
                   "path": f"gcn10 executable: VRT mosaic of a tiled DEFLATE GeoTIFF on {base} -> 18 GeoTIFFs per block on {base}",
                   "last_block_log_line": last_line}
            if warm:
                warm.sort()
                med = warm[len(warm) // 2]
                nworkers = max(1, len(per_worker))
                res.update({"ms_per_block_warm": med * 1e3, "warm_blocks": len(warm),
                            "value": nworkers * float(w) * rows / med / 1e9, "unit": UNIT,
                            "note": "value = workers x pixels / median warm per-block time (all 18 rasters per block)"})
            if r.returncode != 0 or files != 18 * nb:
                res["stderr_tail"] = r.stderr[-800:]
        except Exception as e:  # rank 0 must reach the barrier below whatever happens: the other ranks wait there
            res = {"error": repr(e)}
        finally:
            shutil.rmtree(root, ignore_errors=True)
    barrier()
    return res


def load_tables_host(lookup_dir):
    """The nine int[256][5] tables: via the host library's CSV reader when built, else the same
    parsing rules restated here (first line skipped, '<lc>_<A|B|C|D>,<cn>', cn.c:13-85)."""
    import numpy as np
    try:
        from gcn10_b200 import hostlib
        return hostlib.load_lookup_tables(lookup_dir)
    except Exception:
        pass
    from tests import lookups
    t = np.full((9, 256, 5), 255, dtype=np.int32)
    for i, v in enumerate(lookups.VARIANTS):
        with open(os.path.join(lookup_dir, f"default_lookup_{v}.csv"), "rb") as f:
            lines = f.read().split(b"\n")[1:]
        for ln in lines:
            if b"," not in ln or b"_" not in ln.split(b",")[0]:
                continue
            code, val = ln.split(b",")[:2]
            lc, letter = code.split(b"_", 1)
            sg = {b"A": 1, b"B": 2, b"C": 3}.get(letter[:1], 4)
            t[i, int(lc), sg] = int(val.strip() or 0)
    return t


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md), MEASURED_PEAKS.json absent"


def profiled_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get("dram_bytes_per_launch")
    except Exception:
        return None


print_json = None


def main():
    sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)
    args = parse_args()
    # stdout must carry exactly one JSON line: libraries (NCCL prints its version banner to stdout on the
    # first collective) are diverted to stderr for the whole run and the line is written to the real stdout
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")
    global print_json
    def print_json(obj):
        out.write(json.dumps(obj) + "\n")
        out.flush()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
