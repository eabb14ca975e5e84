"""bench.py's file-to-file leg must never strand the other ranks: whatever happens to the program on rank 0 (no GPU in
this container, a full RAM disk, a missing log directory), the leg returns a dict for the JSON line and passes both of
its barriers.  (The numbers themselves are GPU-box business: tests/test_gpu_program.py, bench.py.)"""
from __future__ import annotations

import os
import sys
import types
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from gcn10_b200 import hostlib, synth  # noqa: E402


class _Group:
    def __init__(self, rank, world=1):
        self.rank, self.world = rank, world


def _tiny_inputs(w=2048, t=1024):
    esa = synth.esa_tile(w, w, 1)
    blobs, offs, sizes, pos = [], [], [], 0
    for ty in range(w // t):
        for tx in range(w // t):
            z = zlib.compress(esa[ty * t:(ty + 1) * t, tx * t:(tx + 1) * t].tobytes(), 6)
            offs.append(pos)
            sizes.append(len(z))
            blobs.append(z)
            pos += len(z)
    _, _, hsx, hsy = synth.block_geometry(-114.0, 42.0, w, w)
    return (np.frombuffer(b"".join(blobs), np.uint8), np.array(offs, np.uint64), np.array(sizes, np.uint32), t, w,
            synth.hsg_tile(hsx, hsy, 2))


def test_program_leg_always_reaches_both_barriers(monkeypatch):
    blob, offs, sizes, t, w, hsg = _tiny_inputs()
    calls = []
    args = types.SimpleNamespace(program_blocks=2)
    res = bench.run_program_leg(args, blob, offs, sizes, t, w, w, hsg, _Group(0), lambda: calls.append(1))
    assert len(calls) == 2
    if os.path.exists(hostlib.EXE_PATH):
        assert isinstance(res, dict) and ("returncode" in res or "error" in res or "skipped" in res)
        if res.get("returncode", 0) != 0:
            assert "stderr_tail" in res, "a failed program run must say why in the line"
    # the other ranks only wait
    calls.clear()
    assert bench.run_program_leg(args, blob, offs, sizes, t, w, w, hsg, _Group(1, 2), lambda: calls.append(1)) is None
    assert len(calls) == 2
    # no room on any scratch directory: skipped, barriers still passed
    import shutil
    monkeypatch.setattr(shutil, "disk_usage", lambda d: types.SimpleNamespace(free=0, total=0, used=0))
    calls.clear()
    res = bench.run_program_leg(args, blob, offs, sizes, t, w, w, hsg, _Group(0), lambda: calls.append(1))
    if os.path.exists(hostlib.EXE_PATH):
        assert "skipped" in res
    assert len(calls) == 2


def test_dump_outputs_is_a_fixed_sample_of_the_planes(tmp_path):
    """--dump-outputs: float32 values at float64 flat indices, the same positions on every run, under 64 MB in all;
    every pixel of a tile small enough."""
    import torch
    small = torch.from_numpy(np.stack([synth.esa_tile(40, 30, k) for k in range(bench.NVAR)]))
    bench.dump_outputs(str(tmp_path / "small"), small, 40, 30)
    vals = np.load(tmp_path / "small" / "cn_drained.npy")
    idx = np.load(tmp_path / "small" / "cn_drained_index.npy")
    assert vals.dtype == np.float32 and idx.dtype == np.float64
    assert np.array_equal(idx, np.arange(40 * 30)) and np.array_equal(vals, small.reshape(bench.NVAR, -1).numpy())
    w = h = 1500
    big = torch.from_numpy(np.stack([synth.esa_tile(w, h, k, "random") for k in range(bench.NVAR)]))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), big, w, h)
    idx = np.load(tmp_path / "a" / "cn_drained_index.npy")
    vals = np.load(tmp_path / "a" / "cn_drained.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "cn_drained_index.npy"))
    assert idx.size <= bench.DUMP_SAMPLE and (np.diff(idx) > 0).all() and vals.shape == (bench.NVAR, idx.size)
    assert np.array_equal(vals, big.reshape(bench.NVAR, -1).numpy()[:, idx.astype(np.int64)])
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
