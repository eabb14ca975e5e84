"""Readers for the committed golden fixtures (tests/golden/, made by make_golden.py from the
reference's own object code)."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def block_cases():
    z = np.load(os.path.join(GOLDEN, "blocks.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    return {n: {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(n + "/")} for n in names}


def window_cases():
    with open(os.path.join(GOLDEN, "windows.json")) as f:
        return json.load(f)


def luts():
    z = np.load(os.path.join(GOLDEN, "luts.npz"))
    return {k: z[k] for k in z.files}


def block_extents():
    """[(id, west, north)] of the 2651 blocks of the reference's shapefile."""
    with open(os.path.join(GOLDEN, "block_extents.json")) as f:
        return [tuple(r) for r in json.load(f)["blocks"]]


def window_inputs(port, c):
    """Cut the ESA / HSG windows of a golden block case with the restated window arithmetic."""
    eh, ew = c["esa"].shape
    hh, hw = c["hsg"].shape
    we = port.window(ew, eh, c["esa_t"], c["bbox"])
    wh = port.window(hw, hh, c["hsg_t"], c["bbox"])
    assert we is not None and wh is not None
    xo, yo, xc, yc, gt = we
    hxo, hyo, hxc, hyc, sgt = wh
    return c["esa"][yo:yo + yc, xo:xo + xc], gt, c["hsg"][hyo:hyo + hyc, hxo:hxo + hxc], sgt


def effective_lut(tabs):
    """uint8 [18, codes, 256] behaviour of int tables for the probe raster of luts.npz."""
    g = luts()
    codes = g["hsg_codes"]
    out = np.full((18, len(codes), 256), 255, dtype=np.uint8)
    for c in range(2):
        for i, hv in enumerate(codes):
            s = hv
            if 11 <= hv <= 14:
                s = 4 if c == 0 else hv - 10
            if s >= 5:
                continue
            for t in range(9):
                v = tabs[t][:, s]
                out[c * 9 + t, i] = np.where(v < 255, v & 0xFF, 255).astype(np.uint8)
    return out
