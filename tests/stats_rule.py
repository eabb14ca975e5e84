"""The statistics rule of the GeoTIFF writer (stats_metadata in gcn10_b200/host/host_tiff.c) restated in Python, for
the tests: the band statistics GDAL computes for a file whose NoData value is 255, as GDAL_METADATA items of sample 0."""
import math
import re

import numpy as np

NODATA = 255
ITEMS = ("STATISTICS_MAXIMUM", "STATISTICS_MEAN", "STATISTICS_MINIMUM", "STATISTICS_STDDEV", "STATISTICS_VALID_PERCENT")


def from_histogram(hist, pixels):
    """{item: value} from 256 pixel counts of a raster of `pixels` pixels: only values other than 255 count, the
    standard deviation is the population one; no valid pixel gives VALID_PERCENT 0 and nothing else."""
    n = [int(c) for c in hist[:NODATA]]                # exact integers
    valid = sum(n)
    pct = 100.0 * valid / pixels
    if valid == 0:
        return {"STATISTICS_VALID_PERCENT": pct}
    vals = [v for v in range(NODATA) if n[v]]
    s = sum(v * n[v] for v in vals)
    s2 = sum(v * v * n[v] for v in vals)
    return {"STATISTICS_MAXIMUM": float(vals[-1]), "STATISTICS_MEAN": s / valid, "STATISTICS_MINIMUM": float(vals[0]),
            "STATISTICS_STDDEV": math.sqrt(valid * s2 - s * s) / valid, "STATISTICS_VALID_PERCENT": pct}


def of_plane(a):
    a = np.asarray(a)
    return from_histogram(np.bincount(a.ravel(), minlength=256), a.size)


def parse(xml):
    """{item: value} of the sample-0 items of a GDAL_METADATA text."""
    return {m.group(1): float(m.group(2))
            for m in re.finditer(r'<Item name="([A-Z_]+)" sample="0">([^<]*)</Item>', xml)}


def close(got, want, rel=1e-12):
    return got.keys() == want.keys() and all(math.isclose(got[k], want[k], rel_tol=rel, abs_tol=0.0) for k in want)
