"""GPU path against the committed golden fixtures (outputs of the reference's own object code)."""
import numpy as np
import pytest

from tests import golden_io

pytestmark = pytest.mark.gpu

BLOCKS = golden_io.block_cases()


@pytest.mark.parametrize("name", sorted(BLOCKS))
def test_gpu_matches_golden_blocks(name, gpu_ctx, port):
    c = BLOCKS[name]
    esa, gt, hsg, sgt = golden_io.window_inputs(port, c)
    got = gpu_ctx.block(np.ascontiguousarray(esa), gt, np.ascontiguousarray(hsg), sgt)
    assert np.array_equal(got, c["planes"])


def test_gpu_lut_probe_default_and_hostile(gpu_ctx, port, tables, lookup_dir, tmp_path):
    from tests.golden.make_golden import lut_probe_raster, write_hostile
    esa, esa_t, hsg, hsg_t, bbox, codes = lut_probe_raster()
    g = golden_io.luts()
    for label, d in (("default", lookup_dir), ("hostile", write_hostile(str(tmp_path / "h")))):
        t = port.load_tables(d)
        xo, yo, xc, yc, gt = port.window(esa.shape[1], esa.shape[0], esa_t, bbox)
        hxo, hyo, hxc, hyc, sgt = port.window(hsg.shape[1], hsg.shape[0], hsg_t, bbox)
        try:
            gpu_ctx.set_luts(t)
            got = gpu_ctx.block(np.ascontiguousarray(esa[yo:yo + yc, xo:xo + xc]), gt,
                                np.ascontiguousarray(hsg[hyo:hyo + hyc, hxo:hxo + hxc]), sgt)
        finally:
            gpu_ctx.set_luts(tables)
        assert np.array_equal(got, g[label]), label
