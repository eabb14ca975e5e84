"""GPU parity: libgcn10cuda (through its C ABI) against the CPU oracle, bit for bit.

The oracle (oracle/cn_oracle.c) is itself pinned to the reference's object code in
tests/test_oracle_pinned.py.  Tolerance: none -- uint8 planes and int32 index maps must be equal.
"""
import numpy as np
import pytest

from gcn10_b200 import capi, synth
from tests.block_options import assemble
from tests.cases import SMALL_CASES, make_block, PX, PX_VRT, HSG_PX

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,kw", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_block_host_api_all_planes(name, kw, gpu_ctx, port, tables):
    b = make_block(**kw)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    for k in range(18):
        assert np.array_equal(got[k], want[k]), f"{name}: plane {k} differs in {(got[k] != want[k]).sum()} px"


@pytest.mark.parametrize("tma", [0, 1])
@pytest.mark.parametrize("rows_per_cta", [1, 7, 128, 1000])
def test_kernel_forms_agree(tma, rows_per_cta, gpu_ctx, port, tables):
    """TMA-staged vs gathered HSG box, several row-chunk heights."""
    b = make_block(w=4500, h=700, seed=21, shift=(0.0003, 0.0007), margin=1)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    gpu_ctx.set_option("tma", tma)
    gpu_ctx.set_option("rows_per_cta", rows_per_cta)
    try:
        got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_option("tma", 1)
        gpu_ctx.set_option("rows_per_cta", 0)
    assert np.array_equal(got, want)


def test_wide_hsg_span_falls_back_to_gather(gpu_ctx, port, tables):
    """Ratio 3: a 4096-pixel strip spans > 256 HSG columns, so no CTA fits the TMA box."""
    b = make_block(w=9000, h=150, hsg_px=1.0 / 12000.0 * 3, seed=23)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    assert np.array_equal(got, want)


@pytest.mark.parametrize("strip_rows,streams", [(1, 1), (37, 3), (512, 4), (100000, 2)])
def test_strip_pipeline_shapes(strip_rows, streams, gpu_ctx, port, tables):
    b = make_block(w=1234, h=999, seed=5)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    gpu_ctx.set_option("strip_rows", strip_rows)
    gpu_ctx.set_option("streams", streams)
    try:
        got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_option("strip_rows", 2048)
        gpu_ctx.set_option("streams", 8)
    assert np.array_equal(got, want)


MASKS = {
    "g_ii_only_drained": 1 << 7,                      # BASELINE config 1
    "nine_drained": capi.MASK_DRAINED,                # BASELINE config 2
    "nine_undrained": capi.MASK_UNDRAINED,
    "same_three_both": (0b000010101) | (0b000010101 << 9),
    "different_per_condition": 0b000000110 | (0b101000000 << 9),
    "single_undrained": 1 << 17,
}


@pytest.mark.parametrize("mname", list(MASKS))
def test_plane_masks(mname, gpu_ctx, port, tables):
    mask = MASKS[mname]
    b = make_block(w=2100, h=333, seed=8, profile="coastal")
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    out = np.full((18, 333, 2100), 7, dtype=np.uint8)
    got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask, out=out)
    for k in range(18):
        if mask & (1 << k):
            assert np.array_equal(got[k], want[k]), (mname, k)
        else:
            assert (got[k] == 7).all(), f"{mname}: unselected plane {k} was written"


def test_lut_edge_values(gpu_ctx, port, tables):
    """cn >= 255 -> nodata, negative cn wraps through (uint8_t), column 0 honoured (cn.c:123-128)."""
    t = tables.copy()
    rng = np.random.default_rng(3)
    t[:, :, :] = rng.integers(-300, 600, size=t.shape)
    t[2, 40, 1] = 255
    t[3, 40, 2] = 254
    t[4, 40, 3] = -1
    t[5, 40, 4] = 256
    b = make_block(w=1500, h=200, seed=9, profile="random")
    b["esa"] = rng.integers(0, 256, size=b["esa"].shape, dtype=np.uint8)      # every byte value
    b["hsg"] = rng.integers(0, 256, size=b["hsg"].shape, dtype=np.uint8)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t)
    try:
        gpu_ctx.set_luts(t)
        got = gpu_ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
    finally:
        gpu_ctx.set_luts(tables)
    assert np.array_equal(got, want)


GEOMS = [
    # (w, h, gt, hsx, hsy, soil_gt)
    (36000, 36000, (-114.0, PX, 0, 42.0, 0, -PX), 1440, 1440, (-114.0, HSG_PX, 0, 42.0, 0, -HSG_PX)),
    (36001, 36001, (-3.0, PX_VRT, 0, 3.0, 0, -PX_VRT), 1441, 1441, (-3.0, HSG_PX, 0, 3.0, 0, -HSG_PX)),
    (36001, 36001, (33.0, PX_VRT, 0, -57.0, 0, -PX_VRT), 1442, 1442, (32.9993, HSG_PX, 0, -56.9989, 0, -HSG_PX)),
    (36000, 36000, (0.0, PX, 0, 0.0, 0, -PX), 1440, 1440, (0.0, HSG_PX, 0, 0.0, 0, -HSG_PX)),
    (36000, 36000, (177.0, PX, 0, 84.0, 0, -PX), 1440, 1440, (177.0, HSG_PX, 0, 84.0, 0, -HSG_PX)),
    # degenerate / absurd transforms: zero and negative HSG pixel, huge offsets, NaN
    (500, 400, (10.0, PX, 0, 5.0, 0, -PX), 30, 20, (10.0, 0.0, 0, 5.0, 0, -HSG_PX)),
    (500, 400, (10.0, PX, 0, 5.0, 0, -PX), 30, 20, (10.0, -HSG_PX, 0, 5.0, 0, HSG_PX)),
    (500, 400, (1e300, PX, 0, -1e300, 0, -PX), 30, 20, (10.0, 1e-300, 0, 5.0, 0, -1e-300)),
    (500, 400, (float("nan"), PX, 0, 5.0, 0, -PX), 30, 20, (10.0, HSG_PX, 0, float("inf"), 0, -HSG_PX)),
    (500, 400, (10.0, -PX, 0, 5.0, 0, PX), 30, 20, (10.0 - 500 * PX, HSG_PX, 0, 5.0 + 400 * PX, 0, -HSG_PX)),
]


@pytest.mark.parametrize("g", range(len(GEOMS)))
def test_index_maps_match_reference_arithmetic(g, gpu_ctx, port):
    w, h, gt, hsx, hsy, sgt = GEOMS[g]
    ci, cj = gpu_ctx.index_maps(w, h, gt, hsx, hsy, sgt)
    assert np.array_equal(ci, port.col_index(w, gt, sgt, hsx))
    assert np.array_equal(cj, port.row_index(h, gt, sgt, hsy))


def _torch():
    import torch
    return torch


@pytest.mark.parametrize("w,h,pitch_extra", [(4096, 300, 0), (4111, 257, 0), (4111, 257, 5), (1000, 100, 3)])
def test_block_device_api(w, h, pitch_extra, gpu_ctx, port, tables):
    """Device-resident entry point; odd pitches exercise the byte-wise kernel."""
    torch = _torch()
    b = make_block(w=w, h=h, seed=31)
    want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
    pitch = (w + 15) // 16 * 16 + pitch_extra
    guard = 3                                                   # sentinel rows above and below every plane
    d_esa = torch.zeros((h, pitch), dtype=torch.uint8, device="cuda")
    d_esa[:, :w] = torch.from_numpy(b["esa"]).cuda()
    hsy, hsx = b["hsg"].shape
    d_hsg = torch.from_numpy(b["hsg"]).cuda().contiguous()
    d_out = torch.full((18, h + 2 * guard, pitch), 3, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream or 1      # 0 would mean "the context's stream"; 1 = cudaStreamLegacy
    gpu_ctx.block_device(d_esa.data_ptr(), w, h, pitch, b["gt"], d_hsg.data_ptr(), hsx, hsy, hsx, b["soil_gt"],
                         capi.MASK_ALL, [d_out[k, guard].data_ptr() for k in range(18)], pitch, stream=st)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    assert np.array_equal(got[:, guard:guard + h, :w], want)
    assert (got[:, guard:guard + h, w:] == 3).all(), "padding columns were written"
    assert (got[:, :guard] == 3).all() and (got[:, guard + h:] == 3).all(), "rows outside the block were written"


def test_block_async_blocks_in_flight(gpu_ctx, port, tables):
    """gcn10_cuda_block_async / gcn10_cuda_wait (SURVEY 8b): three blocks of different shapes queued back to back on
    one context from page-locked buffers, other compute calls refused meanwhile, results bit-exact."""
    lib = gpu_ctx.lib
    shapes = [(4111, 700, capi.MASK_ALL), (2048, 300, capi.MASK_DRAINED), (5000, 1300, 0b000010101 | (0b101 << 9))]
    blocks, pins, handles = [], [], []
    gpu_ctx.set_option("strip_rows", 256)
    try:
        for i, (w, h, mask) in enumerate(shapes):
            b = make_block(w=w, h=h, seed=40 + i, shift=(0.0002 * i, 0.0003), margin=1)
            e = capi.PinnedArray(lib, (h, w))
            o = capi.PinnedArray(lib, (18, h, w))
            e.array[:] = b["esa"]
            o.array[:] = 9
            pins += [e, o]
            blocks.append((b, mask))
            handles.append(gpu_ctx.block_async(e.array, b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask, out=o.array))
        with pytest.raises(capi.Gcn10Error):
            gpu_ctx.index_maps(100, 100, blocks[0][0]["gt"], 10, 10, blocks[0][0]["soil_gt"])
        with pytest.raises(capi.Gcn10Error):
            gpu_ctx.set_luts(tables)
        for (b, mask), hd in zip(blocks, handles):
            got = gpu_ctx.wait(hd)
            want = port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], tables)
            for k in range(18):
                if mask & (1 << k):
                    assert np.array_equal(got[k], want[k]), k
                else:
                    assert (got[k] == 9).all()
        assert gpu_ctx.last_kernel_ms() > 0
        # the context is free again
        ci, _ = gpu_ctx.index_maps(100, 100, blocks[0][0]["gt"], 10, 10, blocks[0][0]["soil_gt"])
        assert ci.shape == (100,)
        # query: a finished block reports 1 before it is waited for
        b, mask = blocks[1]
        hd = gpu_ctx.block_async(pins[2].array, b["gt"], b["hsg"], b["soil_gt"], plane_mask=mask, out=pins[3].array)
        gpu_ctx.lib.gcn10_cuda_synchronize(gpu_ctx.h)
        assert gpu_ctx.query(hd)
        gpu_ctx.wait(hd)
    finally:
        gpu_ctx.set_option("strip_rows", 2048)
        for p in pins:
            p.free()


def test_pcie_probe(gpu_ctx):
    r = gpu_ctx.pcie_probe(64 << 20, 2)
    assert all(v > 0.5 for v in r.values()), r


def test_contexts_in_concurrent_host_threads(port, tables):
    """SURVEY 8(b) threading: a context per worker thread, no state shared between contexts.  Three threads, each with
    its own context on cuda:0 and its own lookup tables (the third one's are permuted, so planes computed with the
    wrong context's tables would show), run different blocks through the plain and the compressed path at once."""
    import threading
    shapes = [dict(w=3100, h=900, seed=71), dict(w=1777, h=1301, seed=72, profile="coastal"),
              dict(w=2500, h=1111, seed=73, shift=(0.0003, 0.0007), margin=1)]
    other = tables.copy()
    other[:, :, 1:5] = tables[::-1, :, 1:5][:, :, ::-1]
    tabs = [tables, tables, other]
    blocks = [make_block(**kw) for kw in shapes]
    wants = [port.block_rows(b["esa"], b["gt"], b["hsg"], b["soil_gt"], t) for b, t in zip(blocks, tabs)]
    errors = []
    start = threading.Barrier(len(blocks))

    def work(i):
        try:
            ctx = capi.Context(0)
            ctx.set_luts(tabs[i])
            b, want = blocks[i], wants[i]
            start.wait()
            for rep in range(3):
                got = ctx.block(b["esa"], b["gt"], b["hsg"], b["soil_gt"])
                if not np.array_equal(got, want):
                    errors.append(f"thread {i} rep {rep}: block() differs")
                res = ctx.block_deflate(b["esa"], b["gt"], b["hsg"], b["soil_gt"], capi.MASK_ALL)
                h, w = b["esa"].shape
                if sorted(res["tiles"]) != list(range(18)):
                    errors.append(f"thread {i} rep {rep}: planes {sorted(res['tiles'])}")
                for k, d in res["tiles"].items():
                    if not np.array_equal(assemble(d, w, h), want[k]):        # asserts a complete tile grid
                        errors.append(f"thread {i} rep {rep}: plane {k} differs")
            ctx.close()
        except Exception as e:                  # noqa: BLE001 -- reported below
            errors.append(f"thread {i}: {e!r}")

    ts = [threading.Thread(target=work, args=(i,)) for i in range(len(blocks))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
