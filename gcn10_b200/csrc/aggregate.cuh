// gcn10_b200/csrc/aggregate.cuh -- option "aggregate" of the compressed-tile calls: the f x f mean raster of every
// selected plane (rule: gcn10_aggregate_* in include/gcn10_cuda.h), gathered strip by strip while the strip's land cover
// is on the device (sm_100a).
//
// aggregate_accumulate_kernel   once per full-resolution strip: per cell and selected plane, the sum and the count of
//                               the pixels that are not 255, added into uint32 accumulators on the context.  A pixel's
//                               value comes from the launch plans' LUT records and soil_slot(), the same tables and
//                               soil remap the Curve Number kernels read, so it serves the fused and the two-kernel
//                               path alike.
// aggregate_finish_kernel       after the block's last strip: gcn10_aggregate_value into one byte raster per plane,
//                               and the accumulators cleared for the next block.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gcn10_cuda.h"
#include "cn_kernels.cuh"

namespace gcn10 {

constexpr int kAggThreads = 256;

// one launch plan (plan_launches): its packed records and where its outputs go in the accumulators
struct AggPlan {
    const uint8_t *lut;             // the plan's records (kLutBytes; narrow layout when rec_bytes == 4)
    int rec_bytes;                  // 16 or 4
    int np, groups;                 // planes per group, groups (drainage conditions)
    int drained[2];
    int acc[18];                    // accumulator plane of the plan's output g * np + k
};

struct AggParams {
    const uint8_t *esa;             // the strip's land cover; row 0 = block row y0
    size_t esa_pitch;
    int y0, rows;                   // block rows of the strip
    int w;                          // block width
    int f, cw, ch;                  // factor, cells per row / column of the block
    int seg, spc;                   // pixels of a thread's column segment, segments per cell (seg * spc >= f)
    int chunk_rows, nchunk;         // a CTA walks at most chunk_rows (<= 32) rows of one cell row: nchunk per cell row
    int ncr;                        // cell rows the strip touches
    const int32_t *col_idx, *row_idx;   // the block's index maps
    const uint8_t *hsg;
    size_t hsg_pitch;
    int swz_shift;
    int nplans;
    AggPlan plan[2];
    int nsel;                       // accumulator planes
    uint2 *acc;                     // [nsel][ch][cw] (sum, count)
};

// grid = (ceil(cw / cells per CTA), cell-row chunks), 256 threads.  A thread owns a segment of at most 32 pixel
// columns of one cell and walks the rows of its CTA's chunk, with the segment's soil codes kept in shared memory while
// the HSG row stays the same; a run of equal (land cover, soil code) pairs -- the same record -- is looked up and
// added once.  Per thread and plane the sums stay in shared memory; then the first
// thread of every cell adds its siblings' and issues one global atomic pair per cell and plane (none for a cell whose
// pixels are all 255 so far).  Cells straddle strips and bands (256-row multiples against f), so partial cells meet
// in those atomics.
__global__ void __launch_bounds__(kAggThreads) aggregate_accumulate_kernel(const __grid_constant__ AggParams p)
{
    __shared__ uint32_t s_sum[GCN10_NPLANES][kAggThreads], s_cnt[GCN10_NPLANES][kAggThreads];
    __shared__ uint8_t s_soil[32][kAggThreads];         // soil code of the thread's k-th pixel column in HSG row hrow
    const int tid = threadIdx.x;
    const int cells = kAggThreads / p.spc;                 // cells per CTA (whole cells only)
    const int cx = blockIdx.x * cells + tid / p.spc;
    const int sub = tid % p.spc;
    const bool active = tid < cells * p.spc && cx < p.cw;
    const int cell_x0 = cx * p.f;
    const int xa = min(cell_x0 + sub * p.seg, p.w);
    const int xb = active ? min(min(xa + p.seg, cell_x0 + p.f), p.w) : xa;
    const int cr0 = p.y0 / p.f;
    int hrow = -1;

    for (int by = blockIdx.y; by < p.ncr * p.nchunk; by += gridDim.y) {
        const int cr = cr0 + by / p.nchunk;
        const int lo = max(p.y0, cr * p.f) + (by % p.nchunk) * p.chunk_rows;
        const int hi = min(min(p.y0 + p.rows, cr * p.f + p.f), lo + p.chunk_rows);
        if (lo >= hi)
            continue;                                       // (uniform over the CTA)
        for (int j = 0; j < p.nsel; j++)
            s_sum[j][tid] = s_cnt[j][tid] = 0;

        uint32_t key = 0xFFFFFFFFu, run = 0;
        auto flush = [&]() {
            if (!run)
                return;
            const uint32_t lc = key & 255u, hv = key >> 8;
            for (int q = 0; q < p.nplans; q++) {
                const AggPlan &P = p.plan[q];
                for (int g = 0; g < P.groups; g++) {
                    const uint32_t sg = soil_slot(hv, P.drained[g]);
                    const uint8_t *rec = P.rec_bytes == 16 ? P.lut + 16u * (lc * 8u + (sg ^ ((lc >> p.swz_shift) & 7u)))
                                                           : P.lut + 4u * (lc * kLut4Stride + sg);
                    for (int k = 0; k < P.np; k++) {
                        const uint32_t v = __ldg(rec + k);
                        if (v != GCN10_NODATA) {
                            const int j = P.acc[g * P.np + k];
                            s_sum[j][tid] += run * v;
                            s_cnt[j][tid] += run;
                        }
                    }
                }
            }
        };
        for (int y = lo; y < hi; y++) {
            const uint8_t *row = p.esa + (size_t)(y - p.y0) * p.esa_pitch;
            const int hr = __ldg(p.row_idx + y);
            if (hr != hrow) {
                // a new HSG row (every ~25 rows): gather the segment's soil codes once
                hrow = hr;
                const uint8_t *hs = p.hsg + (size_t)hr * p.hsg_pitch;
                for (int x = xa; x < xb; x++)
                    s_soil[x - xa][tid] = __ldg(hs + __ldg(p.col_idx + x));
            }
            for (int x = xa; x < xb; x++) {
                const uint32_t k2 = (uint32_t)__ldg(row + x) | ((uint32_t)s_soil[x - xa][tid] << 8);
                if (k2 != key) {
                    flush();
                    key = k2;
                    run = 0;
                }
                run++;
            }
        }
        flush();
        __syncthreads();
        if (active && sub == 0) {
            for (int j = 0; j < p.nsel; j++) {
                uint32_t s = 0, n = 0;
                for (int t = tid; t < tid + p.spc; t++) {
                    s += s_sum[j][t];
                    n += s_cnt[j][t];
                }
                if (n) {
                    uint2 *a = p.acc + ((size_t)j * p.ch + cr) * p.cw + cx;
                    atomicAdd(&a->x, s);
                    atomicAdd(&a->y, n);
                }
            }
        }
        __syncthreads();
    }
}

struct AggFinishParams {
    uint2 *acc;                     // [nsel][ch][cw]
    uint8_t *out;                   // plane j at out + j * plane_stride, rows `pitch` apart
    size_t pitch, plane_stride;
    int cw, ch, nsel;
};

__global__ void __launch_bounds__(256) aggregate_finish_kernel(const __grid_constant__ AggFinishParams p)
{
    const long long cells = (long long)p.cw * p.ch, n = cells * p.nsel;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(i / cells);
        const long long r = i - j * cells;
        const int cy = (int)(r / p.cw), cx = (int)(r - (long long)cy * p.cw);
        const uint2 a = p.acc[i];
        p.out[(size_t)j * p.plane_stride + (size_t)cy * p.pitch + cx] = gcn10_aggregate_value(a.x, a.y);
        p.acc[i] = make_uint2(0, 0);
    }
}

}  // namespace gcn10
