// gcn10_b200/csrc/overviews.cuh -- nearest-neighbour overview levels of a block's land cover (sm_100a).
//
// A block's Curve Number planes are a function of (land cover byte, HSG cell) per pixel, so overview level k of
// every plane is the fused encoder run on the land cover and index maps sampled by the rule of gcn10_overview_src
// (include/gcn10_cuda.h): esa_k[i][j] = esa[R_k(i)][C_k(j)], row_idx_k[i] = row_idx[R_k(i)], col_idx_k[j] =
// col_idx[C_k(j)].  An overview pixel is then a full-resolution output pixel, bit for bit.  This kernel builds
// those inputs strip by strip, while the strip's land cover is on the device anyway: one launch per full-resolution
// strip writes, for every level, the level rows whose source row lies in the strip.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gcn10_cuda.h"

namespace gcn10 {

struct OverviewLevel {
    uint8_t *esa;                   // level land cover, row 0 = level row 0
    int32_t *col_idx;               // [roundup16(w)]
    int32_t *row_idx;               // [level rows]
    size_t pitch;                   // multiple of 256
    int w;
    int k;                          // reduction 2^k
    int i_lo, i_hi;                 // level rows this strip holds the source of
};

struct OverviewParams {
    const uint8_t *src;             // the strip's land cover; row 0 = block row src_y0
    size_t src_pitch;
    int src_y0;
    int w, h;                       // the block
    const int32_t *col_idx;         // the block's maps
    const int32_t *row_idx;
    int with_cols;                  // the strip holds block row 0: write the column maps too
    int nlev;
    OverviewLevel lv[GCN10_MAX_OVERVIEWS];
};

// grid (x, nlev): blockIdx.y is the level; each thread writes four level pixels with one 32-bit store (the level
// pitch is a multiple of 256, so the bytes past the level's width stay inside the row)
__global__ void __launch_bounds__(256) overview_decimate_kernel(const OverviewParams p)
{
    const OverviewLevel &L = p.lv[blockIdx.y];
    const int k = L.k;
    const int words = (L.w + 3) >> 2;
    const long long n = (long long)(L.i_hi - L.i_lo) * words;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long t = t0; t < n; t += stride) {
        const int i = L.i_lo + (int)(t / words);
        const int j = (int)(t % words) * 4;
        const uint8_t *row = p.src + (size_t)(gcn10_overview_src(i, k, p.h) - p.src_y0) * p.src_pitch;
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; b++)
            v |= (uint32_t)__ldg(row + gcn10_overview_src(j + b, k, p.w)) << (8 * b);
        *reinterpret_cast<uint32_t *>(L.esa + (size_t)i * L.pitch + j) = v;
    }
    for (long long i = L.i_lo + t0; i < L.i_hi; i += stride)
        L.row_idx[i] = __ldg(p.row_idx + gcn10_overview_src((int)i, k, p.h));
    if (p.with_cols) {
        const int wpad = (L.w + 15) & ~15;
        for (long long j = t0; j < wpad; j += stride)
            L.col_idx[j] = __ldg(p.col_idx + gcn10_overview_src((int)j, k, p.w));
    }
}

}  // namespace gcn10
