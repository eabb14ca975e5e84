// gcn10_b200/csrc/stats.cuh -- option "stats" of the compressed-tile calls on the two-kernel path: the histograms of a
// strip's device planes (the fused path counts record ids inside cn_deflate_fused_kernel instead).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace gcn10 {

struct PlaneHistParams {
    const uint8_t *planes;          // the j-th selected plane of the strip at planes + j * plane_stride
    size_t plane_stride, pitch;     // (both multiples of 16, as the planes' base: 16-byte loads)
    int w, rows;                    // valid pixels: w x rows per plane
    int plane_ids[18];              // plane number of the j-th selected plane
    unsigned long long *hist;       // [18][256] pixels per plane and value, accumulated
};

// grid = (CTAs per plane, selected planes), 256 threads, four CTAs an SM; a CTA counts fewer than 2^32 pixels (the
// launch sizes the grid so).  Every warp keeps its own 32-bit histogram in shared memory, so that only lanes of one warp
// can meet on a bin; the CTA adds the eight to the global histogram once.  A thread counts 64 pixels of a row at a time
// (four 16-byte loads in flight): a word that continues the current run counts four pixels in one step, runs that end
// inside the 64 pixels go to the warp's histogram directly, and the run the 64 pixels end with is summed over the lanes
// of the warp that end with the same value and added by one of them.
__global__ void __launch_bounds__(256, 4) plane_histogram_kernel(const __grid_constant__ PlaneHistParams p)
{
    __shared__ uint32_t s_hw[8][256];
    for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x)
        s_hw[i >> 8][i & 255] = 0;
    __syncthreads();
    const int j = blockIdx.y, lane = threadIdx.x & 31;
    uint32_t *s_h = s_hw[threadIdx.x >> 5];
    const uint8_t *plane = p.planes + (size_t)j * p.plane_stride;
    const int chunks = (p.w + 63) >> 6;
    const int chunks32 = (chunks + 31) & ~31;      // whole warps run the loop: the warp-wide steps need every lane
    for (int y = blockIdx.x; y < p.rows; y += gridDim.x) {
        const uint4 *row = reinterpret_cast<const uint4 *>(plane + (size_t)y * p.pitch);
        for (int c = threadIdx.x; c < chunks32; c += blockDim.x) {
            uint32_t cur = 0, n = 0;
            if (c < chunks) {
                // (the pitch is a multiple of 256 >= w: all four loads stay inside the row; bytes from w on are skipped)
                const int nv = min(64, p.w - 64 * c);
                const uint4 v0 = row[4 * c], v1 = row[4 * c + 1], v2 = row[4 * c + 2], v3 = row[4 * c + 3];
                cur = v0.x & 255u;
                // four pixels from x0 = 64 c + base on
                auto word = [&](uint32_t wv, int base) {
                    if (base + 4 <= nv && wv == cur * 0x01010101u) {
                        n += 4;
                        return;
                    }
#pragma unroll
                    for (int b = 0; b < 4; b++) {
                        const uint32_t px = (wv >> (8 * b)) & 255u;
                        if (base + b < nv) {
                            if (px != cur) {
                                atomicAdd(&s_h[cur], n);
                                cur = px;
                                n = 0;
                            }
                            n++;
                        }
                    }
                };
                word(v0.x, 0), word(v0.y, 4), word(v0.z, 8), word(v0.w, 12);
                word(v1.x, 16), word(v1.y, 20), word(v1.z, 24), word(v1.w, 28);
                word(v2.x, 32), word(v2.y, 36), word(v2.z, 40), word(v2.w, 44);
                word(v3.x, 48), word(v3.y, 52), word(v3.z, 56), word(v3.w, 60);
            }
            const unsigned same = __match_any_sync(0xffffffffu, cur);
            const unsigned total = __reduce_add_sync(same, n);
            if (total && lane == __ffs(same) - 1)
                atomicAdd(&s_h[cur], total);
        }
    }
    __syncthreads();
    unsigned long long v = 0;
#pragma unroll
    for (int wv = 0; wv < 8; wv++)
        v += s_hw[wv][threadIdx.x];
    if (v)
        atomicAdd(p.hist + (size_t)p.plane_ids[j] * 256 + threadIdx.x, v);
}

}  // namespace gcn10
