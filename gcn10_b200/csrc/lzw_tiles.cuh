// gcn10_b200/csrc/lzw_tiles.cuh -- GPU-side decode of LZW-compressed GeoTIFF tiles (TIFF Compression 5, sm_100a).
//
// The LZW twin of inflate_tiles_kernel: same parameters (InflateParams: one launch covers every part of a window, window
// clipping with scratch copies, sparse tiles, a status per tile, longest streams first), same destination plane, same
// flush routine.  It is a kernel of its own so that the DEFLATE inflater compiles as before.
//
// One CTA = one tile = two warps:
//   decoder warp  tops up the 2 KB compressed-input ring; lane 0 reads the codes and turns them into batches of up to
//                 64 (output position, source) pairs (lzw_core.h), keeping the 4096-entry (start, length) table in
//                 shared memory.  The decoder never needs output bytes, so it runs ahead of the writer freely.
//   writer warp   produces the bytes of a batch, 8 per lane in flight: each byte follows its copy source back
//                 (lzw::resolve) to a literal, to the 8 KB history ring, or -- LZW strings reach back across the whole
//                 tile -- to the plane / scratch copy where earlier pieces were flushed; then it flushes the finished
//                 2 KB pieces of the ring with inflate_flush.  All bytes of a batch are independent of each other.
// The warps hand over through a double-buffered queue guarded by mbarriers.  Shared memory per CTA: ~35 KB (table
// 24 KB, history 8 KB, input ring 2 KB, queues 1 KB) -> six tiles per SM.
#pragma once

#include "inflate_tiles.cuh"
#include "lzw_core.h"

namespace gcn10 {

struct LzwSmem {
    uint32_t tstart[lzw::kCodes];
    uint16_t tlen[lzw::kCodes];
    uint32_t ring[inflate::kRingWords];
    uint32_t qpos[2][lzw::kBatch], qsrc[2][lzw::kBatch];
    int meta[2][4];                     // n, event, error, output position behind the batch
    unsigned long long bar_full[2], bar_empty[2];
    int final_err;
    int pad[3];
    uint8_t window[inflate::kWindow];
};

constexpr int kLzwSmem = (int)sizeof(LzwSmem);
constexpr int kLzwThreads = 64;         // decoder warp, writer warp
constexpr int kLzwUnroll = 8;           // bytes per lane in flight in the writer

__global__ void __launch_bounds__(kLzwThreads)
lzw_tiles_kernel(const __grid_constant__ InflateParams p)
{
    using namespace inflate;
    extern __shared__ __align__(16) uint8_t smem_lzw[];
    LzwSmem &sm = *reinterpret_cast<LzwSmem *>(smem_lzw);
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile = p.order ? p.order[blockIdx.x] : (int)blockIdx.x;
    int pi = 0;
    while (pi + 1 < p.nparts && tile >= p.part[pi + 1].first_tile)
        pi++;
    const InflatePart &pt = p.part[pi];
    const int local = tile - pt.first_tile;
    const int tx = local % pt.tiles_x, ty = local / pt.tiles_x;

    TileDst d;
    d.dst = pt.dst;
    d.pitch = p.pitch;
    d.dx0 = tx * pt.tile_w - pt.x_off;
    d.dy0 = ty * pt.tile_h - pt.y_off;
    d.w = pt.w;
    d.h = pt.h;
    d.tile_w = pt.tile_w;
    d.tw_shift = pt.tw_shift;
    d.rows16 = (pt.tile_w & 15) == 0;
    const int sidx = p.scratch_index ? p.scratch_index[tile] : -1;
    d.scratch = sidx >= 0;
    if (d.scratch) {
        d.hist = p.scratch + (size_t)sidx * (size_t)p.scratch_stride;
        d.hist_pitch = (size_t)pt.tile_w;
    }
    else {
        d.hist = pt.dst + (ptrdiff_t)d.dy0 * (ptrdiff_t)p.pitch + d.dx0;
        d.hist_pitch = p.pitch;
    }

    const uint32_t size = p.sizes[tile];
    if (size == 0) {
        const int x0 = max(d.dx0, 0), x1 = min(d.dx0 + pt.tile_w, pt.w);
        const int y0 = max(d.dy0, 0), y1 = min(d.dy0 + pt.tile_h, pt.h);
        for (int y = y0 + warp; y < y1; y += kLzwThreads / 32)
            for (int x = x0 + lane; x < x1; x += 32)
                pt.dst[(size_t)y * p.pitch + x] = 0;
        if (threadIdx.x == 0)
            p.status[tile] = 0;
        return;
    }

    const uint8_t *src = p.blob + p.offsets[tile];
    const uint8_t *base = reinterpret_cast<const uint8_t *>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)15);
    const uint32_t first = (uint32_t)(src - base);
    const uint32_t out_end = (uint32_t)pt.tile_w * (uint32_t)pt.tile_h;
    if (threadIdx.x == 0) {
        for (int k = 0; k < 2; k++) {
            mbar_init(smem_u32(&sm.bar_full[k]), 1);
            mbar_init(smem_u32(&sm.bar_empty[k]), 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == 0) {
        // ------------------------------------------------------------------ decoder warp
        uint32_t filled = 0;
        auto top_up = [&](uint32_t cons) {
            while (filled < cons + 1024u) {
                const uint4 v = __ldg(reinterpret_cast<const uint4 *>(base + filled) + lane);
                *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(sm.ring) + ((filled + 16u * lane) & 2047u)) = v;
                filled += 512u;
            }
            __syncwarp();
        };
        lzw::Lane s;
        top_up(first & ~3u);
        if (lane == 0)
            lzw::lane_init(s, sm.ring, first, size, out_end);
        int b = 0;
        for (uint32_t use = 0;; use++) {
            top_up(__shfl_sync(full, s.cons, 0));
            warp_wait(&sm.bar_empty[b], ((use >> 1) + 1u) & 1u);
            int ev = kEvMore;
            if (lane == 0) {
                const int n = lzw::decode_codes(s, sm.ring, sm.tstart, sm.tlen, sm.qpos[b], sm.qsrc[b], &ev);
                sm.meta[b][0] = n;
                sm.meta[b][1] = ev;
                sm.meta[b][2] = s.err;
                sm.meta[b][3] = (int)s.out;
            }
            ev = __shfl_sync(full, ev, 0);
            warp_signal(&sm.bar_full[b], lane);
            b ^= 1;
            if (ev != kEvMore)
                break;
        }
    }
    else {
        // ------------------------------------------------------------------ writer warp
        Ring window;
        window.base = (uint32_t)__cvta_generic_to_shared(sm.window);
        uint32_t b0 = 0, flushed = 0;
        int werr = 0, b = 0;
        for (uint32_t use = 0;; use++) {
            warp_wait(&sm.bar_full[b], (use >> 1) & 1u);
            const int n = sm.meta[b][0], ev = sm.meta[b][1];
            const uint32_t b1 = (uint32_t)sm.meta[b][3];
            if (ev == kEvError) {
                werr = sm.meta[b][2];
                break;
            }
            const uint32_t *qpos = sm.qpos[b], *qsrc = sm.qsrc[b];
            int k = 0;                  // this lane's code: its positions only grow
            for (uint32_t g = b0; g < b1; g += 32u * kLzwUnroll) {
                uint32_t r[kLzwUnroll];
#pragma unroll
                for (int u = 0; u < kLzwUnroll; u++) {
                    const uint32_t q = g + (uint32_t)lane + 32u * (uint32_t)u;
                    r[u] = lzw::kLit;
                    if (q < b1) {
                        while (k + 1 < n && qpos[k + 1] <= q)
                            k++;
                        r[u] = lzw::resolve(qpos, qsrc, n, b0, q, k);
                    }
                }
                uint32_t v[kLzwUnroll];
#pragma unroll
                for (int u = 0; u < kLzwUnroll; u++)
                    v[u] = (r[u] & lzw::kLit) ? (r[u] & 255u) : r[u] >= flushed ? window.ld8(r[u]) : hist_byte(d, r[u]);
#pragma unroll
                for (int u = 0; u < kLzwUnroll; u++) {
                    const uint32_t q = g + (uint32_t)lane + 32u * (uint32_t)u;
                    if (q < b1)
                        window.st8(q, v[u]);
                }
            }
            __syncwarp();
            warp_signal(&sm.bar_empty[b], lane);
            b ^= 1;
            b0 = b1;
            // finished pieces -> plane (and scratch copy); later batches read them back from there
            while (flushed + kFlushChunk <= b0) {
                inflate_flush(sm.window, d, flushed, kFlushChunk, lane);
                flushed += kFlushChunk;
                __syncwarp();
            }
            if (ev == kEvEnd)
                break;
        }
        if (!werr && flushed < out_end)
            inflate_flush(sm.window, d, flushed, out_end - flushed, lane);
        if (lane == 0)
            sm.final_err = werr;
    }
    __syncthreads();
    if (threadIdx.x == 0)
        p.status[tile] = sm.final_err;
}

}  // namespace gcn10
