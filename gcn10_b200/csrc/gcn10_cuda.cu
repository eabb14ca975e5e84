// gcn10_b200/csrc/gcn10_cuda.cu -- host side of libgcn10cuda.so (C ABI in include/gcn10_cuda.h).
//
// Replaces the per-pixel part of the reference's process_block() (/root/reference/src/cn.c:208-290):
// upload of the two windows that load_raster() produced, the fp64 index maps, the fused
// resample + remap + lookup kernel, and download of the planes that go to save_raster().
//
// There is deliberately no CPU implementation in this file: if CUDA is unavailable every
// compute entry point returns an error.
#include "../../include/gcn10_cuda.h"
#include "cn_kernels.cuh"
#include "deflate_tiles.cuh"
#include "inflate_tiles.cuh"
#include "lzw_tiles.cuh"
#include "cn_deflate_fused.cuh"
#include "aggregate.cuh"
#include "overviews.cuh"
#include "stats.cuh"
#include "tile_code.h"

#include <algorithm>
#include <cctype>
#include <sched.h>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <new>
#include <vector>

using namespace gcn10;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t e_ = (expr);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return fail(e_ == cudaErrorMemoryAllocation ? GCN10_ENOMEM : GCN10_ECUDA,        \
                        "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__);\
    } while (0)

constexpr int kMaxStreams = 8;

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct HostBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct StripSlot {
    DevBuf esa;
    DevBuf out;                 // nplanes * strip_rows * pitch
    cudaEvent_t k0 = nullptr, k1 = nullptr, done = nullptr;
    cudaEvent_t k2 = nullptr;   // tile-deflate path: behind everything the strip computes (encoder + re-ordering kernels)
    bool timed = false;
    // tile-deflate path
    DevBuf blob, table;         // compressed tiles; [cursor(16 B) | offsets u64[] | sizes u32[]]
    DevBuf blob2, order;        // option "ordered": the strip re-laid in table order, and the scan's offsets
    HostBuf h_blob, h_table;    // page-locked mirrors
    cudaEvent_t enc_done = nullptr;
    cudaEvent_t ov = nullptr;   // option "overviews": behind the strip's overview_decimate_kernel
    cudaEvent_t ag = nullptr;   // option "aggregate": behind the strip's aggregate_accumulate_kernel
    int y0 = 0, rows = 0;
    int level = 0, y_base = 0, tiles_x = 0, level_w = 0, level_h = 0;     // what the strip reports to the sink
    int agg = 0;                // ... and the factor of a mean-raster strip (0 = a Curve Number strip)
    bool busy = false;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

}  // namespace

// one compressed land-cover window on its way to / resident on the device (two per context, so that the next
// block's tiles can be uploaded and inflated while the current block's strips run: gcn10_cuda_tiles_prefetch)
struct TileSlot {
    DevBuf in_blob, in_table, esa_full, scratch;   // scratch: whole-tile copies of the tiles the window clips
    HostBuf h_status;           // [ntiles] status codes | launch order | offsets (u64) | sizes (u32): page-locked staging
    cudaEvent_t inf0 = nullptr, inf1 = nullptr, done = nullptr;     // around the inflate kernel; behind the status copy
    bool pending = false;       // inflate issued, result not consumed yet
    bool deferred = false;      // ... uploads issued, the kernel waits for the strips of the block in hand (launch_inflate)
    InflateParams ip;           // the deferred launch
    size_t n_lzw = 0;           // LZW tiles: the last n_lzw entries of the launch order, decoded by lzw_tiles_kernel
    uint64_t seq = 0;           // issue order of pending slots
    const void *key_blob = nullptr, *key_off = nullptr;
    size_t key_bytes = 0, ntiles = 0, dpitch = 0;
    int key_w = 0, key_h = 0, key_parts = 0;
};

struct gcn10_ctx {
    int device = -1;
    int sm_count = 148;
    cudaStream_t streams[kMaxStreams] = {};
    cudaStream_t ship_streams[kMaxStreams] = {};    // high priority: ship_strip_kernel of the slot with the same index
    int nstreams = 8;
    int strip_rows = 2048;
    int rows_per_cta = 0;       // 0 = auto (see auto_rows_per_cta)
    int use_tma = 1;
    int inflate_probe = 0;      // measurement aid for tools/inflate_bench.py (see InflateParams::probe)
    int fused = 1;              // compressed-tile calls use cn_deflate_fused_kernel (0 = CN kernel + tile encoder)
    int ordered = 0;            // 1 = strips are re-laid in table order before they leave the device
    int cog = 0;                // 1 = Cloud Optimized GeoTIFF order: overview levels first, smallest first; with
                                // "ordered" every tile also gets its block leader and trailer on the device
    int ship = 0;               // 1 = strips leave through ship_strip_kernel; 0 = size read-back, then a D2H copy of that size
                                // (measured on B200: 11.8 vs 12.2 ms per block -- the copy engine does not compete for SMs)
    DevBuf fused_tab;           // idmap [256][16] | val [256][32] | lit9 [256][6] u64
    unsigned fused_mask = 0;    // plane mask the tables were built for (0 = none)
    int fused_ok = 0;           // the mask's value records fit the id space
    uint8_t fused_cls[18] = {}; // 9-bit-literal class of the j-th selected plane
    int tuned_code = 1;         // tile streams use the tuned Huffman code of tile_code.h (0 = RFC 1951 fixed code)
    FusedCode fused_code = {};  // header_bits == 0: fixed code
    EncodeTiledFn encode_tiled = nullptr;

    bool have_lut = false;
    int host_tables[GCN10_NVARIANTS][256][5];
    DevBuf lut;                 // packed records for the current plane selection
    unsigned lut_mask[2] = { 0xFFFFFFFFu, 0xFFFFFFFFu };   // variant masks the records were packed for
    int swz_shift = 1;

    DevBuf col_idx, row_idx, hsg;
    StripSlot slots[kMaxStreams];
    // compressed-input path: the tiles' bytes, their tables and the inflated land-cover plane of a block
    TileSlot tslot[2];
    cudaStream_t pre_stream = nullptr;      // uploads + inflate kernels
    int defer_inflate = 1;                  // option: hold a prefetched block's inflate kernel back (launch_inflate)
    uint64_t tile_seq = 0;
    float last_inflate_ms = 0.f;
    float last_kernel_ms = 0.f;
    uint64_t launches = 0;
    // options "overviews" and "stats" gather the block in hand strip by strip, and band by band: blk_next is the block
    // row the next band must start at (-1 = no block open), blk_w x blk_h and blk_mask what the block's first band had
    int blk_w = 0, blk_h = 0, blk_next = -1;
    unsigned blk_mask = 0;
    // option "overviews": the land cover and index maps of every overview level of the block in hand
    int overviews = 0;
    DevBuf ov_buf;
    OverviewLevel ov_lv[GCN10_MAX_OVERVIEWS] = {};
    int ov_h[GCN10_MAX_OVERVIEWS] = {};
    // option "stats": the block's pixel counts on the device, [256] per record id (fused path) | [18][256] per plane and
    // value (two-kernel path); the last completed block's histograms on the host (gcn10_cuda_last_histograms)
    int stats = 0;
    DevBuf stats_buf;
    bool blk_fused = false;             // a strip of the block in hand counted record ids
    bool stats_ready = false;
    uint64_t stats_hist[GCN10_NPLANES][256] = {};
    uint8_t fused_rec[kFusedIds][GCN10_NPLANES] = {};  // value record of every id of the fused tables (fused_mask)
    // option "aggregate": the block's per-cell (sum, count) accumulators [selected planes][ch][cw], all zero between
    // blocks (agg_clean), and the mean rasters the finish kernel makes of them [selected planes][ch][pitch]
    int aggregate = 0;
    DevBuf agg_acc, agg_out;
    bool agg_clean = false;
    cudaEvent_t agg_ready = nullptr;    // behind aggregate_finish_kernel
    // asynchronous raw-plane blocks (gcn10_cuda_block_async): frame guard, per-stream end-of-block marks, timer events
    cudaEvent_t frame_ready = nullptr;
    cudaEvent_t tail[kMaxStreams] = {};
    bool tail_valid[kMaxStreams] = {};
    int pending_events = 0;             // blocks queued by gcn10_cuda_block_async and not yet waited for
    std::vector<cudaEvent_t> timer_pool;
};

struct gcn10_event {
    gcn10_ctx *ctx = nullptr;
    int nstreams = 0;
    int status = 0;                     // error met while queueing (reported by gcn10_cuda_wait)
    std::vector<cudaEvent_t> timers;    // kernel start / end per strip
    std::vector<cudaEvent_t> ends;      // behind the block's last copy, per stream
};

namespace {

int ensure(DevBuf &b, size_t bytes)
{
    if (b.cap >= bytes && b.p)
        return GCN10_OK;
    if (b.p)
        cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
    CUDA_TRY(cudaMalloc(&b.p, bytes));
    b.cap = bytes;
    return GCN10_OK;
}

void release(DevBuf &b)
{
    if (b.p)
        cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

int ensure_host(HostBuf &b, size_t bytes)
{
    if (b.cap >= bytes && b.p)
        return GCN10_OK;
    if (b.p)
        cudaFreeHost(b.p);
    b.p = nullptr;
    b.cap = 0;
    CUDA_TRY(cudaHostAlloc(&b.p, bytes, cudaHostAllocPortable));
    b.cap = bytes;
    return GCN10_OK;
}

void release_host(HostBuf &b)
{
    if (b.p)
        cudaFreeHost(b.p);
    b.p = nullptr;
    b.cap = 0;
}

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// (uint8_t)v when v < 255, else 255: what calculate_cn() leaves in a plane prefilled with 255
// (cn.c:126-128,289)
inline uint8_t cn_byte(int v) { return v < 255 ? (uint8_t)v : (uint8_t)GCN10_NODATA; }

int popcount9(unsigned m) { return __builtin_popcount(m & 0x1FFu); }

// Pick the bank-swizzle shift: spread the land-cover classes that actually have table rows over
// the 8 16-byte bank groups of shared memory, so that neighbouring pixels of different classes
// (same soil group) do not serialise their record fetches.
int choose_swizzle(const int tables[GCN10_NVARIANTS][256][5])
{
    bool live[256];
    for (int lc = 0; lc < 256; lc++) {
        live[lc] = false;
        for (int t = 0; t < GCN10_NVARIANTS && !live[lc]; t++)
            for (int s = 0; s < 5; s++)
                if (tables[t][lc][s] < 255) {
                    live[lc] = true;
                    break;
                }
    }
    int best = 0, best_cost = 1 << 30;
    for (int sh = 0; sh <= 5; sh++) {
        int cnt[8] = { 0 };
        for (int lc = 0; lc < 256; lc++)
            if (live[lc])
                cnt[(lc >> sh) & 7]++;
        int cost = 0;
        for (int g = 0; g < 8; g++)
            cost += cnt[g] * cnt[g];
        if (cost < best_cost) {
            best_cost = cost;
            best = sh;
        }
    }
    return best;
}

// Record (lc, slot') = the CN bytes of the selected variants, in selection order, for land cover
// lc and soil-group slot s = slot' ^ ((lc >> shift) & 7).  Slots 5..7 (invalid soil group, cn.c:123-124)
// hold 255 everywhere.
// With at most kNarrowPlanes selected variants the records are 4 bytes, rows kLut4Stride words apart, no swizzle.
void pack_lut_records(const int tables[GCN10_NVARIANTS][256][5], unsigned variant_mask, int shift,
                      std::vector<uint8_t> &rec)
{
    const bool narrow = popcount9(variant_mask) <= kNarrowPlanes;
    rec.assign((size_t)kLutBytes, (uint8_t)GCN10_NODATA);
    for (int lc = 0; lc < 256; lc++) {
        for (int s = 0; s < 5; s++) {
            int slot = s ^ ((lc >> shift) & 7);
            uint8_t *r = narrow ? &rec[((size_t)lc * kLut4Stride + s) * 4] : &rec[((size_t)lc * 8 + slot) * 16];
            int k = 0;
            for (int t = 0; t < GCN10_NVARIANTS; t++)
                if (variant_mask & (1u << t))
                    r[k++] = cn_byte(tables[t][lc][s]);
        }
    }
}

// Rows each CTA walks.  Measured on B200 (profiles/r01_kernel_sweeps.md): short chunks keep the
// co-resident CTAs inside a narrow band of rows and leave no tail wave, long ones amortise the per-CTA
// prologue (LUT + HSG box fills).  Bulk-store kernel: 12 rows is best for <= 9 planes (2 CTAs/SM), 32 for
// 10..18 planes (1 CTA/SM); direct-store kernel: 12 / 16.
int auto_rows_per_cta(int planes) { return planes > 9 ? (GCN10_BULK_STORE ? 32 : 16) : planes <= kNarrowPlanes ? 32 : 12; }

// ---- strip hand-over ------------------------------------------------------------------------

// A strip's compressed tiles leave the device without a host round trip: this kernel runs behind the encoder on
// the strip's stream, reads the arena's fill level where the encoder left it and writes exactly that many bytes,
// plus the offset / size tables, into page-locked host memory through its device mapping (coalesced 16-byte
// stores = posted PCIe writes).  The host only waits for the event behind it.  If the host arena is too small
// the copy stops at `h_cap`; the fill level in the table tells the host, which grows the arena and fetches the
// strip with a plain copy.
__global__ void __launch_bounds__(64)
ship_strip_kernel(const uint4 *__restrict__ blob, const unsigned long long *__restrict__ cursor,
                  const uint32_t *__restrict__ table, uint32_t table_words, uint4 *__restrict__ h_blob,
                  unsigned long long h_cap, uint32_t *__restrict__ h_table)
{
    const unsigned long long used = min(*cursor, h_cap);
    const size_t n16 = (size_t)((used + 15ull) >> 4);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride)
        h_blob[i] = blob[i];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < table_words; i += stride)
        h_table[i] = table[i];
}
// Small CTAs on a high-priority stream: 64 threads x <= 40 registers fit beside two resident CTAs of the fused
// encoder (2 x 256 threads x 120 registers leave 4096 registers per SM), so a strip starts to leave while the next
// strip's encoder already fills the SMs.
constexpr int kShipThreads = 64;
constexpr int kShipCtas = 2 * 148;

// ---- ordered strips -------------------------------------------------------------------------

// The encoders place a tile's streams wherever the arena's bump allocator stood when the tile's CTA finished.  With
// the option "ordered" the strip is re-laid in table order -- [plane][tile row][tile column], every stream on a
// 16-byte boundary -- before it leaves the device, so that the consumer can write a plane's share of the strip (or a
// whole tile row of it) to its GeoTIFF with ONE write instead of one per tile.  Two small kernels behind the
// encoder: an exclusive scan of the rounded sizes (one CTA) and a warp-per-tile copy.  The total is unchanged.
//
// FRAMED (options "cog" and "ordered"): every stream also gets the block leader and trailer of a Cloud Optimized
// GeoTIFF -- its byte count as a uint32 LE in the 4 bytes before it, its last 4 bytes repeated after it.  A tile's slot
// is round16(size + 8): [stream | trailer | zero padding | the NEXT tile's leader], and the first tile's leader sits
// in the strip's first 16 bytes, so every stream still starts on a 16-byte boundary and the uint4 copy stays.  The
// total changes: the scan writes it to the word `cursor` points at (the table's second 8 bytes), 0 when the re-laid
// strip does not fit the second arena.
template <bool FRAMED>
__device__ __forceinline__ unsigned long long laid_bytes(uint32_t size)
{
    return ((unsigned long long)size + (FRAMED ? 8ull : 0ull) + 15ull) & ~15ull;
}

template <bool FRAMED>
__global__ void __launch_bounds__(1024)
order_scan_kernel(const uint32_t *__restrict__ sizes, int n, unsigned long long *__restrict__ new_off,
                  unsigned long long *__restrict__ cursor, unsigned long long cap2)
{
    if (!FRAMED && *cursor > cap2)
        return;                 // the strip does not fit the second arena: it leaves unordered
    __shared__ unsigned long long s_part[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + 1023) / 1024;
    const int i0 = tid * per, i1 = min(n, i0 + per);
    unsigned long long sum = 0;
    for (int i = i0; i < i1; i++)
        sum += laid_bytes<FRAMED>(sizes[i]);
    unsigned long long inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o)
            inc += t;
    }
    if (lane == 31)
        s_part[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        unsigned long long v = s_part[lane], w = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o)
                w += t;
        }
        s_part[lane] = w - v;
    }
    __syncthreads();
    unsigned long long at = s_part[warp] + inc - sum + (FRAMED ? 16ull : 0ull);
    for (int i = i0; i < i1; i++) {
        new_off[i] = at;
        at += laid_bytes<FRAMED>(sizes[i]);
    }
    if (FRAMED && tid == 1023)
        *cursor = at <= cap2 ? at : 0ull;
}

template <bool FRAMED>
__global__ void __launch_bounds__(256)
order_copy_kernel(const uint8_t *__restrict__ blob, unsigned long long *__restrict__ offsets, const uint32_t *__restrict__ sizes,
                  const unsigned long long *__restrict__ new_off, uint8_t *__restrict__ blob2, int n,
                  const unsigned long long *__restrict__ cursor, unsigned long long cap2)
{
    if (FRAMED ? *cursor == 0ull : *cursor > cap2)
        return;
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
        const uint4 *src = reinterpret_cast<const uint4 *>(blob + offsets[i]);
        uint4 *dst = reinterpret_cast<uint4 *>(blob2 + new_off[i]);
        const uint32_t size = sizes[i];
        const uint32_t n16 = FRAMED ? size >> 4 : (size + 15u) >> 4;
        for (uint32_t k = lane; k < n16; k += 32u)
            dst[k] = src[k];
        if (FRAMED) {
            // the slot's last one or two words: the stream's tail, the trailer, zeros, the next tile's leader
            const uint8_t *sb = blob + offsets[i];
            const uint32_t end = (uint32_t)laid_bytes<true>(size);
            const uint32_t lead = i + 1 < n ? sizes[i + 1] : 0u;
            for (uint32_t k = n16 + lane; k < end >> 4; k += 32u) {
                uint32_t v[4];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    v[q] = 0u;
#pragma unroll
                    for (int b = 0; b < 4; b++) {
                        const uint32_t p = k * 16u + (uint32_t)(q * 4 + b);
                        const uint32_t byte = p < size + 4u ? (uint32_t)sb[p < size ? p : p - 4u]
                                              : p >= end - 4u ? (lead >> (8u * (p - (end - 4u)))) & 255u : 0u;
                        v[q] |= byte << (8 * b);
                    }
                }
                dst[k] = make_uint4(v[0], v[1], v[2], v[3]);
            }
            if (i == 0 && lane == 0)
                reinterpret_cast<uint4 *>(blob2)[0] = make_uint4(0u, 0u, 0u, size);     // the first tile's leader
        }
        __syncwarp();
        if (lane == 0)
            offsets[i] = new_off[i];
    }
}

// ---- kernel dispatch ------------------------------------------------------------------------

typedef void (*BlockKernel)(const BlockParams, const CUtensorMap);

template <int NP>
BlockKernel pick_g(int groups)
{
    return groups == 2 ? (BlockKernel)cn_block_kernel<NP, 2> : (BlockKernel)cn_block_kernel<NP, 1>;
}

BlockKernel pick_kernel(int np, int groups)
{
    switch (np) {
    case 1: return pick_g<1>(groups);
    case 2: return pick_g<2>(groups);
    case 3: return pick_g<3>(groups);
    case 4: return pick_g<4>(groups);
    case 5: return pick_g<5>(groups);
    case 6: return pick_g<6>(groups);
    case 7: return pick_g<7>(groups);
    case 8: return pick_g<8>(groups);
    case 9: return pick_g<9>(groups);
    }
    return nullptr;
}

struct LaunchPlan {
    int np = 0, groups = 0;     // planes per group, number of groups in this launch
    int drained[2] = { 1, 0 };
    unsigned variant_mask = 0;  // variants (bits 0..8) the LUT records must be packed for
    int plane_ids[18];          // original plane index of each compacted output
};

// Split a plane mask into launches.  Both drainage conditions share one launch (one read of the
// land cover) when they ask for the same variants; otherwise each condition gets its own.
int plan_launches(unsigned plane_mask, LaunchPlan plans[2])
{
    unsigned md = plane_mask & 0x1FFu, mu = (plane_mask >> 9) & 0x1FFu;
    int n = 0;
    auto fill = [](LaunchPlan &lp, unsigned vm, int g0_drained, int groups) {
        lp.np = popcount9(vm);
        lp.groups = groups;
        lp.variant_mask = vm;
        lp.drained[0] = g0_drained;
        lp.drained[1] = 0;
        int k = 0;
        for (int g = 0; g < groups; g++) {
            int cond = (groups == 2) ? g : (g0_drained ? 0 : 1);
            for (int t = 0; t < 9; t++)
                if (vm & (1u << t))
                    lp.plane_ids[k++] = cond * 9 + t;
        }
    };
    if (md && md == mu) {
        fill(plans[n++], md, 1, 2);
    }
    else {
        if (md)
            fill(plans[n++], md, 1, 1);
        if (mu)
            fill(plans[n++], mu, 0, 1);
    }
    return n;
}

int upload_lut(gcn10_ctx *c, unsigned variant_mask, int slot, cudaStream_t st)
{
    // two cached record sets (one per launch of a split plan)
    if (c->lut_mask[slot] == variant_mask)
        return GCN10_OK;
    int rc = ensure(c->lut, 2 * (size_t)kLutBytes);
    if (rc)
        return rc;
    std::vector<uint8_t> rec;
    pack_lut_records(c->host_tables, variant_mask, c->swz_shift, rec);
    // synchronous w.r.t. the host vector's lifetime
    CUDA_TRY(cudaMemcpyAsync((uint8_t *)c->lut.p + (size_t)slot * kLutBytes, rec.data(), kLutBytes,
                             cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    c->lut_mask[slot] = variant_mask;
    return GCN10_OK;
}

int make_hsg_map(gcn10_ctx *c, const uint8_t *d_hsg, int hsx, int hsy, size_t pitch, CUtensorMap *map, int *usable)
{
    *usable = 0;
    memset(map, 0, sizeof(*map));
    if (!c->use_tma || !c->encode_tiled)
        return GCN10_OK;
    if (((uintptr_t)d_hsg & 15u) || (pitch & 15u) || hsy < 1 || hsx < 1)
        return GCN10_OK;        // TMA needs a 16-byte aligned base and row stride
    cuuint64_t dims[2] = { (cuuint64_t)hsx, (cuuint64_t)hsy };
    cuuint64_t strides[1] = { (cuuint64_t)pitch };
    cuuint32_t box[2] = { (cuuint32_t)kBoxCols, (cuuint32_t)kBoxRows };
    cuuint32_t estr[2] = { 1, 1 };
    CUresult r = c->encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)d_hsg, dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                 CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_SUCCESS)
        *usable = 1;
    return GCN10_OK;
}

int launch_index_maps(gcn10_ctx *c, int w, int h, const double gt[6], int hsx, int hsy, const double sgt[6],
                      cudaStream_t st)
{
    int w_pad = (int)round_up((size_t)w, kVecPx);
    int rc = ensure(c->col_idx, sizeof(int32_t) * (size_t)w_pad);
    if (rc)
        return rc;
    rc = ensure(c->row_idx, sizeof(int32_t) * (size_t)h);
    if (rc)
        return rc;
    int n = w_pad + h;
    index_map_kernel<<<(n + 255) / 256, 256, 0, st>>>(w, w_pad, h, gt[0], gt[1], gt[3], gt[5],
                                                      sgt[0], sgt[1], sgt[3], sgt[5], hsx, hsy,
                                                      (int32_t *)c->col_idx.p, (int32_t *)c->row_idx.p);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return GCN10_OK;
}

// Launch the fused kernel(s) for `rows` rows starting at block row y_base.  d_out holds the 18
// plane pointers already offset to the first row of this launch.
int launch_rows(gcn10_ctx *c, const LaunchPlan &lp, int lut_slot, const uint8_t *d_esa, size_t esa_pitch, int w,
                int rows, int y_base, const uint8_t *d_hsg, size_t hsg_pitch, int hsx, int hsy,
                const CUtensorMap &map, int tma_ok, uint8_t *const d_out[GCN10_NPLANES], size_t out_pitch,
                cudaStream_t st, const int32_t *col_idx = nullptr, const int32_t *row_idx = nullptr)
{
    BlockParams p;
    memset(&p, 0, sizeof(p));
    p.esa = d_esa;
    p.esa_pitch = esa_pitch;
    p.w = w;
    p.h = rows;
    p.y_base = y_base;
    p.col_idx = col_idx ? col_idx : (const int32_t *)c->col_idx.p;      // (an overview level's maps, or the block's)
    p.row_idx = row_idx ? row_idx : (const int32_t *)c->row_idx.p;
    p.hsg = d_hsg;
    p.hsg_pitch = hsg_pitch;
    p.hsx = hsx;
    p.hsy = hsy;
    p.lut = (const uint4 *)((const uint8_t *)c->lut.p + (size_t)lut_slot * kLutBytes);
    p.rec_bytes = lp.np <= kNarrowPlanes ? 4 : 16;
    p.swz_shift = c->swz_shift;
    p.rows_per_cta = c->rows_per_cta > 0 ? c->rows_per_cta : auto_rows_per_cta(lp.np * lp.groups);
    p.use_tma = tma_ok;
    p.group_drained[0] = lp.drained[0];
    p.group_drained[1] = lp.drained[1];
    p.out_pitch = out_pitch;
    bool aligned = (((uintptr_t)d_esa | esa_pitch | out_pitch) & 15u) == 0;
    for (int k = 0; k < lp.np * lp.groups; k++) {
        p.out[k] = d_out[lp.plane_ids[k]];
        if (!p.out[k])
            return fail(GCN10_EINVAL, "output plane %d selected by the mask but its pointer is NULL", lp.plane_ids[k]);
        if ((uintptr_t)p.out[k] & 15u)
            aligned = false;
    }

    int x_bytes = 0;
    if (aligned && (w & ~(kVecPx - 1)) > 0) {
        int w16 = w & ~(kVecPx - 1);
        while ((rows + p.rows_per_cta - 1) / p.rows_per_cta > 65535)     // gridDim.y limit, only for absurdly tall rasters
            p.rows_per_cta *= 2;
        dim3 grid((w16 + kStripPx - 1) / kStripPx, (rows + p.rows_per_cta - 1) / p.rows_per_cta);
        BlockKernel k = pick_kernel(lp.np, lp.groups);
        k<<<grid, kThreads, smem_bytes_for(lp.np, lp.groups), st>>>(p, map);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        x_bytes = w16;
    }
    if (x_bytes < w) {
        long long n = (long long)(w - x_bytes) * rows;
        int blocks = (int)std::min<long long>((n + 255) / 256, (long long)c->sm_count * 16);
        cn_bytes_kernel<<<blocks, 256, 0, st>>>(p, x_bytes, lp.np, lp.groups);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    return GCN10_OK;
}

// The value record of a (land cover, soil class) pair = its Curve Number in every selected plane
// (cn.c:88-131: dual-group remap per drainage condition, table lookup, 255 for anything else).  Distinct
// records get ids 0..254; id 255 is the all-zero record of the tile padding.  Fails (fused_ok = 0) when
// the tables hold more than 255 distinct records; the two-kernel path is used then.
int build_fused_tables(gcn10_ctx *c, unsigned plane_mask, cudaStream_t st)
{
    if (c->fused_mask == plane_mask)
        return GCN10_OK;
    int plane_ids[GCN10_NPLANES], nsel = 0;
    for (int k = 0; k < GCN10_NPLANES; k++)
        if (plane_mask & (1u << k))
            plane_ids[nsel++] = k;
    const int valb = nsel <= 9 ? 16 : 32;
    std::vector<uint8_t> host(4096 + kFusedIds * 32 + kFusedIds * 8 + sizeof(TileCode::header_words) + 256, 0);
    uint8_t *idmap = host.data(), *val = host.data() + 4096;
    unsigned long long *lit9 = (unsigned long long *)(host.data() + 4096 + kFusedIds * 32);
    std::vector<std::vector<uint8_t>> records;
    c->fused_ok = 1;
    for (int lc = 0; lc < 256 && c->fused_ok; lc++) {
        for (int sc = 0; sc < 16; sc++) {
            std::vector<uint8_t> rec((size_t)nsel, (uint8_t)GCN10_NODATA);
            // soil class -> raw code: 0, 1..4, 11..14, anything else
            const int code = sc <= 4 ? sc : (sc <= 8 ? 11 + (sc - 5) : 255);
            for (int j = 0; j < nsel && sc <= 9; j++) {
                const int cond = plane_ids[j] / 9, t = plane_ids[j] % 9;
                int sg = code;
                if (code >= 11 && code <= 14)
                    sg = cond == 0 ? 4 : code - 10;         // drained: 11..14 -> 4; undrained: 11->1 .. 14->4 (cn.c:92-109)
                if (sg < 5)
                    rec[j] = cn_byte(c->host_tables[t][lc][sg]);
            }
            size_t id = 0;
            while (id < records.size() && records[id] != rec)
                id++;
            if (id == records.size()) {
                if (records.size() >= (size_t)kFusedPad) {
                    c->fused_ok = 0;
                    break;
                }
                records.push_back(rec);
            }
            idmap[sc * 256 + lc] = (uint8_t)id;
        }
    }
    // planes whose records need 9-bit literals (values >= 144, in practice nodata 255) at the same ids share
    // one bit-position counter in the kernel; at most kFusedClasses distinct patterns are supported
    // the tuned Huffman code: every byte value a plane can hold (table values, nodata, the zero padding)
    bool present[256] = { false };
    present[0] = true;
    for (size_t id = 0; id < records.size(); id++)
        for (int j = 0; j < nsel; j++)
            present[records[id][j]] = true;
    TileCode tc;
    memset(&c->fused_code, 0, sizeof(c->fused_code));
    const bool tuned = c->fused_ok && c->tuned_code && build_tile_code(present, tc);
    std::vector<std::vector<uint8_t>> patterns;
    memset(c->fused_cls, 0, sizeof(c->fused_cls));
    for (int j = 0; j < nsel && c->fused_ok && !tuned; j++) {
        std::vector<uint8_t> pat(records.size());
        for (size_t id = 0; id < records.size(); id++)
            pat[id] = records[id][j] >= 144;
        size_t q = 0;
        while (q < patterns.size() && patterns[q] != pat)
            q++;
        if (q == patterns.size()) {
            if (patterns.size() >= (size_t)kFusedClasses) {
                c->fused_ok = 0;
                break;
            }
            patterns.push_back(pat);
        }
        c->fused_cls[j] = (uint8_t)q;
    }
    if (c->fused_ok) {
        memset(c->fused_rec, 0, sizeof(c->fused_rec));
        for (size_t id = 0; id < records.size(); id++) {
            for (int j = 0; j < nsel; j++)
                val[id * valb + j] = c->fused_rec[id][j] = records[id][j];
            for (size_t q = 0; q < patterns.size() && !tuned; q++)      // (all literals equally long in the tuned code)
                if (patterns[q][id])
                    lit9[id] |= 1ull << (21 * q);
        }
        int rc = ensure(c->fused_tab, host.size());
        if (rc)
            return rc;
        if (tuned) {
            memset(c->fused_cls, 0, sizeof(c->fused_cls));
            uint8_t *hw = host.data() + 4096 + kFusedIds * 32 + kFusedIds * 8;
            memcpy(hw, tc.header_words, sizeof(tc.header_words));
            memcpy(hw + sizeof(tc.header_words), tc.lit_rank, 256);
            FusedCode &fc = c->fused_code;
            fc.header_bits = tc.header_bits;
            fc.lit_bits = tc.lit_bits;
            fc.lit_first = tc.lit_first;
            memcpy(fc.len_code, tc.len_code, sizeof(fc.len_code));
            memcpy(fc.len_bits, tc.len_bits, sizeof(fc.len_bits));
            fc.eob_code = tc.eob_code;
            fc.eob_bits = tc.eob_bits;
            memcpy(fc.dist_code, tc.dist_code, sizeof(fc.dist_code));
            memcpy(fc.dist_bits, tc.dist_bits, sizeof(fc.dist_bits));
            fc.header_words = (const uint32_t *)((const uint8_t *)c->fused_tab.p + 4096 + kFusedIds * 32 + kFusedIds * 8);
            fc.lit_rank = (const uint8_t *)c->fused_tab.p + 4096 + kFusedIds * 32 + kFusedIds * 8 + sizeof(tc.header_words);
        }
        CUDA_TRY(cudaMemcpyAsync(c->fused_tab.p, host.data(), host.size(), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    c->fused_mask = plane_mask;
    return GCN10_OK;
}

int check_geometry(const void *esa, int w, int h, size_t esa_pitch, const double *gt, const void *hsg, int hsx,
                   int hsy, size_t hsg_pitch, const double *sgt, unsigned mask, const void *out, size_t out_pitch)
{
    if (!esa || !hsg || !gt || !sgt || !out)
        return fail(GCN10_EINVAL, "NULL argument");
    if (w <= 0 || h <= 0 || hsx <= 0 || hsy <= 0)
        return fail(GCN10_EINVAL, "non-positive raster size (%d x %d, hsg %d x %d)", w, h, hsx, hsy);
    if (esa_pitch < (size_t)w || out_pitch < (size_t)w || hsg_pitch < (size_t)hsx)
        return fail(GCN10_EINVAL, "pitch smaller than row width");
    if ((mask & GCN10_MASK_ALL) == 0 || (mask & ~GCN10_MASK_ALL))
        return fail(GCN10_EINVAL, "plane mask 0x%x selects nothing or unknown planes", mask);
    return GCN10_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------

extern "C" {

const char *gcn10_cuda_version(void) { return "gcn10cuda 0.1.0 (sm_100a)"; }

const char *gcn10_cuda_last_error(void) { return g_err; }

int gcn10_cuda_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess)
        return fail(GCN10_ENODEV, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return n;
}

int gcn10_cuda_create(int device, gcn10_ctx **out)
{
    if (!out)
        return fail(GCN10_EINVAL, "NULL out pointer");
    *out = nullptr;
    int n = gcn10_cuda_device_count();
    if (n < 0)
        return n;
    if (device < 0 || device >= n)
        return fail(GCN10_ENODEV, "device %d out of range (%d visible)", device, n);
    CUDA_TRY(cudaSetDevice(device));
    gcn10_ctx *c = new (std::nothrow) gcn10_ctx();
    if (c) {
        // development aid: the default of option "streams" from the environment
        const char *e = getenv("GCN10_STREAMS");
        if (e && atoi(e) >= 1 && atoi(e) <= kMaxStreams)
            c->nstreams = atoi(e);
    }
    if (!c)
        return fail(GCN10_ENOMEM, "context allocation failed");
    c->device = device;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    if (prop.major < 10) {
        delete c;
        return fail(GCN10_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    }
    int prio_lo = 0, prio_hi = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    // priorities: the strips of the block in hand outrank the prefetched inflate of the NEXT block (pre_stream stays
    // at the lowest priority), so a block's first compressed tiles reach the copy engine as early as possible -- where
    // the device->host link is the bottleneck (eight GPUs on one host fabric) the inflate then fills the gaps instead of
    // delaying the stream of tiles; the ship kernels outrank both
    const int prio_strip = prio_hi < prio_lo ? std::min(prio_lo - 1, prio_hi + 1) : prio_lo;
    for (int i = 0; i < kMaxStreams; i++) {
        CUDA_TRY(cudaStreamCreateWithPriority(&c->streams[i], cudaStreamNonBlocking, prio_strip));
        CUDA_TRY(cudaStreamCreateWithPriority(&c->ship_streams[i], cudaStreamNonBlocking, prio_hi));
    }
    for (int i = 0; i < kMaxStreams; i++) {
        CUDA_TRY(cudaEventCreate(&c->slots[i].k0));
        CUDA_TRY(cudaEventCreate(&c->slots[i].k1));
        CUDA_TRY(cudaEventCreateWithFlags(&c->slots[i].k2, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->slots[i].done, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->slots[i].enc_done, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->slots[i].ov, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->slots[i].ag, cudaEventDisableTiming));
    }
    CUDA_TRY(cudaFuncSetAttribute((const void *)deflate_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kEncSmem));
    CUDA_TRY(cudaFuncSetAttribute((const void *)cn_deflate_fused_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  fused_smem_bytes<9>()));
    CUDA_TRY(cudaFuncSetAttribute((const void *)cn_deflate_fused_kernel<18>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  fused_smem_bytes<18>()));
    CUDA_TRY(cudaFuncSetAttribute((const void *)cn_deflate_fused_kernel<9>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    CUDA_TRY(cudaFuncSetAttribute((const void *)cn_deflate_fused_kernel<18>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    CUDA_TRY(cudaFuncSetAttribute((const void *)inflate_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kInflateSmem));
    CUDA_TRY(cudaFuncSetAttribute((const void *)lzw_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLzwSmem));
    CUDA_TRY(cudaFuncSetAttribute((const void *)lzw_tiles_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    CUDA_TRY(cudaFuncSetAttribute((const void *)inflate_tiles_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    CUDA_TRY(cudaStreamCreateWithPriority(&c->pre_stream, cudaStreamNonBlocking, prio_lo));
    CUDA_TRY(cudaEventCreateWithFlags(&c->frame_ready, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&c->agg_ready, cudaEventDisableTiming));
    for (int i = 0; i < kMaxStreams; i++)
        CUDA_TRY(cudaEventCreateWithFlags(&c->tail[i], cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
        CUDA_TRY(cudaEventCreate(&c->tslot[i].inf0));
        CUDA_TRY(cudaEventCreate(&c->tslot[i].inf1));
        CUDA_TRY(cudaEventCreateWithFlags(&c->tslot[i].done, cudaEventDisableTiming));
    }
    // cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
        c->encode_tiled = (EncodeTiledFn)fn;
    for (int np = 1; np <= 9; np++)
        for (int g = 1; g <= 2; g++)
            CUDA_TRY(cudaFuncSetAttribute((const void *)pick_kernel(np, g),
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes_for(np, g)));
    *out = c;
    return GCN10_OK;
}

void gcn10_cuda_destroy(gcn10_ctx *c)
{
    if (!c)
        return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    release(c->lut);
    release(c->col_idx);
    release(c->row_idx);
    release(c->hsg);
    release(c->fused_tab);
    release(c->ov_buf);
    release(c->stats_buf);
    release(c->agg_acc);
    release(c->agg_out);
    if (c->agg_ready) cudaEventDestroy(c->agg_ready);
    for (int i = 0; i < 2; i++) {
        release(c->tslot[i].in_blob);
        release(c->tslot[i].in_table);
        release(c->tslot[i].esa_full);
        release(c->tslot[i].scratch);
        release_host(c->tslot[i].h_status);
        if (c->tslot[i].inf0) cudaEventDestroy(c->tslot[i].inf0);
        if (c->tslot[i].inf1) cudaEventDestroy(c->tslot[i].inf1);
        if (c->tslot[i].done) cudaEventDestroy(c->tslot[i].done);
    }
    if (c->pre_stream) cudaStreamDestroy(c->pre_stream);
    if (c->frame_ready) cudaEventDestroy(c->frame_ready);
    for (int i = 0; i < kMaxStreams; i++)
        if (c->tail[i]) cudaEventDestroy(c->tail[i]);
    for (cudaEvent_t t : c->timer_pool)
        cudaEventDestroy(t);
    for (int i = 0; i < kMaxStreams; i++) {
        release(c->slots[i].esa);
        release(c->slots[i].out);
        release(c->slots[i].blob);
        release(c->slots[i].blob2);
        release(c->slots[i].order);
        release(c->slots[i].table);
        release_host(c->slots[i].h_blob);
        release_host(c->slots[i].h_table);
        if (c->slots[i].enc_done) cudaEventDestroy(c->slots[i].enc_done);
        if (c->slots[i].ov) cudaEventDestroy(c->slots[i].ov);
        if (c->slots[i].ag) cudaEventDestroy(c->slots[i].ag);
        if (c->slots[i].k0) cudaEventDestroy(c->slots[i].k0);
        if (c->slots[i].k1) cudaEventDestroy(c->slots[i].k1);
        if (c->slots[i].k2) cudaEventDestroy(c->slots[i].k2);
        if (c->slots[i].done) cudaEventDestroy(c->slots[i].done);
        if (c->streams[i]) cudaStreamDestroy(c->streams[i]);
        if (c->ship_streams[i]) cudaStreamDestroy(c->ship_streams[i]);
    }
    delete c;
}

int gcn10_cuda_set_luts(gcn10_ctx *c, const int tables[GCN10_NVARIANTS][256][5])
{
    if (!c || !tables)
        return fail(GCN10_EINVAL, "NULL argument");
    if (c->pending_events)
        return fail(GCN10_EINVAL, "asynchronous blocks are pending on this context: gcn10_cuda_wait() for them first");
    CUDA_TRY(cudaSetDevice(c->device));
    memcpy(c->host_tables, tables, sizeof(c->host_tables));
    c->swz_shift = choose_swizzle(c->host_tables);
    c->lut_mask[0] = c->lut_mask[1] = 0xFFFFFFFFu;
    c->fused_mask = 0;
    c->have_lut = true;
    return GCN10_OK;
}

int gcn10_cuda_set_option(gcn10_ctx *c, const char *key, long value)
{
    if (!c || !key)
        return fail(GCN10_EINVAL, "NULL argument");
    if (!strcmp(key, "strip_rows") && value >= 1) c->strip_rows = (int)value;
    else if (!strcmp(key, "streams") && value >= 1 && value <= kMaxStreams) c->nstreams = (int)value;
    else if (!strcmp(key, "defer_inflate") && (value == 0 || value == 1)) c->defer_inflate = (int)value;
    else if (!strcmp(key, "rows_per_cta") && value >= 0) c->rows_per_cta = (int)value;
    else if (!strcmp(key, "tma") && (value == 0 || value == 1)) c->use_tma = (int)value;
    else if (!strcmp(key, "fused") && (value == 0 || value == 1)) c->fused = (int)value;
    else if (!strcmp(key, "ship") && (value == 0 || value == 1)) c->ship = (int)value;
    else if (!strcmp(key, "ordered") && (value == 0 || value == 1)) c->ordered = (int)value;
    else if (!strcmp(key, "cog") && (value == 0 || value == 1)) c->cog = (int)value;
    else if (!strcmp(key, "overviews") && value >= 0 && value <= GCN10_MAX_OVERVIEWS) {
        c->overviews = (int)value;
        c->blk_next = -1;
    }
    else if (!strcmp(key, "stats") && (value == 0 || value == 1)) {
        c->stats = (int)value;
        c->blk_next = -1;
        c->stats_ready = false;
    }
    else if (!strcmp(key, "aggregate") && (value == 0 || (value >= 2 && value <= GCN10_MAX_AGGREGATE))) {
        c->aggregate = (int)value;
        c->blk_next = -1;
    }
    else if (!strcmp(key, "inflate_probe") && value >= 0 && value <= 2) c->inflate_probe = (int)value;
    else if (!strcmp(key, "tuned_code") && (value == 0 || value == 1)) {
        c->tuned_code = (int)value;
        c->fused_mask = 0;
    }
    else return fail(GCN10_EINVAL, "unknown option or bad value: %s=%ld", key, value);
    return GCN10_OK;
}

int gcn10_cuda_synchronize(gcn10_ctx *c)
{
    if (!c)
        return fail(GCN10_EINVAL, "NULL context");
    CUDA_TRY(cudaSetDevice(c->device));
    for (int i = 0; i < kMaxStreams; i++) {
        CUDA_TRY(cudaStreamSynchronize(c->streams[i]));
        CUDA_TRY(cudaStreamSynchronize(c->ship_streams[i]));
    }
    return GCN10_OK;
}

int gcn10_cuda_last_kernel_ms(gcn10_ctx *c, float *ms)
{
    if (!c || !ms)
        return fail(GCN10_EINVAL, "NULL argument");
    *ms = c->last_kernel_ms;
    return GCN10_OK;
}

int gcn10_cuda_launch_count(gcn10_ctx *c, uint64_t *launches)
{
    if (!c || !launches)
        return fail(GCN10_EINVAL, "NULL argument");
    *launches = c->launches;
    return GCN10_OK;
}

int gcn10_cuda_last_histograms(gcn10_ctx *c, uint64_t hist[GCN10_NPLANES][256])
{
    if (!c || !hist)
        return fail(GCN10_EINVAL, "NULL argument");
    if (!c->stats_ready)
        return fail(GCN10_EINVAL, "no block has completed with option \"stats\" on since it was set");
    memcpy(hist, c->stats_hist, sizeof(c->stats_hist));
    return GCN10_OK;
}

int gcn10_cuda_index_maps(gcn10_ctx *c, int w, int h, const double gt[6], int hsx, int hsy,
                          const double soil_gt[6], int32_t *col_index, int32_t *row_index)
{
    if (!c || !gt || !soil_gt || !col_index || !row_index)
        return fail(GCN10_EINVAL, "NULL argument");
    if (w <= 0 || h <= 0 || hsx <= 0 || hsy <= 0)
        return fail(GCN10_EINVAL, "non-positive size");
    if (c->pending_events)
        return fail(GCN10_EINVAL, "asynchronous blocks are pending on this context: gcn10_cuda_wait() for them first");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->streams[0];
    int rc = launch_index_maps(c, w, h, gt, hsx, hsy, soil_gt, st);
    if (rc)
        return rc;
    CUDA_TRY(cudaMemcpyAsync(col_index, c->col_idx.p, sizeof(int32_t) * (size_t)w, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(row_index, c->row_idx.p, sizeof(int32_t) * (size_t)h, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return GCN10_OK;
}

int gcn10_cuda_block_device(gcn10_ctx *c,
                            const uint8_t *d_esa, int w, int h, size_t esa_pitch, const double gt[6],
                            const uint8_t *d_hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                            unsigned plane_mask, uint8_t *const d_out[GCN10_NPLANES], size_t out_pitch,
                            void *stream)
{
    if (!c)
        return fail(GCN10_EINVAL, "NULL context");
    int rc = check_geometry(d_esa, w, h, esa_pitch, gt, d_hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask, d_out,
                            out_pitch);
    if (rc)
        return rc;
    if (!c->have_lut)
        return fail(GCN10_ENOLUT, "gcn10_cuda_set_luts() has not been called");
    if (c->pending_events)
        return fail(GCN10_EINVAL, "asynchronous blocks are pending on this context: gcn10_cuda_wait() for them first");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->streams[0];

    LaunchPlan plans[2];
    int nplans = plan_launches(plane_mask, plans);
    for (int i = 0; i < nplans; i++)
        if ((rc = upload_lut(c, plans[i].variant_mask, i, st)))
            return rc;
    if ((rc = launch_index_maps(c, w, h, gt, hsx, hsy, soil_gt, st)))
        return rc;
    CUtensorMap map;
    int tma_ok = 0;
    make_hsg_map(c, d_hsg, hsx, hsy, hsg_pitch, &map, &tma_ok);
    for (int i = 0; i < nplans; i++)
        if ((rc = launch_rows(c, plans[i], i, d_esa, esa_pitch, w, h, 0, d_hsg, hsg_pitch, hsx, hsy, map, tma_ok,
                              d_out, out_pitch, st)))
            return rc;
    return GCN10_OK;
}

// ---- raw planes back: enqueue / wait ----------------------------------------------------------------------------
//
// Everything a block needs is queued on the context's streams without the host waiting for any of it: the frame
// (HSG window + fp64 index maps) on stream 0, guarded by an event the strip streams wait for; then the row strips
// round-robin over the streams, each stream owning one staging slot (slot reuse is ordered by the stream itself).
// A following block's frame waits, on the device, for the previous block's strips (they read the shared frame
// buffers).  gcn10_cuda_wait() blocks for the block's last copies and adds up the kernel times.

static int block_rows_enqueue(gcn10_ctx *c,
                              const uint8_t *esa, int w, int h, int row0, int nrows, size_t esa_pitch,
                              const double gt[6],
                              const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                              unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch,
                              gcn10_event **done)
{
    if (!c || !done)
        return fail(GCN10_EINVAL, "NULL context");
    *done = nullptr;
    int rc = check_geometry(esa, w, h, esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask, out, out_pitch);
    if (rc)
        return rc;
    if (row0 < 0 || nrows <= 0 || row0 > h - nrows)
        return fail(GCN10_EINVAL, "row range [%d, %d+%d) outside the block's %d rows", row0, row0, nrows, h);
    if (!c->have_lut)
        return fail(GCN10_ENOLUT, "gcn10_cuda_set_luts() has not been called");
    for (int k = 0; k < GCN10_NPLANES; k++)
        if ((plane_mask & (1u << k)) && !out[k])
            return fail(GCN10_EINVAL, "output plane %d selected by the mask but its pointer is NULL", k);
    CUDA_TRY(cudaSetDevice(c->device));

    LaunchPlan plans[2];
    const int nplans = plan_launches(plane_mask, plans);
    int nplanes = 0;
    for (int i = 0; i < nplans; i++)
        nplanes += plans[i].np * plans[i].groups;

    const size_t hsg_dpitch = round_up((size_t)hsx, 256);
    const size_t dpitch = round_up((size_t)w, 256);
    const int ns = c->nstreams;
    const int strip = std::max(1, std::min(c->strip_rows, nrows));
    const int nstrips = (nrows + strip - 1) / strip;
    // (re)allocation frees device memory, which waits for the device by itself; sizes only ever grow
    bool grow = c->hsg.cap < hsg_dpitch * (size_t)hsy;
    for (int i = 0; i < ns; i++)
        grow = grow || c->slots[i].esa.cap < dpitch * (size_t)strip ||
               c->slots[i].out.cap < dpitch * (size_t)strip * (size_t)nplanes;
    if (grow && (rc = gcn10_cuda_synchronize(c)))
        return rc;

    cudaStream_t s0 = c->streams[0];
    // the previous block's strips read the frame buffers this block is about to overwrite
    for (int i = 1; i < kMaxStreams; i++)
        if (c->tail_valid[i])
            CUDA_TRY(cudaStreamWaitEvent(s0, c->tail[i], 0));
    for (int i = 0; i < nplans; i++)
        if ((rc = upload_lut(c, plans[i].variant_mask, i, s0)))
            return rc;
    if ((rc = ensure(c->hsg, hsg_dpitch * (size_t)hsy)))
        return rc;
    CUDA_TRY(cudaMemcpy2DAsync(c->hsg.p, hsg_dpitch, hsg, hsg_pitch, (size_t)hsx, (size_t)hsy,
                               cudaMemcpyHostToDevice, s0));
    if ((rc = launch_index_maps(c, w, h, gt, hsx, hsy, soil_gt, s0)))
        return rc;
    CUtensorMap map;
    int tma_ok = 0;
    make_hsg_map(c, (const uint8_t *)c->hsg.p, hsx, hsy, hsg_dpitch, &map, &tma_ok);
    CUDA_TRY(cudaEventRecord(c->frame_ready, s0));
    for (int i = 0; i < ns; i++) {
        if ((rc = ensure(c->slots[i].esa, dpitch * (size_t)strip)) ||
            (rc = ensure(c->slots[i].out, dpitch * (size_t)strip * (size_t)nplanes)))
            return rc;
        if (i)
            CUDA_TRY(cudaStreamWaitEvent(c->streams[i], c->frame_ready, 0));
    }

    gcn10_event *ev = new (std::nothrow) gcn10_event();
    if (!ev)
        return fail(GCN10_ENOMEM, "event allocation failed");
    ev->ctx = c;
    ev->timers.resize(2 * (size_t)nstrips);
    ev->ends.resize((size_t)ns);
    auto take = [&](cudaEvent_t &t) {
        if (!c->timer_pool.empty()) {
            t = c->timer_pool.back();
            c->timer_pool.pop_back();
        }
        else if (cudaEventCreate(&t) != cudaSuccess) {
            t = nullptr;
        }
    };
    for (auto &t : ev->timers)
        take(t);
    for (auto &t : ev->ends)
        take(t);

    int si = 0, sidx = 0;
    // y0 counts rows of the caller's band: esa / out row 0 is block row `row0`
    for (int y0 = 0; y0 < nrows && !rc; y0 += strip, si = (si + 1) % ns, sidx++) {
        const int rows = std::min(strip, nrows - y0);
        StripSlot &sl = c->slots[si];
        cudaStream_t st = c->streams[si];
        cudaEvent_t k0 = ev->timers[2 * sidx], k1 = ev->timers[2 * sidx + 1];
        cudaMemcpy2DAsync(sl.esa.p, dpitch, esa + (size_t)y0 * esa_pitch, esa_pitch, (size_t)w, (size_t)rows,
                          cudaMemcpyHostToDevice, st);
        uint8_t *d_out[GCN10_NPLANES] = { nullptr };
        int k = 0;
        for (int i = 0; i < nplans; i++)
            for (int j = 0; j < plans[i].np * plans[i].groups; j++, k++)
                d_out[plans[i].plane_ids[j]] = (uint8_t *)sl.out.p + (size_t)k * dpitch * (size_t)strip;
        if (k0)
            cudaEventRecord(k0, st);
        for (int i = 0; i < nplans && !rc; i++)
            rc = launch_rows(c, plans[i], i, (const uint8_t *)sl.esa.p, dpitch, w, rows, row0 + y0,
                             (const uint8_t *)c->hsg.p, hsg_dpitch, hsx, hsy, map, tma_ok, d_out, dpitch, st);
        if (k1)
            cudaEventRecord(k1, st);
        for (int p = 0; p < GCN10_NPLANES && !rc; p++)
            if (d_out[p])
                cudaMemcpy2DAsync(out[p] + (size_t)y0 * out_pitch, out_pitch, d_out[p], dpitch, (size_t)w,
                                  (size_t)rows, cudaMemcpyDeviceToHost, st);
    }
    // the block is complete when every stream has passed this point
    for (int i = 0; i < ns; i++) {
        cudaEventRecord(c->tail[i], c->streams[i]);
        c->tail_valid[i] = true;
        if (ev->ends[i])
            cudaEventRecord(ev->ends[i], c->streams[i]);
    }
    ev->nstreams = ns;
    c->pending_events++;
    const cudaError_t ce = cudaGetLastError();
    if (!rc && ce != cudaSuccess)
        rc = fail(GCN10_ECUDA, "queueing the block failed: %s", cudaGetErrorString(ce));
    ev->status = rc;
    *done = ev;
    return GCN10_OK;            // a queueing error is reported by gcn10_cuda_wait, after the streams have drained
}

int gcn10_cuda_block_async(gcn10_ctx *c,
                           const uint8_t *esa, int w, int h, size_t esa_pitch, const double gt[6],
                           const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                           unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch,
                           gcn10_event **done)
{
    return block_rows_enqueue(c, esa, w, h, 0, h, esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask, out,
                              out_pitch, done);
}

int gcn10_cuda_event_query(gcn10_event *ev)
{
    if (!ev || !ev->ctx)
        return fail(GCN10_EINVAL, "NULL event");
    gcn10_ctx *c = ev->ctx;
    if (cudaSetDevice(c->device) != cudaSuccess)
        return fail(GCN10_ECUDA, "cudaSetDevice failed");
    for (int i = 0; i < ev->nstreams; i++) {
        const cudaError_t e = ev->ends[i] ? cudaEventQuery(ev->ends[i]) : cudaStreamQuery(c->streams[i]);
        if (e == cudaErrorNotReady)
            return 0;
        if (e != cudaSuccess)
            return fail(GCN10_ECUDA, "cudaEventQuery: %s", cudaGetErrorString(e));
    }
    return 1;
}

int gcn10_cuda_wait(gcn10_event *ev)
{
    if (!ev || !ev->ctx)
        return fail(GCN10_EINVAL, "NULL event");
    gcn10_ctx *c = ev->ctx;
    int rc = ev->status;
    cudaSetDevice(c->device);
    for (int i = 0; i < ev->nstreams; i++) {
        const cudaError_t e = ev->ends[i] ? cudaEventSynchronize(ev->ends[i]) : cudaStreamSynchronize(c->streams[i]);
        if (e != cudaSuccess && !rc)
            rc = fail(GCN10_ECUDA, "block failed on the device: %s", cudaGetErrorString(e));
    }
    float kernel_ms = 0.f;
    for (size_t i = 0; i + 1 < ev->timers.size(); i += 2) {
        float ms = 0.f;
        if (!rc && ev->timers[i] && ev->timers[i + 1] &&
            cudaEventElapsedTime(&ms, ev->timers[i], ev->timers[i + 1]) == cudaSuccess)
            kernel_ms += ms;
    }
    cudaGetLastError();
    for (cudaEvent_t t : ev->timers)
        if (t)
            c->timer_pool.push_back(t);
    for (cudaEvent_t t : ev->ends)
        if (t)
            c->timer_pool.push_back(t);
    if (!rc)
        c->last_kernel_ms = kernel_ms;
    if (--c->pending_events <= 0) {
        c->pending_events = 0;
        for (int i = 0; i < kMaxStreams; i++)
            c->tail_valid[i] = false;       // (the newest block was waited for: every stream has drained)
    }
    delete ev;
    return rc;
}

int gcn10_cuda_block(gcn10_ctx *c,
                     const uint8_t *esa, int w, int h, size_t esa_pitch, const double gt[6],
                     const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                     unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch)
{
    return gcn10_cuda_block_rows(c, esa, w, h, 0, h, esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask,
                                 out, out_pitch);
}

int gcn10_cuda_block_rows(gcn10_ctx *c,
                          const uint8_t *esa, int w, int h, int row0, int nrows, size_t esa_pitch,
                          const double gt[6],
                          const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                          unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch)
{
    gcn10_event *ev = nullptr;
    const int rc = block_rows_enqueue(c, esa, w, h, row0, nrows, esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt,
                                      plane_mask, out, out_pitch, &ev);
    if (rc)
        return rc;
    return gcn10_cuda_wait(ev);
}

static int deflate_rows_impl(gcn10_ctx *c,
                             const uint8_t *esa, size_t esa_pitch, const uint8_t *d_esa, size_t d_esa_pitch,
                             cudaEvent_t esa_ready, int w, int h, int row0, int nrows,
                             const double gt[6],
                             const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                             unsigned plane_mask, gcn10_tile_sink sink, void *user,
                             const std::function<int()> &before_first_sink = nullptr);
static int free_slot(gcn10_ctx *c, TileSlot **out);

int gcn10_cuda_block_deflate(gcn10_ctx *c,
                             const uint8_t *esa, int w, int h, size_t esa_pitch, const double gt[6],
                             const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                             unsigned plane_mask, gcn10_tile_sink sink, void *user)
{
    if (!c || !c->cog)
        return gcn10_cuda_block_deflate_rows(c, esa, w, h, 0, h, esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt,
                                             plane_mask, sink, user);
    // option "cog": the levels are made before the first strip, so the whole raster goes to the device first, into the
    // land-cover plane of a tile slot that holds no prefetched block; from there the block runs as the tiles path does
    int rc = check_geometry(esa, w, h, esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask, (const void *)sink,
                            (size_t)w);
    if (rc)
        return rc;
    if (!c->have_lut)
        return fail(GCN10_ENOLUT, "gcn10_cuda_set_luts() has not been called");
    if (c->pending_events)
        return fail(GCN10_EINVAL, "asynchronous blocks are pending on this context: gcn10_cuda_wait() for them first");
    CUDA_TRY(cudaSetDevice(c->device));
    TileSlot *sl = nullptr;
    if ((rc = free_slot(c, &sl)))
        return rc;
    const size_t dpitch = round_up((size_t)w, 256);
    if ((rc = ensure(sl->esa_full, dpitch * (size_t)h)))
        return rc;
    // (on the upload stream: a dropped prefetch of this slot may still have work on the plane queued there)
    CUDA_TRY(cudaMemcpy2DAsync(sl->esa_full.p, dpitch, esa, esa_pitch, (size_t)w, (size_t)h, cudaMemcpyHostToDevice,
                               c->pre_stream));
    CUDA_TRY(cudaEventRecord(sl->done, c->pre_stream));
    return deflate_rows_impl(c, nullptr, 0, (const uint8_t *)sl->esa_full.p, dpitch, sl->done, w, h, 0, h, gt, hsg, hsx,
                             hsy, hsg_pitch, soil_gt, plane_mask, sink, user);
}

// Strips of whole tile rows: [H2D of the land-cover rows ->] Curve Number kernel -> tile DEFLATE -> D2H of
// the compressed tiles -> sink.  The land cover comes either from the caller's host raster (esa) or from a
// device-resident plane (d_esa, valid once `esa_ready` has fired: the compressed-input path).
static int launch_inflate(gcn10_ctx *c, TileSlot &sl, cudaEvent_t after);

// Option "stats", after the block's last strip has been handed over (so every kernel that counted has finished): the
// device counts come back once, and the per-id counts of the fused path become plane histograms through the value
// records of the block's plane mask -- a pixel's value in every plane is a function of its record id.
static int finish_histograms(gcn10_ctx *c, cudaStream_t st)
{
    std::vector<unsigned long long> h((size_t)kFusedIds + (size_t)GCN10_NPLANES * 256);
    CUDA_TRY(cudaMemcpyAsync(h.data(), c->stats_buf.p, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int p = 0; p < GCN10_NPLANES; p++)
        for (int v = 0; v < 256; v++)
            c->stats_hist[p][v] = h[(size_t)kFusedIds + (size_t)p * 256 + v];
    if (c->blk_fused) {
        int rc = build_fused_tables(c, c->blk_mask, st);        // (the tables of the block's mask: cached, no work)
        if (rc)
            return rc;
        int plane_ids[GCN10_NPLANES], nsel = 0;
        for (int p = 0; p < GCN10_NPLANES; p++)
            if (c->blk_mask & (1u << p))
                plane_ids[nsel++] = p;
        for (int id = 0; id < kFusedPad; id++)
            for (int j = 0; j < nsel && h[id]; j++)
                c->stats_hist[plane_ids[j]][c->fused_rec[id][j]] += h[id];
    }
    c->stats_ready = true;
    return GCN10_OK;
}

static int deflate_rows_impl(gcn10_ctx *c,
                             const uint8_t *esa, size_t esa_pitch, const uint8_t *d_esa, size_t d_esa_pitch,
                             cudaEvent_t esa_ready, int w, int h, int row0, int nrows,
                             const double gt[6],
                             const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                             unsigned plane_mask, gcn10_tile_sink sink, void *user,
                             const std::function<int()> &before_first_sink)
{
    if (!c)
        return fail(GCN10_EINVAL, "NULL context");
    if (!sink)
        return fail(GCN10_EINVAL, "NULL sink");
    if (row0 < 0 || nrows <= 0 || row0 > h - nrows || row0 % kTile != 0 || (nrows % kTile != 0 && row0 + nrows != h))
        return fail(GCN10_EINVAL, "row band [%d, +%d) must start on a 256-row tile boundary and end on one or at "
                                  "the block's last row (%d)", row0, nrows, h);
    int rc = check_geometry(esa ? esa : d_esa, w, h, esa ? esa_pitch : d_esa_pitch, gt, hsg, hsx, hsy, hsg_pitch, soil_gt,
                            plane_mask, (const void *)sink, (size_t)w);
    if (rc)
        return rc;
    if (!c->have_lut)
        return fail(GCN10_ENOLUT, "gcn10_cuda_set_luts() has not been called");
    if (c->pending_events)
        return fail(GCN10_EINVAL, "asynchronous blocks are pending on this context: gcn10_cuda_wait() for them first");
    // option "cog": the levels come first, so the whole block's land cover must be on the device before the first strip
    // (the callers upload or inflate it there)
    const bool cog = c->cog;
    if (cog && (!d_esa || row0 != 0 || nrows != h))
        return fail(GCN10_EINVAL, "option cog: the block must be resident on the device and handed over in one call");
    // options "overviews", "stats" and "aggregate": every band feeds the block's levels, histograms and mean rasters, so
    // the bands of a block must come in order and without gaps (with "stats" or "aggregate" also with the same planes);
    // the band that ends the block emits the levels and the mean rasters and completes the histograms
    const int nlev = c->overviews ? gcn10_overview_levels(w, h, c->overviews) : 0;
    const int agg = c->aggregate;
    const bool gather = nlev || c->stats || agg;
    if (gather && row0 != 0 &&
        (row0 != c->blk_next || w != c->blk_w || h != c->blk_h || ((c->stats || agg) && plane_mask != c->blk_mask))) {
        rc = fail(GCN10_EINVAL, "%s: band [%d, +%d) of a %d x %d block does not continue the block's previous band "
                                "(next row %d); a block starts with row 0",
                  nlev ? "overviews" : c->stats ? "stats" : "aggregate", row0, nrows, w, h, c->blk_next);
        c->blk_next = -1;
        return rc;
    }
    c->blk_next = -1;           // (until this call has succeeded)
    const bool ends_block = row0 + nrows == h;
    const bool emit_levels = nlev && ends_block;
    const bool emit_agg = agg && ends_block;
    CUDA_TRY(cudaSetDevice(c->device));
    if (gather && row0 == 0) {
        c->blk_w = w;
        c->blk_h = h;
        c->blk_mask = plane_mask;
    }
    if (nlev && row0 == 0) {
        size_t off[GCN10_MAX_OVERVIEWS][3], total = 0;
        for (int k = 1; k <= nlev; k++) {
            OverviewLevel &L = c->ov_lv[k - 1];
            L.k = k;
            L.w = gcn10_overview_dim(w, k);
            c->ov_h[k - 1] = gcn10_overview_dim(h, k);
            L.pitch = round_up((size_t)L.w, 256);
            off[k - 1][0] = total;
            total += L.pitch * (size_t)c->ov_h[k - 1];
            off[k - 1][1] = total;
            total += round_up(sizeof(int32_t) * round_up((size_t)L.w, kVecPx), 256);
            off[k - 1][2] = total;
            total += round_up(sizeof(int32_t) * (size_t)c->ov_h[k - 1], 256);
        }
        if ((rc = ensure(c->ov_buf, total)))
            return rc;
        for (int k = 0; k < nlev; k++) {
            c->ov_lv[k].esa = (uint8_t *)c->ov_buf.p + off[k][0];
            c->ov_lv[k].col_idx = (int32_t *)((uint8_t *)c->ov_buf.p + off[k][1]);
            c->ov_lv[k].row_idx = (int32_t *)((uint8_t *)c->ov_buf.p + off[k][2]);
        }
    }

    LaunchPlan plans[2];
    const int nplans = plan_launches(plane_mask, plans);
    int nplanes = 0, plane_ids[GCN10_NPLANES];
    for (int k = 0; k < GCN10_NPLANES; k++)
        if (plane_mask & (1u << k))
            plane_ids[nplanes++] = k;

    cudaStream_t s0 = c->streams[0];
    constexpr size_t kStatsWords = (size_t)kFusedIds + (size_t)GCN10_NPLANES * 256;
    if (c->stats && row0 == 0) {
        // (done before the strips start: s0 is synchronised below)
        if ((rc = ensure(c->stats_buf, kStatsWords * sizeof(unsigned long long))))
            return rc;
        CUDA_TRY(cudaMemsetAsync(c->stats_buf.p, 0, kStatsWords * sizeof(unsigned long long), s0));
        c->blk_fused = false;
        c->stats_ready = false;
    }
    // option "aggregate": a block starts with zero accumulators (the finish kernel leaves them so; a new buffer or an
    // abandoned block is cleared here)
    const int acw = agg ? gcn10_aggregate_dim(w, agg) : 0, ach = agg ? gcn10_aggregate_dim(h, agg) : 0;
    const size_t apitch = round_up((size_t)acw, 256);
    if (agg && row0 == 0) {
        const size_t cap_was = c->agg_acc.cap;
        if ((rc = ensure(c->agg_acc, sizeof(uint2) * (size_t)nplanes * ach * acw)) ||
            (rc = ensure(c->agg_out, apitch * (size_t)ach * nplanes)))
            return rc;
        if (c->agg_acc.cap != cap_was || !c->agg_clean)
            CUDA_TRY(cudaMemsetAsync(c->agg_acc.p, 0, c->agg_acc.cap, s0));
        c->agg_clean = false;
    }
    unsigned long long *id_hist = c->stats ? (unsigned long long *)c->stats_buf.p : nullptr;
    unsigned long long *plane_hist = c->stats ? id_hist + kFusedIds : nullptr;
    for (int i = 0; i < nplans; i++)
        if ((rc = upload_lut(c, plans[i].variant_mask, i, s0)))
            return rc;
    const size_t hsg_dpitch = round_up((size_t)hsx, 256);
    if ((rc = ensure(c->hsg, hsg_dpitch * (size_t)hsy)))
        return rc;
    CUDA_TRY(cudaMemcpy2DAsync(c->hsg.p, hsg_dpitch, hsg, hsg_pitch, (size_t)hsx, (size_t)hsy,
                               cudaMemcpyHostToDevice, s0));
    if ((rc = launch_index_maps(c, w, h, gt, hsx, hsy, soil_gt, s0)))
        return rc;
    CUtensorMap map;
    int tma_ok = 0;
    make_hsg_map(c, (const uint8_t *)c->hsg.p, hsx, hsy, hsg_dpitch, &map, &tma_ok);
    CUDA_TRY(cudaStreamSynchronize(s0));

    const bool fused = c->fused && !build_fused_tables(c, plane_mask & GCN10_MASK_ALL, s0) && c->fused_ok;
    if (c->stats && fused)
        c->blk_fused = true;

    // strips of whole tile rows
    const size_t dpitch = round_up((size_t)w, 256);
    const int ns = c->nstreams;
    const int strip = std::max(kTile, std::min(c->strip_rows, (int)round_up((size_t)nrows, kTile)) / kTile * kTile);
    const int tiles_x = (w + kTile - 1) / kTile;
    // the strips of this call: the band's full-resolution rows; then, when the band ends the block, every overview
    // level, level 1 first, in strips of at most `lstrip` level rows (they use the same slots, at most tiles_x wide).
    // With option "cog" the levels come first instead, the smallest first (nlev .. 1), then the full resolution.
    struct StripJob {
        int level, y0, rows, w, h, y_base;      // y0: row in the caller's band (level 0) or in the level
        const uint8_t *d_esa;                   // nullptr: staged from the caller's host raster
        size_t pitch;
        const int32_t *col_idx, *row_idx;       // nullptr: the block's
        int agg;                                // a strip of the mean rasters (d_esa: their first row)
    };
    std::vector<StripJob> jobs;
    const int lstrip = emit_levels ? std::max(kTile, std::min(c->strip_rows, (int)round_up((size_t)c->ov_h[0], kTile)) / kTile * kTile)
                                   : 0;
    auto push_level = [&](int k) {
        const OverviewLevel &L = c->ov_lv[k];
        for (int y0 = 0; y0 < c->ov_h[k]; y0 += lstrip)
            jobs.push_back({ k + 1, y0, std::min(lstrip, c->ov_h[k] - y0), L.w, c->ov_h[k], y0,
                             L.esa + (size_t)y0 * L.pitch, L.pitch, L.col_idx, L.row_idx });
    };
    for (int k = (cog && emit_levels ? nlev : 0) - 1; k >= 0; k--)
        push_level(k);
    const int first_full = (int)jobs.size();
    for (int y0 = 0; y0 < nrows; y0 += strip)
        jobs.push_back({ 0, y0, std::min(strip, nrows - y0), w, h, row0 + y0,
                         d_esa ? d_esa + (size_t)y0 * d_esa_pitch : nullptr, d_esa_pitch, nullptr, nullptr });
    for (int k = 0; k < (!cog && emit_levels ? nlev : 0); k++)
        push_level(k);
    // then, when the band ends the block, the mean rasters in strips of at most `astrip` cell rows
    const int astrip = emit_agg ? std::max(kTile, std::min(c->strip_rows, (int)round_up((size_t)ach, kTile)) / kTile * kTile) : 0;
    const int first_agg = (int)jobs.size();
    for (int y0 = 0; emit_agg && y0 < ach; y0 += astrip)
        jobs.push_back({ 0, y0, std::min(astrip, ach - y0), acw, ach, y0, (const uint8_t *)c->agg_out.p + (size_t)y0 * apitch,
                         apitch, nullptr, nullptr, agg });
    const int strip_cap = std::max(std::max(strip, lstrip), astrip);
    const int strip_tile_rows = strip_cap / kTile;
    const size_t ntile_slot = (size_t)nplanes * strip_tile_rows * tiles_x;
    const size_t blob_cap = ntile_slot * (size_t)round_up(kStoredBytes, 16);
    const size_t table_bytes = 16 + ntile_slot * (sizeof(unsigned long long) + sizeof(uint32_t));
    // ordered strips: the second arena holds what a strip really compresses to (a quarter of the worst case, at least
    // 16 MB); a strip that does not fit leaves unordered -- still a valid strip, the consumer only loses the single write
    const size_t blob2_cap = std::min(blob_cap, std::max<size_t>(blob_cap / 4, (size_t)16 << 20));
    for (int i = 0; i < ns; i++) {
        StripSlot &sl = c->slots[i];
        if ((esa && (rc = ensure(sl.esa, dpitch * (size_t)strip))) ||
            (!fused && (rc = ensure(sl.out, dpitch * (size_t)strip_cap * nplanes))) ||
            (rc = ensure(sl.blob, blob_cap)) || (rc = ensure(sl.table, table_bytes)) ||
            (c->ordered && ((rc = ensure(sl.blob2, blob2_cap)) || (rc = ensure(sl.order, ntile_slot * sizeof(unsigned long long))))) ||
            (rc = ensure_host(sl.h_table, table_bytes)))
            return rc;
        // the host mirror of the blob only has to hold what a strip really compresses to; start at 1/16 of
        // the worst case and grow on demand
        if ((rc = ensure_host(sl.h_blob, std::max<size_t>(blob_cap / 16, 1 << 20))))
            return rc;
        sl.busy = false;
        sl.timed = false;
        if (esa_ready)
            CUDA_TRY(cudaStreamWaitEvent(c->streams[i], esa_ready, 0));
    }

    const int nstrips = (int)jobs.size();
    float kernel_ms = 0.f;

    // option "aggregate": what every accumulate launch shares -- a thread's segment of at most 32 pixel columns, a cell
    // row's rows walked in equal chunks of at most 32 per CTA, and each launch plan's records and outputs
    AggParams ap;
    memset(&ap, 0, sizeof(ap));
    if (agg) {
        ap.w = w;
        ap.f = agg;
        ap.cw = acw;
        ap.ch = ach;
        ap.spc = (agg + 31) / 32;
        ap.seg = (agg + ap.spc - 1) / ap.spc;
        ap.nchunk = (agg + 31) / 32;
        ap.chunk_rows = (agg + ap.nchunk - 1) / ap.nchunk;
        ap.col_idx = (const int32_t *)c->col_idx.p;
        ap.row_idx = (const int32_t *)c->row_idx.p;
        ap.hsg = (const uint8_t *)c->hsg.p;
        ap.hsg_pitch = hsg_dpitch;
        ap.swz_shift = c->swz_shift;
        ap.nplans = nplans;
        for (int i = 0; i < nplans; i++) {
            AggPlan &P = ap.plan[i];
            P.lut = (const uint8_t *)c->lut.p + (size_t)i * kLutBytes;
            P.rec_bytes = plans[i].np <= kNarrowPlanes ? 4 : 16;
            P.np = plans[i].np;
            P.groups = plans[i].groups;
            P.drained[0] = plans[i].drained[0];
            P.drained[1] = plans[i].drained[1];
            for (int k = 0; k < plans[i].np * plans[i].groups; k++)
                P.acc[k] = (int)(std::find(plane_ids, plane_ids + nplanes, plans[i].plane_ids[k]) - plane_ids);
        }
        ap.nsel = nplanes;
        ap.acc = (uint2 *)c->agg_acc.p;
    }

    // behind the encoder on the strip's stream: either the ship kernel (exact bytes + tables straight into the
    // page-locked arena, nothing for the host to do but wait), or the table read-back of the two-phase path
    // option "cog" with "ordered": the re-laid strip carries every tile's leader and trailer, and its size is the table's
    // second word (framed_bytes; 0 = it did not fit the second arena and leaves unordered and unframed)
    const bool framed = cog && c->ordered;
    auto hand_over = [&](StripSlot &sl, cudaStream_t st) -> int {
        CUDA_TRY(cudaEventRecord(sl.k1, st));
        unsigned long long *framed_bytes = (unsigned long long *)sl.table.p + 1;
        if (c->ordered) {
            const int n = nplanes * ((sl.rows + kTile - 1) / kTile) * sl.tiles_x;
            unsigned long long *d_offsets = (unsigned long long *)((uint8_t *)sl.table.p + 16);
            const uint32_t *d_sizes = (const uint32_t *)((uint8_t *)sl.table.p + 16 + ntile_slot * sizeof(unsigned long long));
            if (framed) {
                order_scan_kernel<true><<<1, 1024, 0, st>>>(d_sizes, n, (unsigned long long *)sl.order.p, framed_bytes,
                                                            (unsigned long long)blob2_cap);
                order_copy_kernel<true><<<2 * c->sm_count, 256, 0, st>>>((const uint8_t *)sl.blob.p, d_offsets, d_sizes,
                                                                         (const unsigned long long *)sl.order.p,
                                                                         (uint8_t *)sl.blob2.p, n, framed_bytes,
                                                                         (unsigned long long)blob2_cap);
            }
            else {
                order_scan_kernel<false><<<1, 1024, 0, st>>>(d_sizes, n, (unsigned long long *)sl.order.p,
                                                             (unsigned long long *)sl.table.p, (unsigned long long)blob2_cap);
                order_copy_kernel<false><<<2 * c->sm_count, 256, 0, st>>>((const uint8_t *)sl.blob.p, d_offsets, d_sizes,
                                                                          (const unsigned long long *)sl.order.p,
                                                                          (uint8_t *)sl.blob2.p, n,
                                                                          (const unsigned long long *)sl.table.p,
                                                                          (unsigned long long)blob2_cap);
            }
            c->launches += 2;
            CUDA_TRY(cudaGetLastError());
        }
        CUDA_TRY(cudaEventRecord(sl.k2, st));
        const void *out_blob = c->ordered ? sl.blob2.p : sl.blob.p;      // (ship: ordered strips always fit, see below)
        if (c->ship) {
            cudaStream_t ss = c->ship_streams[&sl - c->slots];
            CUDA_TRY(cudaStreamWaitEvent(ss, sl.k2, 0));
            ship_strip_kernel<<<kShipCtas, kShipThreads, 0, ss>>>((const uint4 *)out_blob,
                                                                  framed ? framed_bytes : (const unsigned long long *)sl.table.p,
                                                                  (const uint32_t *)sl.table.p, (uint32_t)(table_bytes / 4),
                                                                  (uint4 *)sl.h_blob.p,
                                                                  (unsigned long long)(sl.h_blob.cap & ~(size_t)15),
                                                                  (uint32_t *)sl.h_table.p);
            c->launches++;
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaEventRecord(sl.enc_done, ss));
        }
        else {
            CUDA_TRY(cudaMemcpyAsync(sl.h_table.p, sl.table.p, table_bytes, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaEventRecord(sl.enc_done, st));
        }
        sl.busy = true;
        return GCN10_OK;
    };

    // the overview levels' share of block rows [y_base, y_base + rows) of the land cover at src: one launch
    auto decimate = [&](const uint8_t *src, size_t src_pitch, int y_base, int rows, cudaStream_t st) -> int {
        OverviewParams op;
        memset(&op, 0, sizeof(op));
        op.src = src;
        op.src_pitch = src_pitch;
        op.src_y0 = y_base;
        op.w = w;
        op.h = h;
        op.col_idx = (const int32_t *)c->col_idx.p;
        op.row_idx = (const int32_t *)c->row_idx.p;
        op.with_cols = y_base == 0;
        op.nlev = nlev;
        // level row i samples block row R(i), which is non-decreasing in i: the first level row at or below block row y
        auto first_row = [&](int y, int k) -> int {
            const int hk = c->ov_h[k - 1];
            if (y >= h)
                return hk;
            const long long f = 1LL << k, a = (long long)y - f / 2;
            return a <= 0 ? 0 : (int)std::min<long long>(hk, (a + f - 1) / f);
        };
        long long most = 0;
        for (int k = 1; k <= nlev; k++) {
            op.lv[k - 1] = c->ov_lv[k - 1];
            op.lv[k - 1].i_lo = first_row(y_base, k);
            op.lv[k - 1].i_hi = first_row(y_base + rows, k);
            most = std::max(most, (long long)(op.lv[k - 1].i_hi - op.lv[k - 1].i_lo) * ((op.lv[k - 1].w + 3) / 4));
        }
        most = std::max<long long>(most, op.with_cols ? round_up((size_t)op.lv[0].w, kVecPx) : 1);
        const int blocks = (int)std::max<long long>(1, std::min<long long>((most + 255) / 256, (long long)c->sm_count * 8));
        overview_decimate_kernel<<<dim3(blocks, nlev), 256, 0, st>>>(op);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        return GCN10_OK;
    };

    auto issue = [&](int s) -> int {
        StripSlot &sl = c->slots[s % ns];
        cudaStream_t st = c->streams[s % ns];
        const StripJob &jb = jobs[s];
        const int y0 = jb.y0, rows = jb.rows;
        const int tile_rows = (rows + kTile - 1) / kTile;
        const int sw = jb.w, stx = (jb.w + kTile - 1) / kTile;
        sl.y0 = y0;
        sl.rows = rows;
        sl.level = jb.level;
        sl.y_base = jb.y_base;
        sl.tiles_x = stx;
        sl.level_w = jb.w;
        sl.level_h = jb.h;
        sl.agg = jb.agg;
        const uint8_t *strip_esa = jb.d_esa ? jb.d_esa : (const uint8_t *)sl.esa.p;
        const size_t strip_esa_pitch = jb.d_esa ? jb.pitch : dpitch;
        if (!jb.d_esa)
            CUDA_TRY(cudaMemcpy2DAsync(sl.esa.p, dpitch, esa + (size_t)y0 * esa_pitch, esa_pitch, (size_t)w, (size_t)rows,
                                       cudaMemcpyHostToDevice, st));
        if (nlev && jb.level == 0 && !jb.agg && !cog) {
            // the overview levels' share of this strip, while its land cover is on the device
            const int r2 = decimate(strip_esa, strip_esa_pitch, jb.y_base, rows, st);
            if (r2)
                return r2;
            CUDA_TRY(cudaEventRecord(sl.ov, st));
        }
        else if (jb.level) {
            // the level's land cover is complete once every full-resolution strip of the block has been sampled: the
            // last decimation on each stream (earlier bands finished theirs before their call returned)
            for (int i = 0; i < ns; i++)
                CUDA_TRY(cudaStreamWaitEvent(st, c->slots[i].ov, 0));
        }
        if (agg && jb.level == 0 && !jb.agg) {
            // the mean rasters' share of this strip, while its land cover is on the device
            AggParams a = ap;
            a.esa = strip_esa;
            a.esa_pitch = strip_esa_pitch;
            a.y0 = jb.y_base;
            a.rows = rows;
            a.ncr = (jb.y_base + rows - 1) / agg - jb.y_base / agg + 1;
            const int cells = kAggThreads / a.spc;
            const dim3 grid((acw + cells - 1) / cells, (unsigned)std::min(a.ncr * a.nchunk, 65535));
            aggregate_accumulate_kernel<<<grid, kAggThreads, 0, st>>>(a);
            c->launches++;
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaEventRecord(sl.ag, st));
        }
        if (jb.agg) {
            // the accumulators are complete once every full-resolution strip of the block has been added (earlier bands
            // finished theirs before their call returned): the first mean strip turns them into the mean rasters, the
            // others wait for that
            if (s == first_agg) {
                for (int i = 0; i < ns; i++)
                    CUDA_TRY(cudaStreamWaitEvent(st, c->slots[i].ag, 0));
                AggFinishParams fp;
                fp.acc = (uint2 *)c->agg_acc.p;
                fp.out = (uint8_t *)c->agg_out.p;
                fp.pitch = apitch;
                fp.plane_stride = apitch * (size_t)ach;
                fp.cw = acw;
                fp.ch = ach;
                fp.nsel = nplanes;
                const long long n = (long long)acw * ach * nplanes;
                aggregate_finish_kernel<<<(int)std::min<long long>((n + 255) / 256, (long long)c->sm_count * 8), 256, 0, st>>>(fp);
                c->launches++;
                CUDA_TRY(cudaGetLastError());
                CUDA_TRY(cudaEventRecord(c->agg_ready, st));
            }
            else {
                CUDA_TRY(cudaStreamWaitEvent(st, c->agg_ready, 0));
            }
        }
        // The encoder kernels run in strip order, at most two at a time (the second fills the first one's last wave):
        // launched side by side on all streams they would all finish together, and the copy of strip 0 -- the head of
        // the chain of copies that ends the block -- would wait for the others.
        // Overview strips are not chained: their grids are small (level k has 1/4^k of the tiles), one alone leaves
        // most SMs idle, and they end the block, so no later copy waits on them (with option "cog" they start it, and
        // the chain begins with the first full-resolution strip).
        if (s - 2 >= first_full && jb.level == 0 && !jb.agg)
            CUDA_TRY(cudaStreamWaitEvent(st, c->slots[(s - 2) % ns].k1, 0));
        CUDA_TRY(cudaEventRecord(sl.k0, st));
        if (fused && !jb.agg) {
            FusedParams fp;
            memset(&fp, 0, sizeof(fp));
            fp.esa = strip_esa;
            fp.esa_pitch = strip_esa_pitch;
            fp.w = sw;
            fp.rows = rows;
            fp.y_base = jb.y_base;
            fp.col_idx = jb.col_idx ? jb.col_idx : (const int32_t *)c->col_idx.p;
            fp.row_idx = jb.row_idx ? jb.row_idx : (const int32_t *)c->row_idx.p;
            fp.hsg = (const uint8_t *)c->hsg.p;
            fp.hsg_pitch = hsg_dpitch;
            fp.idmap = (const uint8_t *)c->fused_tab.p;
            fp.val = (const uint8_t *)c->fused_tab.p + 4096;
            fp.lit9 = (const unsigned long long *)((const uint8_t *)c->fused_tab.p + 4096 + kFusedIds * 32);
            memcpy(fp.cls, c->fused_cls, sizeof(fp.cls));
            fp.code = c->fused_code;
            fp.nsel = nplanes;
            fp.tiles_x = stx;
            fp.tile_rows = tile_rows;
            fp.blob = (uint8_t *)sl.blob.p;
            fp.cursor = (unsigned long long *)sl.table.p;
            fp.offsets = (unsigned long long *)((uint8_t *)sl.table.p + 16);
            fp.sizes = (uint32_t *)((uint8_t *)sl.table.p + 16 + ntile_slot * sizeof(unsigned long long));
            fp.id_hist = jb.level == 0 ? id_hist : nullptr;     // (the levels' pixels are level-0 pixels again)
            CUDA_TRY(cudaMemsetAsync(sl.table.p, 0, 16, st));
            if (nplanes <= 9)
                cn_deflate_fused_kernel<9><<<dim3(stx, tile_rows), kTile, fused_smem_bytes<9>(), st>>>(fp);
            else
                cn_deflate_fused_kernel<18><<<dim3(stx, tile_rows), kTile, fused_smem_bytes<18>(), st>>>(fp);
            c->launches++;
            CUDA_TRY(cudaGetLastError());
            return hand_over(sl, st);
        }
        uint8_t *d_out[GCN10_NPLANES] = { nullptr };
        for (int k = 0; k < nplanes; k++)
            d_out[plane_ids[k]] = jb.agg ? (uint8_t *)jb.d_esa + (size_t)k * apitch * (size_t)ach     // the mean rasters
                                         : (uint8_t *)sl.out.p + (size_t)k * dpitch * (size_t)strip_cap;
        for (int i = 0; i < nplans && !jb.agg; i++) {
            int r2 = launch_rows(c, plans[i], i, strip_esa, strip_esa_pitch, sw, rows, jb.y_base, (const uint8_t *)c->hsg.p,
                                 hsg_dpitch, hsx, hsy, map, tma_ok, d_out, dpitch, st, jb.col_idx, jb.row_idx);
            if (r2)
                return r2;
        }
        if (plane_hist && jb.level == 0 && !jb.agg) {
            PlaneHistParams hp;
            memset(&hp, 0, sizeof(hp));
            hp.planes = (const uint8_t *)sl.out.p;
            hp.plane_stride = dpitch * (size_t)strip_cap;
            hp.pitch = dpitch;
            hp.w = sw;
            hp.rows = rows;
            memcpy(hp.plane_ids, plane_ids, sizeof(int) * (size_t)nplanes);
            hp.hist = plane_hist;
            // (at least one CTA per 2^31 pixels of a plane, for the kernel's 32-bit counts)
            const long long ctas_wanted = std::max<long long>(4 * c->sm_count / nplanes, ((long long)rows * sw >> 31) + 1);
            const int ctas = (int)std::max<long long>(1, std::min<long long>(rows, ctas_wanted));
            plane_histogram_kernel<<<dim3(ctas, nplanes), 256, 0, st>>>(hp);
            c->launches++;
            CUDA_TRY(cudaGetLastError());
        }
        TileEncParams ep;
        memset(&ep, 0, sizeof(ep));
        for (int k = 0; k < nplanes; k++)
            ep.plane[k] = d_out[plane_ids[k]];
        ep.pitch = jb.agg ? apitch : dpitch;
        ep.w = sw;
        ep.rows = rows;
        ep.tiles_x = stx;
        ep.tile_rows = tile_rows;
        ep.blob = (uint8_t *)sl.blob.p;
        ep.cursor = (unsigned long long *)sl.table.p;
        ep.offsets = (unsigned long long *)((uint8_t *)sl.table.p + 16);
        ep.sizes = (uint32_t *)((uint8_t *)sl.table.p + 16 + ntile_slot * sizeof(unsigned long long));
        CUDA_TRY(cudaMemsetAsync(sl.table.p, 0, 16, st));
        deflate_tiles_kernel<<<dim3(stx, tile_rows, nplanes), kTile, kEncSmem, st>>>(ep);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        return hand_over(sl, st);
    };

    // an error inside the loop must not leave strips running on buffers the caller is about to reuse
    auto bail = [&](int code) -> int {
        for (int i = 0; i < ns; i++) {
            cudaStreamSynchronize(c->streams[i]);
            cudaStreamSynchronize(c->ship_streams[i]);
        }
        for (int i = 0; i < ns; i++)
            c->slots[i].busy = false;
        return code;
    };

    // the last strip (of any level) is on its way: a prefetched block's inflate kernel may have the SMs behind it.  (Letting it go
    // earlier -- once every strip slot is in use -- was measured: its CTAs keep the SMs until they retire, the encoder
    // kernels of the remaining strips wait for milliseconds and the chain of copies runs dry; 10.6 ms against 7.5.)
    auto release = [&](int s) -> int {
        if (s != nstrips - 1)
            return GCN10_OK;
        for (int i = 0; i < 2; i++)
            if (c->tslot[i].pending && c->tslot[i].deferred) {
                int r2 = launch_inflate(c, c->tslot[i], c->slots[s % ns].k2);
                if (r2)
                    return r2;
            }
        return GCN10_OK;
    };
    if (cog && emit_levels) {
        // the whole plane is resident: one decimation over rows [0, h), behind the land cover (esa_ready) on stream 0,
        // before the first level strip; the level strips wait for every slot's mark
        if ((rc = decimate(d_esa, d_esa_pitch, 0, h, c->streams[0])))
            return bail(rc);
        for (int i = 0; i < ns; i++)
            CUDA_TRY(cudaEventRecord(c->slots[i].ov, c->streams[0]));
    }
    for (int s = 0; s < std::min(ns, nstrips); s++)
        if ((rc = issue(s)) || (rc = release(s)))
            return bail(rc);
    for (int s = 0; s < nstrips; s++) {
        StripSlot &sl = c->slots[s % ns];
        cudaStream_t st = c->streams[s % ns];
        cudaError_t ce = cudaEventSynchronize(sl.enc_done);
        if (ce != cudaSuccess)
            return bail(fail(GCN10_ECUDA, "strip %d: %s", s, cudaGetErrorString(ce)));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, sl.k0, sl.k1);
        kernel_ms += ms;
        const size_t used = (size_t) * (const unsigned long long *)sl.h_table.p;
        if (used > blob_cap)
            return bail(fail(GCN10_ECUDA, "tile encoder overran its arena (%zu > %zu)", used, blob_cap));
        // where the strip leaves from: the re-laid copy when it fit the second arena, with framed_bytes bytes when framed
        const size_t laid = framed ? (size_t)((const unsigned long long *)sl.h_table.p)[1] : 0;
        const bool relaid = c->ordered && (framed ? laid != 0 : used <= blob2_cap);
        const size_t bytes = relaid && framed ? laid : used;
        if (!c->ship || bytes > (sl.h_blob.cap & ~(size_t)15) || (c->ordered && !relaid)) {
            // two-phase path, or a strip that outgrew the host arena: (grow it and) copy exactly `bytes` bytes
            if ((rc = ensure_host(sl.h_blob, bytes ? bytes + bytes / 4 : 16)))
                return bail(rc);
            ce = cudaMemcpyAsync(sl.h_blob.p, relaid ? sl.blob2.p : sl.blob.p, bytes, cudaMemcpyDeviceToHost, st);
            if (ce == cudaSuccess)
                ce = cudaStreamSynchronize(st);
            if (ce != cudaSuccess)
                return bail(fail(GCN10_ECUDA, "strip %d copy: %s", s, cudaGetErrorString(ce)));
        }
        // (device land cover that was still being produced when the strips were queued: its verdict, before any
        // strip reaches the caller)
        if (s == 0 && before_first_sink && (rc = before_first_sink()))
            return bail(rc);
        gcn10_tile_strip ts;
        ts.tile_row0 = sl.y_base / kTile;
        ts.n_tile_rows = (sl.rows + kTile - 1) / kTile;
        ts.tiles_x = sl.tiles_x;
        ts.n_planes = nplanes;
        ts.plane_ids = plane_ids;
        ts.offsets = (const uint64_t *)((const uint8_t *)sl.h_table.p + 16);
        ts.sizes = (const uint32_t *)((const uint8_t *)sl.h_table.p + 16 + ntile_slot * sizeof(unsigned long long));
        ts.blob = (const uint8_t *)sl.h_blob.p;
        ts.blob_bytes = bytes;
        ts.level = sl.level;
        ts.level_w = sl.level_w;
        ts.level_h = sl.level_h;
        ts.aggregate = sl.agg;
        ts.framed = framed && relaid;
        // NB: the tables are laid out [plane][strip_tile_rows (capacity)][tiles_x] only when the strip is
        // full; the kernel indexes with the strip's own tile_rows, which is what n_tile_rows reports
        const int sink_rc = sink(user, &ts);
        sl.busy = false;
        if (sink_rc)
            return bail(fail(GCN10_EINVAL, "tile sink returned %d", sink_rc));
        if (s + ns < nstrips && ((rc = issue(s + ns)) || (rc = release(s + ns))))
            return bail(rc);
    }
    c->last_kernel_ms = kernel_ms;
    if (emit_agg)
        c->agg_clean = true;
    if (c->stats && ends_block && (rc = finish_histograms(c, s0)))
        return rc;
    if (gather && !ends_block)
        c->blk_next = row0 + nrows;
    return GCN10_OK;
}

int gcn10_cuda_block_deflate_rows(gcn10_ctx *c,
                                  const uint8_t *esa, int w, int h, int row0, int nrows, size_t esa_pitch,
                                  const double gt[6],
                                  const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                                  unsigned plane_mask, gcn10_tile_sink sink, void *user)
{
    if (!esa)
        return fail(GCN10_EINVAL, "NULL argument");
    if (c && c->cog)
        return fail(GCN10_EINVAL, "option cog: a band does not hold the whole block; use gcn10_cuda_block_deflate");
    return deflate_rows_impl(c, esa, esa_pitch, nullptr, 0, nullptr, w, h, row0, nrows, gt, hsg, hsx, hsy, hsg_pitch,
                             soil_gt, plane_mask, sink, user);
}

// Upload the compressed tiles of every part and inflate them into sl.esa_full (pitch sl.dpitch) on the context's
// upload stream, without waiting: ONE kernel launch for all parts (a 36-tile edge part launched on its own would
// cost a whole tile's decode latency).  The per-tile status codes are in sl.h_status once that stream has drained.
// The inflate kernel of a slot whose uploads are on the upload stream already.  after != nullptr: not before that event
// -- the inflater keeps every SM's shared memory and registers for milliseconds, so a prefetched block's kernel is held
// back until the block in hand has issued its last strip (deflate_rows_impl) instead of starving the strips that
// follow it.
static int launch_inflate(gcn10_ctx *c, TileSlot &sl, cudaEvent_t after)
{
    if (!sl.deferred)
        return GCN10_OK;
    sl.deferred = false;
    cudaStream_t st = c->pre_stream;
    if (after)
        CUDA_TRY(cudaStreamWaitEvent(st, after, 0));
    CUDA_TRY(cudaEventRecord(sl.inf0, st));
    // a window whose tiles are all of one codec is one launch; a mosaic that mixes codecs takes one per codec
    if (sl.ntiles > sl.n_lzw) {
        inflate_tiles_kernel<<<(unsigned)(sl.ntiles - sl.n_lzw), kInflateThreads, kInflateSmem, st>>>(sl.ip);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    if (sl.n_lzw) {
        InflateParams lp = sl.ip;
        lp.order += sl.ntiles - sl.n_lzw;
        lzw_tiles_kernel<<<(unsigned)sl.n_lzw, kLzwThreads, kLzwSmem, st>>>(lp);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(sl.inf1, st));
    CUDA_TRY(cudaMemcpyAsync(sl.h_status.p, sl.ip.status, sl.ntiles * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(sl.done, st));
    return GCN10_OK;
}

// defer: only the uploads are issued; launch_inflate() follows (at the latest when the slot is consumed)
static int inflate_to_device(gcn10_ctx *c, TileSlot &sl, const gcn10_tile_part *parts, int nparts, int fill, int w, int h,
                             bool defer = false)
{
    if (!parts || nparts < 1)
        return fail(GCN10_EINVAL, "NULL argument");
    if (nparts > kInflateMaxParts)
        return fail(GCN10_EINVAL, "%d mosaic parts; at most %d are supported", nparts, kInflateMaxParts);
    if (w <= 0 || h <= 0)
        return fail(GCN10_EINVAL, "non-positive size");
    size_t ntiles = 0, blob_total = 0;
    long long covered = 0;
    for (int k = 0; k < nparts; k++) {
        const gcn10_tile_part &pt = parts[k];
        const gcn10_tile_source *src = &pt.tiles;
        if (!src->offsets || !src->sizes || (!src->blob && src->blob_bytes))
            return fail(GCN10_EINVAL, "NULL argument");
        if (pt.w <= 0 || pt.h <= 0 || src->tile_w <= 0 || src->tile_h <= 0 || src->tiles_x <= 0 || src->tiles_y <= 0)
            return fail(GCN10_EINVAL, "non-positive size");
        if (src->compression != 0 && src->compression != 8 && src->compression != 32946 && src->compression != 5)
            return fail(GCN10_EINVAL, "part %d: TIFF compression %d is not supported (0, 8 and 32946 = zlib, 5 = LZW)", k,
                        src->compression);
        if ((long long)src->tile_w * src->tile_h > (1ll << 28))
            return fail(GCN10_EINVAL, "tile of %d x %d pixels is too large", src->tile_w, src->tile_h);
        if (pt.dst_x < 0 || pt.dst_y < 0 || (long long)pt.dst_x + pt.w > w || (long long)pt.dst_y + pt.h > h)
            return fail(GCN10_EINVAL, "part %d (%d x %d at %d, %d) lies outside the %d x %d window", k, pt.w, pt.h, pt.dst_x,
                        pt.dst_y, w, h);
        if (src->x_off < 0 || src->y_off < 0 || (long long)src->x_off + pt.w > (long long)src->tiles_x * src->tile_w ||
            (long long)src->y_off + pt.h > (long long)src->tiles_y * src->tile_h)
            return fail(GCN10_EINVAL, "the %d x %d tile grid does not cover the %d x %d window at (%d, %d)", src->tiles_x,
                        src->tiles_y, pt.w, pt.h, src->x_off, src->y_off);
        const size_t n = (size_t)src->tiles_x * src->tiles_y;
        for (size_t i = 0; i < n; i++)
            if (src->sizes[i] && (src->offsets[i] > src->blob_bytes || src->sizes[i] > src->blob_bytes - src->offsets[i]))
                return fail(GCN10_EINVAL, "tile %zu lies outside the blob", ntiles + i);
        ntiles += n;
        // parts that address the same host buffer (several sources staged in one blob) share one device copy
        bool shared = false;
        for (int j = 0; j < k && !shared; j++)
            shared = parts[j].tiles.blob == src->blob && parts[j].tiles.blob_bytes == src->blob_bytes;
        if (!shared)
            blob_total += round_up(src->blob_bytes, 16);
        covered += (long long)pt.w * pt.h;
    }
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->pre_stream;
    const size_t dpitch = round_up((size_t)w, 256);
    int rc;
    // the kernel's 512-byte input refills may run ~2 KB past a stream: keep that readable
    if ((rc = ensure(sl.in_blob, round_up(blob_total, 256) + 4096)) ||
        (rc = ensure(sl.in_table, ntiles * 24)) ||
        (rc = ensure_host(sl.h_status, ntiles * (3 * sizeof(int) + 12))) ||
        (rc = ensure(sl.esa_full, dpitch * (size_t)h)))
        return rc;
    unsigned long long *d_off = (unsigned long long *)sl.in_table.p;
    uint32_t *d_size = (uint32_t *)((uint8_t *)sl.in_table.p + ntiles * 8);
    int *d_status = (int *)((uint8_t *)sl.in_table.p + ntiles * 12);
    int *d_order = (int *)((uint8_t *)sl.in_table.p + ntiles * 16);
    int *d_scratch = (int *)((uint8_t *)sl.in_table.p + ntiles * 20);
    // page-locked staging: [status | order | offsets | sizes | scratch slots]
    int *h_order = (int *)sl.h_status.p + ntiles;
    unsigned long long *h_off = (unsigned long long *)((int *)sl.h_status.p + 2 * ntiles);
    uint32_t *h_size = (uint32_t *)(h_off + ntiles);
    int *h_scratch = (int *)(h_size + ntiles);
    std::vector<uint8_t> is_lzw(ntiles);
    // tiles that are not stored whole in the plane (clipped by their part's rectangle) keep a scratch copy: the
    // inflater reads history older than its 8 KB ring back from where the bytes were flushed to
    size_t nscratch = 0, scratch_stride = 0;

    InflateParams ip;
    memset(&ip, 0, sizeof(ip));
    // window pixels no part covers read as the fill value (GDAL initialises a VRT read with the band's nodata)
    if (covered < (long long)w * h)
        CUDA_TRY(cudaMemsetAsync(sl.esa_full.p, fill & 255, dpitch * (size_t)h, st));
    size_t t0 = 0, b_next = 0, part_base[kInflateMaxParts];
    for (int k = 0; k < nparts; k++) {
        const gcn10_tile_part &pt = parts[k];
        const gcn10_tile_source *src = &pt.tiles;
        const size_t n = (size_t)src->tiles_x * src->tiles_y;
        int same = -1;
        for (int j = 0; j < k && same < 0; j++)
            if (parts[j].tiles.blob == src->blob && parts[j].tiles.blob_bytes == src->blob_bytes)
                same = j;
        const size_t b0 = same >= 0 ? part_base[same] : b_next;
        part_base[k] = b0;
        for (size_t i = 0; i < n; i++) {
            h_off[t0 + i] = (unsigned long long)b0 + src->offsets[i];
            h_size[t0 + i] = src->sizes[i];
            is_lzw[t0 + i] = src->compression == 5;
        }
        if (same < 0) {
            if (src->blob_bytes)
                CUDA_TRY(cudaMemcpyAsync((uint8_t *)sl.in_blob.p + b0, src->blob, src->blob_bytes, cudaMemcpyHostToDevice, st));
            b_next += round_up(src->blob_bytes, 16);
        }
        for (size_t i = 0; i < n; i++) {
            const long long tx0 = (long long)(i % (size_t)src->tiles_x) * src->tile_w - src->x_off;
            const long long ty0 = (long long)(i / (size_t)src->tiles_x) * src->tile_h - src->y_off;
            const bool whole = tx0 >= 0 && ty0 >= 0 && tx0 + src->tile_w <= pt.w && ty0 + src->tile_h <= pt.h;
            h_scratch[t0 + i] = (whole || !src->sizes[i]) ? -1 : (int)nscratch++;
        }
        scratch_stride = std::max(scratch_stride, round_up((size_t)src->tile_w * (size_t)src->tile_h, 256));
        InflatePart &q = ip.part[k];
        q.first_tile = (int)t0;
        q.tiles_x = src->tiles_x;
        q.tiles_y = src->tiles_y;
        q.tile_w = src->tile_w;
        q.tile_h = src->tile_h;
        q.tw_shift = (src->tile_w & (src->tile_w - 1)) == 0 ? __builtin_ctz((unsigned)src->tile_w) : -1;
        q.x_off = src->x_off;
        q.y_off = src->y_off;
        q.dst = (uint8_t *)sl.esa_full.p + (size_t)pt.dst_y * dpitch + pt.dst_x;
        q.w = pt.w;
        q.h = pt.h;
        t0 += n;
    }
    // longest streams first: a tile's decode time grows with its compressed size, and a block has only a
    // few tiles per resident CTA slot, so the order sets the tail.  LZW tiles go behind the zlib ones (their kernel
    // takes the tail of the order).
    size_t n_lzw = 0;
    for (size_t i = 0; i < ntiles; i++) {
        h_order[i] = (int)i;
        n_lzw += is_lzw[i];
    }
    std::stable_sort(h_order, h_order + ntiles, [&](int a, int b) {
        return is_lzw[a] != is_lzw[b] ? is_lzw[a] < is_lzw[b] : h_size[a] > h_size[b];
    });
    CUDA_TRY(cudaMemcpyAsync(d_order, h_order, ntiles * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_off, h_off, ntiles * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_size, h_size, ntiles * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_scratch, h_scratch, ntiles * 4, cudaMemcpyHostToDevice, st));
    if (nscratch && (rc = ensure(sl.scratch, nscratch * scratch_stride)))
        return rc;
    ip.scratch = (uint8_t *)sl.scratch.p;
    ip.scratch_index = d_scratch;
    ip.scratch_stride = scratch_stride;
    ip.blob = (const uint8_t *)sl.in_blob.p;
    ip.offsets = d_off;
    ip.sizes = d_size;
    ip.pitch = dpitch;
    ip.status = d_status;
    ip.order = d_order;
    ip.probe = c->inflate_probe;
    ip.nparts = nparts;
    sl.ip = ip;
    sl.ntiles = ntiles;
    sl.n_lzw = n_lzw;
    sl.deferred = true;
    if (!defer && (rc = launch_inflate(c, sl, nullptr)))
        return rc;
    sl.pending = true;
    sl.seq = ++c->tile_seq;
    sl.key_blob = parts[0].tiles.blob;
    sl.key_off = parts[0].tiles.offsets;
    sl.key_bytes = blob_total;
    sl.key_parts = nparts;
    sl.key_w = w;
    sl.key_h = h;
    sl.ntiles = ntiles;
    sl.dpitch = dpitch;
    return GCN10_OK;
}

static gcn10_tile_part whole_window_part(const gcn10_tile_source *src, int w, int h)
{
    gcn10_tile_part pt;
    memset(&pt, 0, sizeof(pt));
    if (src)
        pt.tiles = *src;
    pt.w = w;
    pt.h = h;
    return pt;
}

// waits for a slot's inflate, hands out the status codes, consumes the slot
static int finish_slot(gcn10_ctx *c, TileSlot &sl, int *tile_status)
{
    sl.pending = false;
    int lrc = launch_inflate(c, sl, nullptr);               // (held back and never released: now)
    if (lrc)
        return lrc;
    CUDA_TRY(cudaEventSynchronize(sl.done));                // this slot only: a later prefetch keeps running
    const int *hs = (const int *)sl.h_status.p;
    size_t bad = 0, first_bad = 0;
    for (size_t i = 0; i < sl.ntiles; i++) {
        if (tile_status)
            tile_status[i] = hs[i];
        if (hs[i] && !bad++)
            first_bad = i;
    }
    cudaEventElapsedTime(&c->last_inflate_ms, sl.inf0, sl.inf1);
    if (bad)
        return fail(GCN10_EDATA, "%zu of %zu compressed tiles could not be decoded (first: tile %zu, inflate error %d)",
                    bad, sl.ntiles, first_bad, hs[first_bad]);
    return GCN10_OK;
}

// a slot without pending work (or, both pending, the older one, whose prefetch is dropped)
static int free_slot(gcn10_ctx *c, TileSlot **out)
{
    TileSlot *sl = !c->tslot[0].pending ? &c->tslot[0] : !c->tslot[1].pending ? &c->tslot[1]
                   : c->tslot[0].seq < c->tslot[1].seq ? &c->tslot[0] : &c->tslot[1];
    if (sl->pending) {
        if (sl->deferred)
            sl->deferred = false;                       // never launched: its uploads drain in stream order
        else
            CUDA_TRY(cudaEventSynchronize(sl->done));
        sl->pending = false;
    }
    *out = sl;
    return GCN10_OK;
}

// the slot a call works with: the oldest prefetched one that matches, else a free one (inflated now)
static int acquire_slot(gcn10_ctx *c, const gcn10_tile_part *parts, int nparts, int fill, int w, int h, TileSlot **out)
{
    if (!parts || nparts < 1)
        return fail(GCN10_EINVAL, "NULL argument");
    size_t blob_total = 0, ntiles = 0;
    for (int k = 0; k < nparts; k++) {
        blob_total += round_up(parts[k].tiles.blob_bytes, 16);
        ntiles += (size_t)std::max(parts[k].tiles.tiles_x, 0) * (size_t)std::max(parts[k].tiles.tiles_y, 0);
    }
    TileSlot *hit = nullptr;
    for (int i = 0; i < 2; i++) {
        TileSlot &sl = c->tslot[i];
        if (sl.pending && sl.key_blob == parts[0].tiles.blob && sl.key_off == parts[0].tiles.offsets &&
            sl.key_bytes == blob_total && sl.key_parts == nparts &&
            sl.key_w == w && sl.key_h == h && sl.ntiles == ntiles && (!hit || sl.seq < hit->seq))
            hit = &sl;
    }
    if (!hit) {
        TileSlot *sl = nullptr;
        int rc = free_slot(c, &sl);
        if (rc || (rc = inflate_to_device(c, *sl, parts, nparts, fill, w, h)))
            return rc;
        hit = sl;
    }
    *out = hit;
    return GCN10_OK;
}

int gcn10_cuda_parts_prefetch(gcn10_ctx *c, const gcn10_tile_part *parts, int nparts, int fill, int w, int h)
{
    if (!c)
        return fail(GCN10_EINVAL, "NULL context");
    TileSlot *sl = !c->tslot[0].pending ? &c->tslot[0] : !c->tslot[1].pending ? &c->tslot[1] : nullptr;
    if (!sl)
        return fail(GCN10_EINVAL, "two prefetched blocks are already waiting; consume one first");
    // The other slot holds a block that has not been run yet: the caller is about to run it (prefetch of block k + 1,
    // then block k).  This block's inflate kernel then waits until that block has issued its last strip.
    const TileSlot &other = c->tslot[sl == &c->tslot[0] ? 1 : 0];
    return inflate_to_device(c, *sl, parts, nparts, fill, w, h, c->defer_inflate && other.pending);
}

int gcn10_cuda_tiles_prefetch(gcn10_ctx *c, const gcn10_tile_source *src, int w, int h)
{
    if (!src)
        return fail(GCN10_EINVAL, "NULL argument");
    const gcn10_tile_part pt = whole_window_part(src, w, h);
    return gcn10_cuda_parts_prefetch(c, &pt, 1, 0, w, h);
}

int gcn10_cuda_inflate_parts(gcn10_ctx *c, const gcn10_tile_part *parts, int nparts, int fill, int w, int h, uint8_t *out,
                             size_t out_pitch, int *tile_status)
{
    if (!c || !out)
        return fail(GCN10_EINVAL, "NULL argument");
    if (w > 0 && out_pitch < (size_t)w)
        return fail(GCN10_EINVAL, "pitch smaller than row width");
    TileSlot *sl = nullptr;
    int rc = acquire_slot(c, parts, nparts, fill, w, h, &sl);
    if (rc)
        return rc;
    cudaStream_t st = c->pre_stream;
    if ((rc = launch_inflate(c, *sl, nullptr)))
        return rc;
    CUDA_TRY(cudaMemcpy2DAsync(out, out_pitch, sl->esa_full.p, sl->dpitch, (size_t)w, (size_t)h, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return finish_slot(c, *sl, tile_status);
}

int gcn10_cuda_inflate_tiles(gcn10_ctx *c, const gcn10_tile_source *src, int w, int h, uint8_t *out, size_t out_pitch,
                             int *tile_status)
{
    if (!src)
        return fail(GCN10_EINVAL, "NULL argument");
    const gcn10_tile_part pt = whole_window_part(src, w, h);
    return gcn10_cuda_inflate_parts(c, &pt, 1, 0, w, h, out, out_pitch, tile_status);
}

int gcn10_cuda_block_parts_deflate(gcn10_ctx *c, const gcn10_tile_part *parts, int nparts, int fill, int w, int h,
                                   const double gt[6],
                                   const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                                   unsigned plane_mask, gcn10_tile_sink sink, void *user)
{
    if (!c)
        return fail(GCN10_EINVAL, "NULL context");
    if (!sink || !hsg || !gt || !soil_gt)
        return fail(GCN10_EINVAL, "NULL argument");
    if (!c->have_lut)
        return fail(GCN10_ENOLUT, "gcn10_cuda_set_luts() has not been called");
    TileSlot *sl = nullptr;
    int rc = acquire_slot(c, parts, nparts, fill, w, h, &sl);
    if (rc)
        return rc;
    // The strips are queued behind the inflate kernel on the device; the host does not wait for it first, so that the
    // block's set-up (soil window upload, index maps, record tables) overlaps the kernel's tail.  A damaged tile must
    // still stop the block before any output tile reaches the sink (the reference skips a block whose land cover cannot
    // be read, cn.c:188-192): the inflater's verdict is read before the first strip is handed over.
    if ((rc = launch_inflate(c, *sl, nullptr)))
        return rc;
    bool judged = false;
    rc = deflate_rows_impl(c, nullptr, 0, (const uint8_t *)sl->esa_full.p, sl->dpitch, sl->done, w, h, 0, h, gt, hsg,
                           hsx, hsy, hsg_pitch, soil_gt, plane_mask, sink, user, [&]() -> int {
                               judged = true;
                               return finish_slot(c, *sl, nullptr);
                           });
    if (!judged) {
        // the call failed before its first strip (bad arguments, CUDA error): the slot is consumed all the same
        const int frc = finish_slot(c, *sl, nullptr);
        if (!rc)
            rc = frc;
    }
    return rc;
}

int gcn10_cuda_block_tiles_deflate(gcn10_ctx *c, const gcn10_tile_source *esa_tiles, int w, int h, const double gt[6],
                                   const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                                   unsigned plane_mask, gcn10_tile_sink sink, void *user)
{
    if (!esa_tiles)
        return fail(GCN10_EINVAL, "NULL argument");
    const gcn10_tile_part pt = whole_window_part(esa_tiles, w, h);
    return gcn10_cuda_block_parts_deflate(c, &pt, 1, 0, w, h, gt, hsg, hsx, hsy, hsg_pitch, soil_gt, plane_mask, sink, user);
}

int gcn10_cuda_last_inflate_ms(gcn10_ctx *c, float *ms)
{
    if (!c || !ms)
        return fail(GCN10_EINVAL, "NULL argument");
    *ms = c->last_inflate_ms;
    return GCN10_OK;
}

int gcn10_cuda_pcie_probe(gcn10_ctx *c, size_t bytes, int reps, double gbs[3])
{
    if (!c || !gbs || bytes < 4096 || reps < 1)
        return fail(GCN10_EINVAL, "bad argument");
    if (c->pending_events)
        return fail(GCN10_EINVAL, "asynchronous blocks are pending on this context: gcn10_cuda_wait() for them first");
    CUDA_TRY(cudaSetDevice(c->device));
    bytes &= ~(size_t)15;
    DevBuf d, cur;
    HostBuf hb;
    int rc;
    if ((rc = ensure(d, bytes)) || (rc = ensure(cur, 16)) || (rc = ensure_host(hb, bytes))) {
        release(d);
        release(cur);
        release_host(hb);
        return rc;
    }
    memset(hb.p, 0x5A, bytes);
    cudaStream_t st = c->streams[0];
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const unsigned long long n = bytes;
    cudaMemcpyAsync(cur.p, &n, sizeof(n), cudaMemcpyHostToDevice, st);
    cudaStreamSynchronize(st);
    for (int leg = 0; leg < 3; leg++) {
        for (int i = -1; i < reps; i++) {           // i = -1: warm-up
            if (i == 0)
                cudaEventRecord(e0, st);
            if (leg == 0)
                cudaMemcpyAsync(d.p, hb.p, bytes, cudaMemcpyHostToDevice, st);
            else if (leg == 1)
                cudaMemcpyAsync(hb.p, d.p, bytes, cudaMemcpyDeviceToHost, st);
            else {
                ship_strip_kernel<<<kShipCtas, kShipThreads, 0, st>>>((const uint4 *)d.p, (const unsigned long long *)cur.p, nullptr, 0u,
                                                             (uint4 *)hb.p, (unsigned long long)bytes, nullptr);
                c->launches++;
            }
        }
        cudaEventRecord(e1, st);
        cudaStreamSynchronize(st);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        gbs[leg] = ms > 0.f ? (double)bytes * reps / (ms * 1e-3) / 1e9 : 0.0;
    }
    const cudaError_t ce = cudaGetLastError();
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    release(d);
    release(cur);
    release_host(hb);
    if (ce != cudaSuccess)
        return fail(GCN10_ECUDA, "pcie probe: %s", cudaGetErrorString(ce));
    return GCN10_OK;
}

int gcn10_cuda_bind_host_thread(int device)
{
    char bus[32] = "";
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    for (char *q = bus; *q; q++)
        *q = (char)tolower((unsigned char)*q);
    char path[256];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE *f = fopen(path, "r");
    int node = -1;
    if (!f || fscanf(f, "%d", &node) != 1)
        node = -1;
    if (f)
        fclose(f);
    if (node < 0)
        return -2;
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f)
        return -3;
    cpu_set_t set;
    CPU_ZERO(&set);
    int a, b, n = 0;
    // cpulist: comma separated ranges "0-15,32-47"
    while (fscanf(f, "%d", &a) == 1) {
        b = a;
        int ch = fgetc(f);
        if (ch == '-') {
            if (fscanf(f, "%d", &b) != 1)
                break;
            ch = fgetc(f);
        }
        for (int cpu = a; cpu <= b && cpu < CPU_SETSIZE; cpu++, n++)
            CPU_SET(cpu, &set);
        if (ch != ',')
            break;
    }
    fclose(f);
    if (n == 0 || sched_setaffinity(0, sizeof(set), &set) != 0)
        return -4;
    return node;
}

void *gcn10_cuda_host_alloc(size_t bytes)
{
    void *p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        fail(GCN10_ENOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
        return nullptr;
    }
    return p;
}

void gcn10_cuda_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

int gcn10_cuda_host_register(void *p, size_t bytes)
{
    if (!p || !bytes)
        return fail(GCN10_EINVAL, "NULL or empty range");
    CUDA_TRY(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return GCN10_OK;
}

int gcn10_cuda_host_unregister(void *p)
{
    if (!p)
        return fail(GCN10_EINVAL, "NULL pointer");
    CUDA_TRY(cudaHostUnregister(p));
    return GCN10_OK;
}

}  // extern "C"
