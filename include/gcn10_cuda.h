/* include/gcn10_cuda.h -- C ABI of libgcn10cuda.so, the B200 (sm_100a) implementation of
 * GCN10's per-block Curve Number hot path.
 *
 * The reference (clawrim/gcn10) has no plugin or FFI interface; its only seam around the
 * hot path is the plain C function
 *
 *     void process_block(int block_id, bool overwrite, int total_blocks);
 *                                            -- /root/reference/src/global.h:58
 *
 * whose body (/root/reference/src/cn.c:134-384) loads two byte rasters with load_raster()
 * (global.h:54-55), runs five full-raster CPU passes per output (cn.c:218-232, 274, 275,
 * 289, 290) and hands 18 byte planes to save_raster() (global.h:56-57).  This library
 * replaces exactly the part between "load_raster returned" and "save_raster is called":
 * the entry points below take the same byte rasters and geotransforms that load_raster()
 * produces and return the same byte planes that save_raster() consumes.  INTEGRATION.md shows
 * the replacement cn.c that a maintainer of the reference would write on top of it, and
 * gcn10_b200/host/ holds this repository's own host program built that way.
 *
 * Conventions
 *   - plain pointers and sizes only; no CUDA, C++ or torch types in any signature
 *     (a stream is passed as an opaque void*: a cudaStream_t / CUstream value, NULL = the
 *     context's own stream);
 *   - every function that can fail returns int: 0 = GCN10_OK, negative = error code, and
 *     gcn10_cuda_last_error() returns a human-readable message for the calling thread;
 *   - a gcn10_ctx is bound to one GPU and must be used by one host thread at a time
 *     (one context per worker thread per GPU, mirroring one MPI rank per process in the
 *     reference, /root/reference/src/main.c:80-82,171);
 *   - there is no CPU fallback: without a usable CUDA device every compute entry point fails
 *     with GCN10_ENODEV / GCN10_ECUDA.
 *
 * Plane numbering (the reference's save order, cn.c:145-147,236,258-259,308):
 *     plane = cond * 9 + hc * 3 + arc,  cond: 0 drained, 1 undrained
 *                                       hc:   0 p, 1 f, 2 g       arc: 0 i, 1 ii, 2 iii
 * A plane mask selects planes by bit (1u << plane).
 */
#ifndef GCN10_CUDA_H
#define GCN10_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCN10_NVARIANTS 9           /* lookup tables per drainage condition             */
#define GCN10_NPLANES   18          /* rasters per block (cn.c:236,258-259)             */
#define GCN10_NODATA    255         /* cn.c:38,289                                       */

#define GCN10_MASK_DRAINED   0x001FFu       /* planes 0..8   (cn_rasters_drained/)      */
#define GCN10_MASK_UNDRAINED 0x3FE00u       /* planes 9..17  (cn_rasters_undrained/)    */
#define GCN10_MASK_ALL       0x3FFFFu

enum {
    GCN10_OK      = 0,
    GCN10_EINVAL  = -1,     /* bad argument (NULL, non-positive size, pitch < width, ...) */
    GCN10_ECUDA   = -2,     /* a CUDA runtime/driver call failed                          */
    GCN10_ENOMEM  = -3,     /* host or device allocation failed                           */
    GCN10_ENOLUT  = -4,     /* gcn10_cuda_set_luts() has not been called                  */
    GCN10_ENODEV  = -5,     /* no CUDA device / device index out of range                 */
    GCN10_EDATA   = -6      /* a compressed input tile is not a valid zlib stream of the tile's size
                               (the recoverable tier: GDALRasterIO failing at raster.c:177-186)  */
};

typedef struct gcn10_ctx gcn10_ctx;

/* Library identification, e.g. "gcn10cuda 0.1.0 (sm_100a)". */
const char *gcn10_cuda_version(void);

/* Message describing the last failure on the calling thread ("" if none). */
const char *gcn10_cuda_last_error(void);

/* Number of CUDA devices visible to the process; negative error code on failure.
 * Replaces MPI_Comm_size() as the worker count (main.c:82). */
int gcn10_cuda_device_count(void);

/* Create / destroy a per-GPU context (streams, LUT storage, staging buffers). */
int gcn10_cuda_create(int device, gcn10_ctx **out);
void gcn10_cuda_destroy(gcn10_ctx *ctx);

/* Install the nine lookup tables.  Element layout and order are exactly those of the
 * reference: int table[256][5] indexed [land cover][soil group] as filled by
 * load_lookup_table() (cn.c:13-85, declared cn.c:148), tables in loop order
 * p_i, p_ii, p_iii, f_i, f_ii, f_iii, g_i, g_ii, g_iii (cn.c:146-147,258-259).
 * A value v is emitted as (uint8_t)v when v < 255 and as 255 otherwise (cn.c:126-128,289). */
int gcn10_cuda_set_luts(gcn10_ctx *ctx, const int tables[GCN10_NVARIANTS][256][5]);

/* One block, inputs and outputs in HOST memory (replaces cn.c:208-290 and the buffers that
 * flow into save_raster at cn.c:363).  Synchronous.  Internally the block is cut into row
 * strips that are pipelined host->device copy / kernel / device->host copy over several
 * streams.  Copies are asynchronous when the buffers are page-locked
 * (gcn10_cuda_host_alloc / gcn10_cuda_host_register), otherwise staged by the driver.
 *
 *   esa, w, h, esa_pitch   land cover window from load_raster (cn.c:187); row y starts at
 *                          esa + y*esa_pitch (the reference has esa_pitch == w)
 *   gt                     its clipped geotransform (raster.c:157-162)
 *   hsg, hsx, hsy,         coarse HYSOGs window (cn.c:195-196) and its geotransform
 *   hsg_pitch, soil_gt
 *   plane_mask             which of the 18 planes to produce
 *   out[18], out_pitch     destination of plane k = out[k] (ignored where the mask bit is 0)
 */
int gcn10_cuda_block(gcn10_ctx *ctx,
                     const uint8_t *esa, int w, int h, size_t esa_pitch, const double gt[6],
                     const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                     unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch);

/* Asynchronous form of gcn10_cuda_block(): queues the whole block -- upload of the HSG window, fp64 index maps, and
 * per row strip the host->device copy, the fused kernel and the device->host copies of the planes -- on the context's
 * streams and returns at once; the host thread is free to read the next block (load_raster of block i+1, cn.c:187)
 * or write the previous one (save_raster, cn.c:363) meanwhile.  esa, hsg and the out[] planes must stay valid, and
 * out[] must not be read, until gcn10_cuda_wait(*done) has returned; page-locked buffers (gcn10_cuda_host_alloc /
 * _register) are what makes the copies truly asynchronous.  Several blocks may be queued on one context; they run in
 * order.  Until every queued block has been waited for, the context accepts no other compute call.
 *
 *     gcn10_event *ev[2];
 *     gcn10_cuda_block_async(ctx, esa[0], ..., out[0], pitch, &ev[0]);
 *     gcn10_cuda_block_async(ctx, esa[1], ..., out[1], pitch, &ev[1]);     -- runs behind block 0
 *     gcn10_cuda_wait(ev[0]);  save_raster(out[0][k], ...);  ...
 */
typedef struct gcn10_event gcn10_event;
int gcn10_cuda_block_async(gcn10_ctx *ctx,
                           const uint8_t *esa, int w, int h, size_t esa_pitch, const double gt[6],
                           const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                           unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch,
                           gcn10_event **done);

/* Blocks until the block behind `done` is complete in host memory, releases the event and returns the block's status
 * (GCN10_OK or the error met while queueing / running it). */
int gcn10_cuda_wait(gcn10_event *done);

/* 1 = the block behind `done` has finished, 0 = still running, negative = error.  Does not release the event. */
int gcn10_cuda_event_query(gcn10_event *done);

/* Rows [row0, row0+nrows) of a w x h block: esa and out[k] point at row `row0` (the caller holds
 * only that band of the rasters), while gt / soil_gt / h still describe the WHOLE block so that the
 * fp64 index maps are the block's (a band with a shifted geotransform origin would not round the
 * same way).  Lets a host program stream a 36000 x 36000 block through a few hundred MB of pinned
 * memory, band by band, aligned to the 256-row tiles of the output GeoTIFFs. */
int gcn10_cuda_block_rows(gcn10_ctx *ctx,
                          const uint8_t *esa, int w, int h, int row0, int nrows, size_t esa_pitch,
                          const double gt[6],
                          const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                          unsigned plane_mask, uint8_t *const out[GCN10_NPLANES], size_t out_pitch);

/* One block, outputs delivered as DEFLATE-compressed 256 x 256 GeoTIFF tiles instead of raw planes.
 *
 * This fuses the reference's save_raster() encode step (raster.c:204-219: GTiff, TILED=YES,
 * COMPRESS=DEFLATE) into the GPU pipeline: after the Curve Number kernel, every tile of every
 * selected plane is compressed on the device into a complete zlib stream (exactly what a TIFF
 * Compression=8 tile holds), and only the compressed tiles cross PCIe.  Tiles on the right / bottom
 * edge are zero padded to 256 x 256.  The block is processed in strips of whole tile rows; `sink` is
 * called once per strip, in order, from the calling thread.  The memory behind strip->blob / offsets /
 * sizes is page-locked, owned by the library and valid only during the call: copy or write it out.
 * A non-zero return from `sink` aborts the block (returned as GCN10_EINVAL).
 *
 * Overviews (option "overviews" = n > 0): after the block's last full-resolution strip the same sink receives the
 * block's overview levels 1 .. gcn10_overview_levels(w, h, n), level 1 first, each in tile-row order, in strips of at
 * most "strip_rows" rows of that level (strip->level, level_w, level_h say which level and its size).  Level k of every
 * plane is the plane sampled by gcn10_overview_src, so each of its pixels is a full-resolution output pixel.  This
 * holds for gcn10_cuda_block_deflate, _block_deflate_rows, _block_tiles_deflate and _block_parts_deflate; the raw-plane
 * calls (gcn10_cuda_block*, _block_device) ignore the option.  The levels cost device memory of about a third of the
 * block (about 0.44 GB for 36001 x 36001), kept on the context.
 *
 * Mean rasters (option "aggregate" = f >= 2): after the full-resolution strips and the overview levels the same sink
 * receives, for every selected plane, the block's f x f mean raster (gcn10_aggregate_dim / _value below) as 256 x 256
 * DEFLATE tiles, in tile-row order, in strips of at most "strip_rows" rows (strip->aggregate = f, level = 0, level_w x
 * level_h = the mean raster's size).  The same four calls deliver it; the raw-plane calls ignore the option.  The
 * full-resolution strips and overview levels are the same bytes as without the option, and "stats" does not count the
 * mean strips.  The accumulators cost 8 bytes per cell and selected plane on the context (computed: about 0.3 GB for
 * 18 planes of 36001 x 36001 at f = 25).
 *
 * Cloud Optimized GeoTIFF order (option "cog" = 1): a COG holds the smallest overview level's tiles first and the full
 * resolution last, so gcn10_cuda_block_deflate, _block_tiles_deflate and _block_parts_deflate then deliver the strips
 * in that order: the overview levels nlev .. 1 (the smallest first, each in tile-row order), then the full-resolution
 * strips, then the mean rasters.  The levels are made in one pass over the block's land cover before the first strip,
 * so the whole block must be on the device: the tiles and parts calls inflate it there anyway, and
 * gcn10_cuda_block_deflate uploads the caller's raster whole (w x h bytes of device memory, in a tile slot that holds
 * no prefetched block) instead of strip by strip.  _block_deflate_rows refuses the option (GCN10_EINVAL): a band does
 * not hold the whole block.  With "ordered" on as well, every tile of a re-laid strip also gets the block leader and
 * trailer of the COG layout on the device (strip->framed, 8 more bytes per tile), so a consumer still writes a plane's
 * share of a strip with one write.  The tile streams, the histograms of "stats" and the mean rasters are the same
 * bytes as without the option; only their order and framing change.  The raw-plane calls ignore the option. */
typedef struct {
    int tile_row0;              /* first tile row (of the block) in this strip                    */
    int n_tile_rows;            /* tile rows in this strip                                        */
    int tiles_x;                /* tiles per tile row = ceil(w / 256)                             */
    int n_planes;               /* planes selected by the mask                                    */
    const int *plane_ids;       /* [n_planes] plane numbers, ascending                            */
    const uint64_t *offsets;    /* [n_planes][n_tile_rows][tiles_x] byte offset of a tile in blob */
    const uint32_t *sizes;      /* [n_planes][n_tile_rows][tiles_x] bytes of its zlib stream      */
    const uint8_t *blob;        /* the compressed tiles of the strip                              */
    size_t blob_bytes;
    /* overview levels (option "overviews"): 0 = a full-resolution strip; k >= 1 = a strip of overview level k,
     * whose level_w x level_h raster has its own tile grid (tile_row0 and tiles_x then refer to that grid).
     * level_w x level_h is the raster the strip's tile grid covers: the block itself at level 0. */
    int level;
    int level_w, level_h;
    /* mean rasters (option "aggregate"): 0 = a Curve Number strip (full resolution or overview); f = a strip of the
     * block's f x f mean raster, whose level_w x level_h = gcn10_aggregate_dim(w, f) x gcn10_aggregate_dim(h, f)
     * cells have their own tile grid (level is then 0) */
    int aggregate;
    /* option "cog" with "ordered": 1 = every tile in blob carries the block leader and trailer of a Cloud Optimized
     * GeoTIFF -- the 4 bytes before blob + offsets[i] hold sizes[i] as a uint32 LE, the 4 bytes after the stream repeat
     * its last 4 bytes (offsets and sizes still address the stream itself).  0 without the option, and for a strip
     * that did not fit the re-laying arena and left unordered. */
    int framed;
} gcn10_tile_strip;

/* Overview levels: nearest-neighbour reductions by 2^k of a block, sampled from full resolution.
 * Every layer (library, GeoTIFF writer, tests) uses these three rules.
 *
 *   gcn10_overview_dim(n, k)        pixels of level k along an n-pixel axis: ceil(n / 2^k) (GDAL's overview size)
 *   gcn10_overview_src(i, k, n)     the full-resolution pixel that level pixel i samples: the one holding the centre
 *                                   of the level cell, min(i * 2^k + 2^(k-1), n - 1); every level samples level 0
 *   gcn10_overview_levels(w, h, m)  levels k = 1, 2, ... are made while level k - 1 is wider or taller than one
 *                                   256-pixel tile, at most m (gdaladdo's automatic rule): 8 for 36000 x 36000 and
 *                                   36001 x 36001, none for a block that fits in one tile */
#ifdef __CUDACC__
#define GCN10_HOST_DEVICE __host__ __device__        /* the library's kernels sample by the same rule */
#else
#define GCN10_HOST_DEVICE
#endif

static inline GCN10_HOST_DEVICE int gcn10_overview_dim(int n, int k) { return (int)(((long long)n + (1LL << k) - 1) >> k); }

static inline GCN10_HOST_DEVICE int gcn10_overview_src(int i, int k, int n)
{
    const long long s = ((long long)i << k) + ((1LL << k) >> 1);
    return s < n - 1 ? (int)s : n - 1;
}

static inline int gcn10_overview_levels(int w, int h, int max_levels)
{
    int k = 0;
    while (k < max_levels && (gcn10_overview_dim(w, k) > 256 || gcn10_overview_dim(h, k) > 256))
        k++;
    return k;
}

#define GCN10_MAX_OVERVIEWS 16

/* Mean rasters (option "aggregate" = f): the f x f mean of every selected plane, the composite Curve Number of a
 * coarse cell (TR-55; GDAL's "-r average").  Every layer (library, GeoTIFF writer, host program, tests) uses these
 * rules.
 *
 *   gcn10_aggregate_dim(n, f)          cells along an n-pixel axis: ceil(n / f).  Cells are aligned to the block's
 *                                      pixel (0, 0); an edge cell covers the pixels it has (GDAL's edge overview cell)
 *   gcn10_aggregate_value(sum, count)  a cell's value from the sum and the number of its pixels that are not 255:
 *                                      the mean rounded half up, (2 sum + count) / (2 count) in integers, and 255
 *                                      only when every pixel of the cell is 255 (GDAL's "average" rule).  Valid values
 *                                      are <= 254, so the mean never collides with nodata.
 *   gcn10_aggregate_gt(gt, f, out)     the mean raster's geotransform: { gt0, gt1 f, gt2 f, gt3, gt4 f, gt5 f }
 *
 * f <= GCN10_MAX_AGGREGATE keeps a cell's sum (<= 1024^2 * 254) and count inside uint32.
 *
 * Edge wart: a window of the shipped VRT is 36001 x 36001 pixels (ceil of 36000.00000000125), so at f = 25 its last
 * cell row and column are one pixel wide.  That pixel is the first pixel of the neighbouring block's window (both
 * windows' pixel offsets are floor of the block's origin in VRT pixels, and the origins are 36000 pixels apart), so
 * the neighbour's first cell covers the footprint in full; the one-pixel cell is the same duplicated pixel that the
 * full-resolution outputs already carry. */
#define GCN10_MAX_AGGREGATE 1024

static inline GCN10_HOST_DEVICE int gcn10_aggregate_dim(int n, int f) { return (int)(((long long)n + f - 1) / f); }

static inline GCN10_HOST_DEVICE uint8_t gcn10_aggregate_value(uint32_t sum, uint32_t count)
{
    return count ? (uint8_t)((2ull * sum + count) / (2ull * count)) : (uint8_t)GCN10_NODATA;
}

static inline void gcn10_aggregate_gt(const double gt[6], int f, double out[6])
{
    out[0] = gt[0];
    out[1] = gt[1] * f;
    out[2] = gt[2] * f;
    out[3] = gt[3];
    out[4] = gt[4] * f;
    out[5] = gt[5] * f;
}

typedef int (*gcn10_tile_sink)(void *user, const gcn10_tile_strip *strip);

int gcn10_cuda_block_deflate(gcn10_ctx *ctx,
                             const uint8_t *esa, int w, int h, size_t esa_pitch, const double gt[6],
                             const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                             unsigned plane_mask, gcn10_tile_sink sink, void *user);

/* Band form of gcn10_cuda_block_deflate (see gcn10_cuda_block_rows): esa points at block row `row0`,
 * which must be a multiple of 256; nrows must be a multiple of 256 unless the band ends the block.
 * With option "overviews", "stats" or "aggregate" the bands of a block feed its levels, histograms and mean rasters,
 * which stay on the context between calls: a band with row0 == 0 starts a block, every later band must start where the
 * previous one ended (same w and h, and with "stats" or "aggregate" the same plane mask; anything else is refused with
 * GCN10_EINVAL), and the band that ends the block (row0 + nrows == h) delivers the levels and the mean rasters after
 * its own strips and completes the histograms. */
int gcn10_cuda_block_deflate_rows(gcn10_ctx *ctx,
                                  const uint8_t *esa, int w, int h, int row0, int nrows, size_t esa_pitch,
                                  const double gt[6],
                                  const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                                  unsigned plane_mask, gcn10_tile_sink sink, void *user);

/* Land cover handed over as the COMPRESSED tiles of a tiled GeoTIFF instead of a decoded raster.
 *
 * The reference obtains its land-cover window from load_raster() (raster.c:106-189), where GDAL inflates
 * the TIFF tiles on the CPU (GDALRasterIO, raster.c:177-179; the ESA WorldCover files are 1024 x 1024
 * DEFLATE tiles, landcover/esa_worldcover_2021.vrt).  With a gcn10_tile_source the caller passes the
 * tiles that intersect the window exactly as they lie in the file (TIFF Compression 8 or 32946: one zlib
 * stream per tile, no predictor) and the library inflates them on the GPU, one warp per tile, directly
 * into the device-resident land-cover plane.  Only compressed bytes cross PCIe.
 *
 *   tile_w, tile_h     TIFF TileWidth / TileLength (any positive size)
 *   tiles_x, tiles_y   the tile grid handed over (row-major in offsets / sizes)
 *   x_off, y_off       position of the window's pixel (0, 0) inside that grid, i.e. window pixel (x, y)
 *                      is pixel (x_off + x, y_off + y) of the grid; the grid must cover the w x h window
 *   blob, blob_bytes   the tiles' bytes (host memory; page-locked memory makes the copy asynchronous)
 *   offsets, sizes     per tile: start of its zlib stream in blob and its length; size 0 = a sparse tile,
 *                      read as zeros (what GDAL returns for a tile that was never written)
 *   compression        the file's TIFF Compression tag: 0, 8 or 32946 = zlib streams; 5 = LZW (new style, no
 *                      predictor: what gdal_translate -co COMPRESS=LZW writes), decoded on the GPU as well, with
 *                      libtiff's rules.  Any other value is refused with GCN10_EINVAL.  Every _tiles_ and _parts_ call
 *                      takes it per part, so the parts of one mosaic may differ.
 *
 * The compression field was appended to the struct; 0 selects zlib, so a caller that zero-initialises the struct
 * keeps working unchanged.  The change is source-compatible but not binary-compatible (gcn10_tile_part embeds the
 * struct): callers must be recompiled.
 */
typedef struct {
    int tile_w, tile_h;
    int tiles_x, tiles_y;
    int x_off, y_off;
    const uint8_t *blob;
    size_t blob_bytes;
    const uint64_t *offsets;
    const uint32_t *sizes;
    int compression;
} gcn10_tile_source;

/* Inflate the tiles of `src` on the GPU and return the w x h window as a raster in HOST memory
 * (the load_raster() half alone).  tile_status, if not NULL, receives tiles_x * tiles_y codes: 0 = ok,
 * 1..10 = the reason a tile could not be decoded (see inflate_core.h; 10 = the stream's Adler-32 trailer does not
 * match the decoded bytes, which zlib reports to GDAL as a data error).  LZW tiles (compression 5) report 8 when the
 * input ends and 9 when EOI comes before the tile is full (libtiff's "Not enough data"), 11 for an old-style
 * (pre-TIFF 5.0, LSB-first) stream, which is not supported, and 12 for a code libtiff refuses: above the next free
 * entry, a first code after Clear above 257, a code before the first Clear, or a table that overflows without a Clear
 * (lzw_core.h).  Returns GCN10_EDATA if any tile failed (the window is then incomplete). */
int gcn10_cuda_inflate_tiles(gcn10_ctx *ctx, const gcn10_tile_source *src, int w, int h,
                             uint8_t *out, size_t out_pitch, int *tile_status);

/* gcn10_cuda_block_deflate with the land cover given as compressed tiles: inflate on the GPU, Curve
 * Number kernel, tile DEFLATE on the GPU, compressed tiles back.  The whole load_raster -> cn.c ->
 * save_raster chain of process_block() (cn.c:187-363) with compressed bytes on PCIe in both directions.
 * Returns GCN10_EDATA (and calls the sink for no strip) if a land-cover tile cannot be decoded. */
int gcn10_cuda_block_tiles_deflate(gcn10_ctx *ctx, const gcn10_tile_source *esa_tiles, int w, int h,
                                   const double gt[6],
                                   const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                                   unsigned plane_mask, gcn10_tile_sink sink, void *user);

/* Starts the upload and the GPU inflate of a block's land-cover tiles and returns without waiting.  The next
 * gcn10_cuda_block_tiles_deflate / gcn10_cuda_inflate_tiles call on this context with the same tile source (same
 * blob and offsets pointers, same size, same w x h) picks the result up instead of starting over, so a caller that knows its next
 * block overlaps that block's upload + inflate with the current block's Curve Number strips:
 *
 *     gcn10_cuda_tiles_prefetch(ctx, &tiles[i + 1], w, h);
 *     gcn10_cuda_block_tiles_deflate(ctx, &tiles[i], w, h, ...);        -- prefetched in the previous iteration
 *
 * The memory behind src->blob / offsets / sizes must stay valid and unchanged until that call has returned.
 * At most two blocks can be waiting.  When the other waiting block has not been run yet (the order above), the upload
 * starts at once but the inflate kernel is queued behind that block's last strip: an inflate kernel occupies every SM
 * for milliseconds, and started earlier it would hold up the strips whose copies end the block in hand (option
 * "defer_inflate").  (Replaces nothing in the reference: its ranks read one block at a time,
 * cn.c:187.) */
int gcn10_cuda_tiles_prefetch(gcn10_ctx *ctx, const gcn10_tile_source *src, int w, int h);

/* Land cover that comes from a MOSAIC of tiled GeoTIFFs -- what the reference's shipped configuration opens:
 * esa_data_path = landcover/esa_worldcover_2021.vrt, a GDAL VRT of 2651 36000 x 36000 files (raster.c:119).  With the
 * VRT's pixel size a 3-degree block window is 36001 x 36001 and touches four files.  A part is one source file's share
 * of the window: its tile grid (as in gcn10_tile_source; x_off / y_off locate the part's pixel (0, 0) inside the grid)
 * and the rectangle of the window it fills.  All parts are uploaded and inflated by one kernel launch; window pixels
 * that no part covers read as `fill` (the VRT band's NoDataValue).  Parts must not overlap.  At most 9 parts.
 * The _parts_ calls are the general form of gcn10_cuda_tiles_prefetch / _inflate_tiles / _block_tiles_deflate. */
typedef struct {
    gcn10_tile_source tiles;
    int dst_x, dst_y;           /* position of the part inside the block window */
    int w, h;                   /* size of the part */
} gcn10_tile_part;

int gcn10_cuda_parts_prefetch(gcn10_ctx *ctx, const gcn10_tile_part *parts, int nparts, int fill, int w, int h);
int gcn10_cuda_inflate_parts(gcn10_ctx *ctx, const gcn10_tile_part *parts, int nparts, int fill, int w, int h,
                             uint8_t *out, size_t out_pitch, int *tile_status);
int gcn10_cuda_block_parts_deflate(gcn10_ctx *ctx, const gcn10_tile_part *parts, int nparts, int fill, int w, int h,
                                   const double gt[6],
                                   const uint8_t *hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                                   unsigned plane_mask, gcn10_tile_sink sink, void *user);

/* Device time of the inflate kernel of the most recent gcn10_cuda_inflate_tiles /
 * gcn10_cuda_block_tiles_deflate call (CUDA events on the launching stream). */
int gcn10_cuda_last_inflate_ms(gcn10_ctx *ctx, float *ms);

/* Same computation with every buffer already in DEVICE memory; asynchronous on `stream`
 * (NULL = the context's own non-blocking stream; to use the legacy default stream pass
 * cudaStreamLegacy, i.e. (void *)1).  Fast path requirements: esa, every selected out[k], and
 * both pitches 16-byte aligned; otherwise a slower byte-wise kernel is used.  hsg may have
 * any alignment (16-byte aligned base and pitch enable the TMA staging path). */
int gcn10_cuda_block_device(gcn10_ctx *ctx,
                            const uint8_t *d_esa, int w, int h, size_t esa_pitch, const double gt[6],
                            const uint8_t *d_hsg, int hsx, int hsy, size_t hsg_pitch, const double soil_gt[6],
                            unsigned plane_mask, uint8_t *const d_out[GCN10_NPLANES], size_t out_pitch,
                            void *stream);

/* The separable pixel -> HSG cell maps of cn.c:219-229, evaluated on the GPU in fp64 with
 * the reference's exact operation order; copies col_index[w] and row_index[h] to the host.
 * Diagnostic / test entry point (the block calls compute these maps internally). */
int gcn10_cuda_index_maps(gcn10_ctx *ctx, int w, int h, const double gt[6],
                          int hsx, int hsy, const double soil_gt[6],
                          int32_t *col_index, int32_t *row_index);

/* Wait for everything queued on the context's streams. */
int gcn10_cuda_synchronize(gcn10_ctx *ctx);

/* Device time of the fused kernels of the most recent gcn10_cuda_block() call (sum over its
 * strips, overview strips included), measured with CUDA events on the launching streams. */
int gcn10_cuda_last_kernel_ms(gcn10_ctx *ctx, float *ms);

/* Number of kernels this context has launched since it was created. */
int gcn10_cuda_launch_count(gcn10_ctx *ctx, uint64_t *launches);

/* Per-plane histograms of the full-resolution pixels of the last block that a compressed-tile call completed with
 * option "stats" on: hist[p][v] = pixels of plane p with value v (255 = nodata).  Rows of planes outside the mask are
 * zero; every selected row sums to w * h.  GCN10_EINVAL if no such block has completed since the option was set
 * (a band call completes its block with the band that ends it; a call that starts a block clears the last one).
 * The GPU counts them while it encodes (gcn10_cuda_block_deflate, _block_deflate_rows, _block_tiles_deflate and
 * _block_parts_deflate; the raw-plane calls ignore the option, their callers hold the planes): overview levels are
 * not counted, and the tiles are the same bytes as without the option. */
int gcn10_cuda_last_histograms(gcn10_ctx *ctx, uint64_t hist[GCN10_NPLANES][256]);

/* Tunables: "strip_rows" (rows per pipelined strip in the host-buffer calls), "streams" (1..8), "rows_per_cta"
 * (0 = automatic), "tma" (0 = always use the gather fallback for HSG staging), "fused" (0 = compressed-tile
 * calls run the Curve Number kernel and the per-plane tile encoder instead of the fused kernel), "ship" (1 = a strip's
 * compressed bytes leave through a kernel that writes them into mapped page-locked memory, instead of the default
 * size read-back + copy-engine transfer), "ordered" (1 = every strip is re-laid on the device in table order -- [plane][tile row][tile column], streams on
 * 16-byte boundaries, offsets ascending -- so that a consumer can write a plane's share of a strip with one write),
 * "tuned_code" (0 = tile streams use RFC 1951's fixed Huffman code instead
 * of the tuned one), "defer_inflate" (0 = the inflate kernel of a prefetched block starts at once instead of behind
 * the last strip of the block in hand), "overviews" (0..16, default 0: the compressed-tile calls also deliver up to that
 * many overview levels of the block, see gcn10_cuda_block_deflate), "stats" (0 / 1, default 0: the compressed-tile calls
 * also count every selected plane's histogram, see gcn10_cuda_last_histograms), "aggregate" (0 or 2 ..
 * GCN10_MAX_AGGREGATE, default 0: the compressed-tile calls also deliver every selected plane's f x f mean raster, see
 * gcn10_cuda_block_deflate), "cog" (0 / 1, default 0: the whole-block compressed-tile calls deliver the overview levels
 * first, smallest first, and with "ordered" frame every tile for a Cloud Optimized GeoTIFF, see gcn10_cuda_block_deflate;
 * _block_deflate_rows refuses it), "inflate_probe" (measurement aid of tools/inflate_bench.py: 1 / 2 switch parts of the inflate
 * kernel's writer off; results are then invalid). */
int gcn10_cuda_set_option(gcn10_ctx *ctx, const char *key, long value);

/* Measures this GPU's host link with page-locked memory: gbs[0] = host->device and gbs[1] = device->host copy
 * bandwidth (cudaMemcpyAsync of `bytes`, `reps` times, CUDA events), gbs[2] = device->host bandwidth of the kernel
 * that ships the compressed strips (coalesced 16-byte stores into mapped host memory).  Diagnostic: bench.py runs it
 * on one rank alone and on all ranks at once to record the fabric ceiling the end-to-end numbers sit under. */
int gcn10_cuda_pcie_probe(gcn10_ctx *ctx, size_t bytes, int reps, double gbs[3]);

/* Pins the calling host thread to the CPUs of the NUMA node the GPU hangs off (from
 * /sys/bus/pci/devices/<bus id>/numa_node and .../node<N>/cpulist), so that page-locked buffers
 * allocated afterwards are node-local and the staging copies do not cross the socket interconnect.
 * On an 8-GPU box this is what keeps eight concurrent H2D/D2H streams from sharing one memory
 * controller.  Returns the node number, or a negative value when the topology cannot be read (no
 * error is raised: the call is an optimisation). */
int gcn10_cuda_bind_host_thread(int device);

/* Page-locked host memory for rasters, so that the strip copies run asynchronously
 * (replaces malloc at raster.c:169 / cn.c:278 in a host program built on this library). */
void *gcn10_cuda_host_alloc(size_t bytes);
void gcn10_cuda_host_free(void *p);
int gcn10_cuda_host_register(void *p, size_t bytes);
int gcn10_cuda_host_unregister(void *p);

#ifdef __cplusplus
}
#endif
#endif /* GCN10_CUDA_H */
