/* gcn10_b200/host/host_tiff.h -- incremental GeoTIFF writer used by the block pipeline
 * (the one-shot gh_tiff_write and the reader are declared in gcn10_host.h). */
#ifndef GCN10_HOST_TIFF_H
#define GCN10_HOST_TIFF_H
#include <stddef.h>
#include <stdint.h>

#include "../../include/gcn10_cuda.h"      /* the overview rules: gcn10_overview_dim / _src / _levels */

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gh_tiffw gh_tiffw;

/* Creates path and reserves the header; tiles are appended with gh_tiffw_write_rows. */
int gh_tiffw_open(const char *path, int w, int h, const double gt[6], gh_tiffw **out, char *err, size_t errlen);
/* Georeferencing tags to write instead of the default EPSG:4326 keys (copied; GTRasterTypeGeoKey is forced to
 * PixelIsArea because the tiepoint written is a pixel corner).  Call before gh_tiffw_close. */
#include "gcn10_host.h"
int gh_tiffw_set_geokeys(gh_tiffw *tw, const gh_geokeys *gk);
/* Overview levels: the file gets gcn10_overview_levels(w, h, n) reduced-resolution images behind the full-resolution
 * one (one IFD each, NewSubfileType 1, chained from IFD0; n = 0: none).  Call after open, before the first data.
 * gh_tiffw_levels returns how many levels the file will have.  gh_tiffw_close fails (and removes the file) unless
 * every tile of every level has been written. */
int gh_tiffw_set_overviews(gh_tiffw *tw, int n);
int gh_tiffw_levels(const gh_tiffw *tw);
/* Statistics (on = 1): the file gets GDAL_NODATA "255" (tag 42113) in every IFD and, in IFD0, GDAL_METADATA (42112)
 * with the band statistics GDAL computes for that NoData value (STATISTICS_MINIMUM / MAXIMUM / MEAN / STDDEV /
 * VALID_PERCENT of sample 0), taken from the full-resolution histogram: gh_tiffw_write_rows counts the rows it
 * compresses, and tiles appended already compressed need gh_tiffw_put_histogram (which adds to the counts).  Call after
 * open, before the first data.  gh_tiffw_close fails (and removes the file) unless the histogram counts w * h pixels. */
int gh_tiffw_set_stats(gh_tiffw *tw, int on);
int gh_tiffw_put_histogram(gh_tiffw *tw, const uint64_t hist[256]);
/* NoData alone (on = 1): GDAL_NODATA "255" in every IFD and no GDAL_METADATA (what the mean rasters of option
 * "aggregate" carry).  gh_tiffw_set_stats writes the tag as well, with its statistics. */
int gh_tiffw_set_nodata(gh_tiffw *tw, int on);
/* Cloud Optimized GeoTIFF layout (on = 1), the order GDAL's COG driver writes and its validator checks: GDAL's ghost
 * area at offset 8 (LAYOUT=IFDS_BEFORE_DATA, BLOCK_ORDER=ROW_MAJOR, BLOCK_LEADER=SIZE_AS_UINT4,
 * BLOCK_TRAILER=LAST_4_BYTES_REPEATED), IFD0 and the level IFDs (largest to smallest) and every table and tag value they
 * point to before the first tile; then the tiles of the smallest level first and the full resolution last, each tile
 * framed by its byte count (uint32 LE) before it and its last 4 bytes after it.  Call after gh_tiffw_set_overviews,
 * _set_stats, _set_nodata and _set_geokeys (which refuse afterwards) and before the first tile: the header region is
 * reserved here, with a GDAL_METADATA slot for the longest statistics text, and filled in by gh_tiffw_close.  The tiles
 * must then come level by level in that order (levels nlev .. 1, then 0), each level in tile-row order: anything else
 * fails the file, which close removes.  gh_tiffw_write_rows refuses a COG (its levels would trail the full resolution);
 * gh_tiffw_put_tile_row(s) / _put_level_tile_rows frame the tiles they are given, gh_tiffw_put_framed_tile_rows takes
 * tiles framed already. */
int gh_tiffw_set_cog(gh_tiffw *tw, int on);
/* Appends rows [y0, y0+nrows): y0 must continue where the previous call stopped and be a multiple
 * of 256; nrows must be a multiple of 256 except for the last band of the raster.  With overviews, the levels are
 * sampled from the same rows (gcn10_overview_src) and compressed here too, a level's tile row as soon as it is full. */
int gh_tiffw_write_rows(gh_tiffw *tw, const uint8_t *data, size_t pitch, int y0, int nrows, int threads);
/* Appends tiles that are already compressed (complete zlib streams of 256 x 256 bytes, e.g. from
 * gcn10_cuda_block_deflate): tile row `tile_row` must be the next one not yet written; sizes / offsets
 * address `blob` for the tiles_x tiles of that row. */
int gh_tiffw_put_tile_row(gh_tiffw *tw, int tile_row, const uint8_t *blob, const uint64_t *offsets,
                          const uint32_t *sizes);
/* Several consecutive tile rows at once ([nrows][tiles_x] offsets / sizes).  When the tiles lie in `blob` in table
 * order with at most alignment gaps between them (gcn10_cuda_set_option "ordered") they are written with one write. */
int gh_tiffw_put_tile_rows(gh_tiffw *tw, int tile_row0, int nrows, const uint8_t *blob, const uint64_t *offsets,
                           const uint32_t *sizes);
/* The same for the tile grid of overview level `level` (0 = the full-resolution image, as gh_tiffw_put_tile_rows):
 * its tile rows too must come in order. */
int gh_tiffw_put_level_tile_rows(gh_tiffw *tw, int level, int tile_row0, int nrows, const uint8_t *blob,
                                 const uint64_t *offsets, const uint32_t *sizes);
/* COG only: tile rows whose tiles already carry their leader and trailer in blob (gcn10_tile_strip.framed: the 4 bytes
 * before blob + offsets[i] hold sizes[i], the 4 after the stream repeat its last 4), in table order with at most
 * alignment padding between them: the share from the first leader to the last trailer is written with one write.  A
 * tile whose framing is wrong fails the file. */
int gh_tiffw_put_framed_tile_rows(gh_tiffw *tw, int level, int tile_row0, int nrows, const uint8_t *blob,
                                  const uint64_t *offsets, const uint32_t *sizes);
/* Runs fn(arg, 0..n-1) on up to `threads` threads (the calling thread included). */
void gh_parallel_for(int n, int threads, void (*fn)(void *arg, int index), void *arg);
/* Writes the tile tables, georeferencing and IFD; 0 ok. */
int gh_tiffw_close(gh_tiffw *tw);
void gh_tiffw_abort(gh_tiffw *tw);

#ifdef __cplusplus
}
#endif
#endif
