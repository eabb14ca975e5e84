/* gcn10_b200/host/gcn10_host.h -- host side of the B200 Curve Number program.
 *
 * The reference's host code is C over MPI + GDAL (/root/reference/src/{main,cn,raster,config,log}.c).
 * Neither library exists in this image, and the per-pixel work now lives in libgcn10cuda.so, so the
 * host side is rebuilt here on libc + zlib + pthreads with the same observable behaviour:
 *
 *   reference                              here
 *   ------------------------------------   -------------------------------------------------
 *   parse_config()        config.c:44-114  gh_config_parse()
 *   load_lookup_table()   cn.c:13-85       gh_load_lookup_table(), once per run instead of 18x per block
 *   read_block_list()     raster.c:23-65   gh_read_block_list()
 *   get_all_blocks()      raster.c:68-103  gh_blocks_open()/gh_blocks_id()       (own .shp/.dbf reader)
 *   OGR bbox by "ID"=n    cn.c:155-184     gh_blocks_bbox()
 *   load_raster()         raster.c:106-189 gh_raster_window() + gh_tiff_read_window() (own GeoTIFF reader)
 *   save_raster()         raster.c:192-227 gh_tiff_write()   (tiled 256x256 DEFLATE GeoTIFF, threaded zlib)
 *   log_message() etc.    log.c            gh_log_*()        (same line format, mutex instead of ranks)
 *   process_block()       cn.c:134-384     gh_process_block() -> gcn10_cuda_block()
 *   main() round-robin    main.c:171       per-GPU worker threads popping a shared block queue
 *
 * Everything here is exported from libgcn10host.so so that the CPU test-suite can exercise it
 * without a GPU; the gcn10 executable links the same objects.
 */
#ifndef GCN10_HOST_H
#define GCN10_HOST_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GH_ERRLEN 512

/* ---- lookup tables (cn.c:13-85) ------------------------------------------------------------ */

/* Reads <dir>/default_lookup_<hc>_<arc>.csv.  0 ok; -1 path too long, -2 cannot open,
 * -3 empty file (all three are fatal in the reference: cn.c:21-48). */
int gh_load_lookup_table(const char *dir, const char *hc, const char *arc, int table[256][5],
                         char *err, size_t errlen);
/* The nine tables in the reference's loop order p_i .. g_iii (cn.c:146-147,258-259). */
int gh_load_lookup_tables(const char *dir, int tables[9][256][5], char *err, size_t errlen);

/* ---- window arithmetic (raster.c:126-162) -------------------------------------------------- */

typedef struct {
    int xoff, yoff, xcount, ycount;
    double gt[6];
} gh_window;

/* bbox = {minx, miny, maxx, maxy} (cn.c:179-182).  0 ok, 1 = "invalid raster bounds". */
int gh_raster_window(int raster_w, int raster_h, const double t[6], const double bbox[4], gh_window *win);

/* ---- config file (config.c:44-114) --------------------------------------------------------- */

typedef struct {
    char *hysogs_data_path;
    char *esa_data_path;
    char *blocks_shp_path;
    char *lookup_table_path;
    char *log_dir;
} gh_config;

/* 0 ok; -1 cannot open; -2 a required key is missing.  err receives the reference's message. */
int gh_config_parse(const char *path, gh_config *cfg, char *err, size_t errlen);
void gh_config_free(gh_config *cfg);

/* ---- block ids and extents ----------------------------------------------------------------- */

/* Whitespace separated integers (raster.c:23-65).  Caller frees *ids.  0 ok, -1 cannot open. */
int gh_read_block_list(const char *path, int **ids, int *n);

typedef struct gh_blocks gh_blocks;
/* Opens <name>.shp and its .dbf; reads every record's bounding box and integer "ID" field. */
int gh_blocks_open(const char *shp_path, gh_blocks **out, char *err, size_t errlen);
int gh_blocks_count(const gh_blocks *b);
int gh_blocks_id(const gh_blocks *b, int index);
/* bbox = {minx, miny, maxx, maxy} of the first record whose ID equals id; 0 ok, 1 not found. */
int gh_blocks_bbox(const gh_blocks *b, int id, double bbox[4]);
void gh_blocks_close(gh_blocks *b);

/* ---- GeoTIFF ------------------------------------------------------------------------------- */

typedef struct gh_tiff gh_tiff;
/* Single-band 8-bit GeoTIFF / BigTIFF, strips or tiles, compression none / DEFLATE / LZW,
 * predictor 1 or 2, north-up geotransform from ModelPixelScale+ModelTiepoint or ModelTransformation. */
int gh_tiff_open(const char *path, gh_tiff **out, char *err, size_t errlen);
int gh_tiff_size(const gh_tiff *t, int *w, int *h);
int gh_tiff_geotransform(const gh_tiff *t, double gt[6]);
/* The file's GeoTIFF georeferencing tags (34735 GeoKeyDirectory, 34736 GeoDoubleParams, 34737 GeoAsciiParams) as they
 * lie in it; the pointers stay valid while the dataset is open.  0 ok, 1 = the file has none.  The block pipeline
 * hands them to its outputs, as the reference copies the source dataset's projection into every raster it writes
 * (raster.c:164-165, 212-214).  A source tagged RasterPixelIsPoint gets GDAL's half-pixel shift in gh_tiff_geotransform. */
typedef struct {
    const uint16_t *keys;
    size_t n_keys;
    const double *doubles;
    size_t n_doubles;
    const char *ascii;
    size_t n_ascii;
} gh_geokeys;
int gh_tiff_geokeys(const gh_tiff *t, gh_geokeys *out);
/* Reads a pixel window into dst (row pitch in bytes); threads > 1 decodes tiles in parallel. */
int gh_tiff_read_window(gh_tiff *t, int xoff, int yoff, int xcount, int ycount, uint8_t *dst, size_t pitch,
                        int threads, char *err, size_t errlen);
/* The compressed tiles of a pixel window, as they lie in the file, for gcn10_cuda_block_tiles_deflate (GPU-side
 * decode).  gh_tiff_window_tiles_plan returns 0 and fills the plan when the dataset can be handed over that
 * way (tiled, DEFLATE or LZW, no predictor), 1 when it cannot (the caller then decodes on the host with
 * gh_tiff_read_window).  gh_tiff_window_tiles_read copies the tiles' bytes into blob (plan->blob_bytes, tiles
 * adjacent in the file are read with one pread) and fills offsets / sizes [tiles_y * tiles_x] (size 0 = sparse). */
typedef struct {
    int tile_w, tile_h;
    int tx0, ty0;               /* first tile column / row of the dataset that the window touches */
    int tiles_x, tiles_y;       /* tile grid covering the window */
    int x_in, y_in;             /* window pixel (0,0) inside that grid */
    size_t blob_bytes;
    int compression;            /* the file's TIFF Compression tag (8 / 32946 DEFLATE, 5 LZW): gcn10_tile_source.compression */
} gh_tile_plan;
int gh_tiff_window_tiles_plan(const gh_tiff *t, int xoff, int yoff, int xcount, int ycount, gh_tile_plan *plan);
int gh_tiff_window_tiles_read(gh_tiff *t, const gh_tile_plan *plan, uint8_t *blob, uint64_t *offsets, uint32_t *sizes,
                              int threads, char *err, size_t errlen);
void gh_tiff_close(gh_tiff *t);

/* ---- a raster as GDALOpen() sees it: one GeoTIFF or a VRT mosaic of GeoTIFFs (host_raster.c) ---------- */

typedef struct gh_raster gh_raster;
/* path: a GeoTIFF (see gh_tiff_open) or a GDAL .vrt whose first band is a 1:1 mosaic of GeoTIFF sources
 * (<SimpleSource> / <ComplexSource> with equal SrcRect and DstRect sizes) -- the structure of the reference's
 * landcover/esa_worldcover_2021.vrt, which its shipped config names as esa_data_path (raster.c:119). */
int gh_raster_open(const char *path, gh_raster **out, char *err, size_t errlen);
int gh_raster_size(const gh_raster *r, int *w, int *h);
int gh_raster_geotransform(const gh_raster *r, double gt[6]);
int gh_raster_is_mosaic(const gh_raster *r);
int gh_raster_source_count(const gh_raster *r);
int gh_raster_have_gdal(void);                  /* 1: built with the GDAL input backend (make GDAL=1) */
const char *gh_raster_backend(const gh_raster *r);      /* "geotiff", "vrt" or "gdal" */
int gh_raster_fill(const gh_raster *r);         /* value of pixels no source covers (VRT NoDataValue, else 0) */
/* georeferencing tags of the raster (a mosaic: of its first source that is open); 0 ok, 1 = none */
int gh_raster_geokeys(const gh_raster *r, gh_geokeys *out);
/* GDALRasterIO(GF_Read) of a window (raster.c:177-179), decoded on the host. */
int gh_raster_read_window(gh_raster *r, int xoff, int yoff, int xcount, int ycount, uint8_t *dst, size_t pitch,
                          int threads, char *err, size_t errlen);
/* The window as compressed tiles, source by source, for gcn10_cuda_block_parts_deflate.  Returns 0 and fills
 * parts[0..*nparts) when every source that touches the window is a tiled DEFLATE or LZW GeoTIFF without predictor
 * (the codec may differ from source to source); 1 when
 * the window has to be decoded on the host instead (other formats, overlapping sources, more than max_parts
 * sources); -1 when a source cannot be opened (err set: the read fails like GDAL's would). */
typedef struct {
    gh_tiff *ds;                /* borrowed: stays open inside the gh_raster */
    gh_tile_plan plan;
    int dst_x, dst_y, w, h;     /* the source's rectangle inside the window */
} gh_raster_part;
int gh_raster_window_parts(gh_raster *r, int xoff, int yoff, int xcount, int ycount, gh_raster_part *parts, int max_parts,
                           int *nparts, char *err, size_t errlen);
void gh_raster_close(gh_raster *r);

/* What save_raster() produces (raster.c:204-219): 1 band Byte, TILED=YES (256x256),
 * COMPRESS=DEFLATE (zlib level 6, no predictor), geotransform + EPSG:4326 keys, no NoData tag. */
int gh_tiff_write(const char *path, const uint8_t *data, int w, int h, size_t pitch, const double gt[6],
                  int threads, char *err, size_t errlen);
/* The same raster as a Cloud Optimized GeoTIFF (gh_tiffw_set_cog) with up to `overviews` overview levels
 * (gcn10_overview_levels), sampled on the host and written smallest first, then the full resolution. */
int gh_tiff_write_cog(const char *path, const uint8_t *data, int w, int h, size_t pitch, const double gt[6], int overviews,
                      int threads, char *err, size_t errlen);

/* ---- logging (log.c) ----------------------------------------------------------------------- */

typedef struct gh_log gh_log;
/* Opens <log_dir>/rank_<worker>.log for append and writes "[ts] [rank r] logging started" (log.c:102-118). */
gh_log *gh_log_open(const char *log_dir, int worker);
/* "[ts] [LEVEL] [rank r] msg" to the file and, if also_console, to stderr (log.c:149-166). */
void gh_log_message(gh_log *lg, const char *level, const char *msg, int also_console);
void gh_log_close(gh_log *lg);

/* ---- the per-block pipeline and the run ---------------------------------------------------- */

typedef struct {
    gh_config cfg;
    int overwrite;              /* -o / --overwrite (main.c:95-97)                                 */
    int n_gpus;                 /* workers; <= 0 means every visible GPU                           */
    int io_threads;             /* DEFLATE / inflate threads per worker                            */
    int workers_per_gpu;        /* blocks in flight per GPU (each with its own context); <= 0 means 1 */
    const char *out_root;       /* directory that receives cn_rasters_<cond>/ (reference: CWD)     */
    int overviews;              /* --overviews: at most this many overview levels per output (0 = none) */
    int stats;                  /* --stats: NoData tag and band statistics in every output                   */
    int aggregate;              /* --aggregate f: also the f x f mean rasters, in cn_rasters_<cond>_agg<f>/ (0 = none) */
    int cog;                    /* --cog: every output (and mean raster) as a Cloud Optimized GeoTIFF               */
} gh_run_options;

/* Runs a list of blocks on the GPUs of this box: one worker thread (+ one gcn10_ctx) per GPU, block
 * ids popped from a shared atomic counter.  Returns the number of blocks that produced all 18 rasters. */
int gh_run_blocks(const gh_run_options *opt, const int *block_ids, int n_blocks);

#ifdef __cplusplus
}
#endif
#endif
