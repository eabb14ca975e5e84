/* gcn10_b200/host/host_pipeline.c -- the per-block pipeline and the per-GPU block queue.
 *
 * gh_process_block() is this program's process_block() (/root/reference/src/cn.c:134-384): same
 * inputs (block id -> bbox -> two raster windows), same 18 outputs with the same names, same log
 * lines and the same two-tier error convention (recoverable: log ERROR and skip the block; fatal:
 * exit(1) where the reference calls MPI_Abort).  What changes is the middle.  Every GPU worker is a
 * three-stage pipeline over the blocks it claims from the shared queue:
 *
 *   loader thread   block geometry (cn.c:155-184), the two window computations (raster.c:126-162), the HSG
 *                   window, and the land cover AS IT LIES IN THE FILES: the compressed tiles of every source
 *                   GeoTIFF that touches the window (a single file, or up to four files of a VRT mosaic), read
 *                   into page-locked memory.  Runs up to two blocks ahead of the GPU; both rasters stay open
 *                   for the whole run (the reference re-opens them per block, raster.c:119,180).
 *   worker thread   gcn10_cuda_parts_prefetch(block i+1): upload + GPU inflate beside block i's strips;
 *                   gcn10_cuda_block_parts_deflate(block i): Curve Numbers and the DEFLATE tiles of
 *                   save_raster() (raster.c:204-219) on the device.
 *   sink            the compressed tiles of the 18 rasters are appended to their GeoTIFFs on the I/O threads
 *                   (files are created when the first strip arrives, i.e. after the land cover decoded cleanly,
 *                   under a temporary name that is renamed on success).
 *
 * Land cover that is not tiled DEFLATE is decoded on the host band by band (gcn10_cuda_block_deflate_rows);
 * with GCN10_HOST_DEFLATE=1 the raw planes come back instead and a zlib thread pool encodes them.
 *
 * gh_run_blocks() replaces the MPI round-robin of main.c:171: one worker and one gcn10_ctx per GPU, block ids
 * popped from a shared atomic counter; the join of the workers is the barrier (main.c:187).  No data moves
 * between workers, exactly as no data moves between ranks.
 */
#define _GNU_SOURCE
#include "gcn10_host.h"
#include "host_tiff.h"
#include "../../include/gcn10_cuda.h"

#include <errno.h>
#include <limits.h>
#include <pthread.h>
#include <stdatomic.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>

enum { BAND_ROWS = 2048, BAND_STRIP_ROWS = 512, NPLANES = GCN10_NPLANES, MAX_PARTS = 9, LOAD_SLOTS = 3 };

static const char *const k_conds[2] = { "drained", "undrained" };      /* cn.c:145 */
static const char *const k_hcs[3] = { "p", "f", "g" };                 /* cn.c:146 */
static const char *const k_arcs[3] = { "i", "ii", "iii" };             /* cn.c:147 */

typedef struct {
    uint8_t *esa;                   /* pinned: BAND_ROWS x pitch */
    uint8_t *planes[NPLANES];       /* pinned: BAND_ROWS x pitch each */
    int y0, rows;
    int state;                      /* 0 free, 1 filled (waiting for its consumer), -1 read failed */
} band_buf;

/* one claimed block on its way to the GPU: what the loader thread prepares */
typedef struct {
    int state;                      /* 0 free, 1 loading, 2 ready, 3 end of queue */
    int block_id;
    int failed;                     /* 1: block not found / esa load failed, 2: hysogs load failed (already logged) */
    gh_window we, wh;
    uint8_t *hsg;
    size_t hsg_cap;
    int gpu_inflate;                /* the land cover is in `parts` as compressed tiles */
    int nparts;
    gcn10_tile_part parts[MAX_PARTS];
    uint8_t *blob;                  /* pinned: the compressed tiles of all parts */
    size_t blob_cap;
    uint64_t *tile_off;
    uint32_t *tile_size;
    size_t tile_cap;
    int prefetched;                 /* gcn10_cuda_parts_prefetch has been issued for it */
    double t_read;
} block_input;

typedef struct worker {
    int index;                      /* worker number: the "rank" of the log lines */
    int device;                     /* its GPU */
    int n_gpus;                     /* GPUs this run uses */
    const gh_run_options *opt;
    int io_threads;                 /* this worker's share of the I/O threads */
    gh_blocks *blocks;
    const int (*tables)[256][5];
    const int *ids;
    int n_ids;
    atomic_int *next;               /* shared queue head */
    atomic_int *done;               /* blocks that produced all 18 rasters */
    gh_log *log;                    /* rank_<index>.log */
    gh_log *log0;                   /* worker 0's log: progress lines go there (log.c:199-207) */
    gcn10_ctx *ctx;
    /* the two rasters, opened once (lazily) and shared by the loader and the band readers under rmu */
    gh_raster *esa_r, *hsg_r;
    pthread_mutex_t rmu;
    /* loader -> worker ring */
    block_input in[LOAD_SLOTS];
    pthread_mutex_t lmu;
    pthread_cond_t lcv;
    size_t pitch_cap;
    int have_planes;
    band_buf bands[2];
    uint8_t *whole;                 /* --cog, land cover decoded on the host: the whole window, pinned */
    size_t whole_cap;
    /* encoder hand-off */
    pthread_mutex_t mu;
    pthread_cond_t cv;
    gh_tiffw *writers[NPLANES];
    int writers_open;
    char paths[NPLANES][PATH_MAX];
    /* --aggregate: the mean rasters' files, opened and closed with the 18 outputs, and (host-deflate path) the host
     * aggregation of each plane */
    gh_tiffw *agg_writers[NPLANES];
    gh_aggregate *aggs[NPLANES];
    char agg_paths[NPLANES][PATH_MAX];
    int out_w, out_h;
    double out_gt[6];
    int cur_block;
    size_t pitch;
    atomic_int encode_failed;       /* set by I/O pool threads, read by the worker */
    int encoder_quit;
} worker;

static double now_s(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

static void fatal(worker *wk, const char *msg)
{
    /* the reference's MPI_Abort(MPI_COMM_WORLD, 1) tier */
    gh_log_message(wk->log, "ERROR", msg, 1);
    exit(1);
}

static int ensure_bands(worker *wk, size_t pitch, int need_planes)
{
    if (wk->pitch_cap >= pitch && (!need_planes || wk->have_planes))
        return 0;
    for (int b = 0; b < 2; b++) {
        gcn10_cuda_host_free(wk->bands[b].esa);
        wk->bands[b].esa = gcn10_cuda_host_alloc(pitch * BAND_ROWS);
        for (int k = 0; k < NPLANES; k++) {
            gcn10_cuda_host_free(wk->bands[b].planes[k]);
            wk->bands[b].planes[k] = need_planes ? gcn10_cuda_host_alloc(pitch * BAND_ROWS) : NULL;
            if (need_planes && !wk->bands[b].planes[k])
                return -1;
        }
        if (!wk->bands[b].esa)
            return -1;
        wk->bands[b].state = 0;
    }
    wk->pitch_cap = pitch;
    wk->have_planes = need_planes;
    return 0;
}

/* cn.c:293-360: "<outdir>/cn_rasters_<cond>/cn_<hc>_<arc>_<id>.tif", or "..._<id>_.tif" when the file exists and
 * overwrite is off; the f x f mean rasters (agg = f) go to "cn_rasters_<cond>_agg<f>/" by the same rule */
static void output_path(const worker *wk, int cond, int hi, int ai, int block_id, int agg, char *path, size_t n)
{
    const char *root = (wk->opt->out_root && *wk->opt->out_root) ? wk->opt->out_root : ".";
    char sfx[32] = "";
    if (agg)
        snprintf(sfx, sizeof sfx, "_agg%d", agg);
    snprintf(path, n, "%s/cn_rasters_%s%s/cn_%s_%s_%d.tif", root, k_conds[cond], sfx, k_hcs[hi], k_arcs[ai], block_id);
    if (!wk->opt->overwrite) {
        FILE *f = fopen(path, "r");
        if (f) {
            fclose(f);
            snprintf(path, n, "%s/cn_rasters_%s%s/cn_%s_%s_%d_.tif", root, k_conds[cond], sfx, k_hcs[hi], k_arcs[ai],
                     block_id);
        }
    }
}

/* --aggregate: drop the mean rasters' files of a block that failed (or that never got its outputs) */
static void abort_agg_writers(worker *wk)
{
    for (int k = 0; k < NPLANES; k++) {
        if (wk->agg_writers[k])
            gh_tiffw_abort(wk->agg_writers[k]);
        wk->agg_writers[k] = NULL;
        gh_aggregate_free(wk->aggs[k]);
        wk->aggs[k] = NULL;
    }
}

/* --aggregate: the 18 mean rasters of the block, w / f x h / f with the scaled geotransform, the land cover's GeoKeys and
 * NoData 255 (a mean grid without it would get 255 averaged in by the next resampling).  0 ok. */
static int open_agg_writers(worker *wk)
{
    const int f = wk->opt->aggregate;
    char err[GH_ERRLEN] = "";
    double gt[6];
    gcn10_aggregate_gt(wk->out_gt, f, gt);
    for (int k = 0; k < NPLANES; k++) {
        if (gh_tiffw_open(wk->agg_paths[k], gcn10_aggregate_dim(wk->out_w, f), gcn10_aggregate_dim(wk->out_h, f), gt,
                          &wk->agg_writers[k], err, sizeof err)) {
            gh_log_message(wk->log, "ERROR", err, 1);
            wk->agg_writers[k] = NULL;
            abort_agg_writers(wk);
            return -1;
        }
        gh_geokeys gk;
        pthread_mutex_lock(&wk->rmu);
        if (wk->esa_r && gh_raster_geokeys(wk->esa_r, &gk) == 0)
            gh_tiffw_set_geokeys(wk->agg_writers[k], &gk);
        pthread_mutex_unlock(&wk->rmu);
        wk->aggs[k] = gh_aggregate_new(wk->out_w, wk->out_h, f);
        if (gh_tiffw_set_nodata(wk->agg_writers[k], 1) || (wk->opt->cog && gh_tiffw_set_cog(wk->agg_writers[k], 1)) ||
            !wk->aggs[k]) {
            snprintf(err, sizeof err, "write error 3 on %s (aggregate)", wk->agg_paths[k]);
            gh_log_message(wk->log, "ERROR", err, 1);
            abort_agg_writers(wk);
            return -1;
        }
    }
    return 0;
}


/* The 18 output files of the current block (cn.c:293-360 names; raster.c:204-219 format), created when the first
 * rows of output exist -- that is, after the land cover has been read and decoded without error.  The reference
 * likewise returns before GDALCreate when the load fails (cn.c:188-192).  0 ok. */
static int open_writers(worker *wk)
{
    if (wk->writers_open)
        return 0;
    char err[GH_ERRLEN] = "";
    int opened = 0;
    for (int k = 0; k < NPLANES; k++) {
        if (gh_tiffw_open(wk->paths[k], wk->out_w, wk->out_h, wk->out_gt, &wk->writers[k], err, sizeof err)) {
            gh_log_message(wk->log, "ERROR", err, 1);                               /* raster.c:220-223 */
            break;
        }
        /* the land cover's projection goes into every output (raster.c:164-165, 212-214) */
        gh_geokeys gk;
        pthread_mutex_lock(&wk->rmu);
        if (wk->esa_r && gh_raster_geokeys(wk->esa_r, &gk) == 0)
            gh_tiffw_set_geokeys(wk->writers[k], &gk);
        pthread_mutex_unlock(&wk->rmu);
        opened++;
        if (gh_tiffw_set_overviews(wk->writers[k], wk->opt->overviews) || gh_tiffw_set_stats(wk->writers[k], wk->opt->stats) ||
            (wk->opt->cog && gh_tiffw_set_cog(wk->writers[k], 1))) {
            snprintf(err, sizeof err, "write error 3 on %s (overviews / stats / cog)", wk->paths[k]);
            gh_log_message(wk->log, "ERROR", err, 1);
            break;
        }
    }
    const int agg_failed = opened == NPLANES && wk->opt->aggregate && open_agg_writers(wk);
    if (opened < NPLANES || agg_failed) {
        for (int k = 0; k < opened; k++) {
            gh_tiffw_abort(wk->writers[k]);
            wk->writers[k] = NULL;
        }
        return -1;
    }
    wk->writers_open = 1;
    return 0;
}

/* encoder thread: compresses and appends filled bands in order */
static void *encoder_main(void *arg)
{
    worker *wk = arg;
    int turn = 0;
    for (;;) {
        pthread_mutex_lock(&wk->mu);
        while (wk->bands[turn].state != 1 && !wk->encoder_quit)
            pthread_cond_wait(&wk->cv, &wk->mu);
        if (wk->bands[turn].state != 1 && wk->encoder_quit) {
            pthread_mutex_unlock(&wk->mu);
            return NULL;
        }
        pthread_mutex_unlock(&wk->mu);
        band_buf *bb = &wk->bands[turn];
        if (open_writers(wk))
            atomic_store(&wk->encode_failed, 1);
        for (int k = 0; k < NPLANES && !atomic_load(&wk->encode_failed); k++)
            if (gh_tiffw_write_rows(wk->writers[k], bb->planes[k], wk->pitch, bb->y0, bb->rows, wk->io_threads) ||
                (wk->opt->aggregate && gh_aggregate_write_rows(wk->aggs[k], wk->agg_writers[k], bb->planes[k], wk->pitch,
                                                               bb->y0, bb->rows, wk->io_threads)))
                atomic_store(&wk->encode_failed, 1);
        pthread_mutex_lock(&wk->mu);
        bb->state = 0;
        pthread_cond_broadcast(&wk->cv);
        pthread_mutex_unlock(&wk->mu);
        turn ^= 1;
    }
}

/* ---- GPU-deflate path: reader thread -> gcn10_cuda_block_deflate_rows -> append compressed tiles ---- */

typedef struct {
    worker *wk;
    const gh_window *we;
    int w, h;
    size_t pitch;
    double t_read;
    char err[GH_ERRLEN];
} reader_job;

static int read_band(worker *wk, const gh_window *we, int y0, int rows, uint8_t *dst, size_t pitch, char *err, size_t errlen)
{
    pthread_mutex_lock(&wk->rmu);       /* the loader thread opens mosaic sources on the same handle */
    int rc = gh_raster_read_window(wk->esa_r, we->xoff, we->yoff + y0, we->xcount, rows, dst, pitch, wk->io_threads, err,
                                   errlen);
    pthread_mutex_unlock(&wk->rmu);
    return rc;
}

static void *reader_main(void *arg)
{
    reader_job *rj = arg;
    worker *wk = rj->wk;
    int turn = 0;
    for (int y0 = 0; y0 < rj->h; y0 += BAND_ROWS, turn ^= 1) {
        band_buf *bb = &wk->bands[turn];
        pthread_mutex_lock(&wk->mu);
        while (bb->state != 0 && !wk->encoder_quit)
            pthread_cond_wait(&wk->cv, &wk->mu);
        int quit = wk->encoder_quit;
        pthread_mutex_unlock(&wk->mu);
        if (quit)
            return NULL;
        int rows = rj->h - y0 < BAND_ROWS ? rj->h - y0 : BAND_ROWS;
        double t0 = now_s();
        int rc = read_band(wk, rj->we, y0, rows, bb->esa, rj->pitch, rj->err, sizeof rj->err);
        rj->t_read += now_s() - t0;
        bb->y0 = y0;
        bb->rows = rows;
        pthread_mutex_lock(&wk->mu);
        bb->state = rc ? -1 : 1;
        pthread_cond_broadcast(&wk->cv);
        pthread_mutex_unlock(&wk->mu);
        if (rc)
            return NULL;
    }
    return NULL;
}

typedef struct {
    worker *wk;
    const gcn10_tile_strip *st;
} sink_job;

/* one plane of a strip: append its tile rows to that plane's GeoTIFF (to the strip's level of it), or to its mean
 * raster's */
static void sink_plane(void *arg, int k)
{
    sink_job *j = arg;
    const gcn10_tile_strip *st = j->st;
    gh_tiffw *tw = st->aggregate ? j->wk->agg_writers[st->plane_ids[k]] : j->wk->writers[st->plane_ids[k]];
    /* the context runs with "ordered" strips: a plane's share of the strip is one contiguous piece of the blob (with
     * --cog framed on the device already, unless the strip left unordered) */
    size_t base = (size_t)k * st->n_tile_rows * (size_t)st->tiles_x;
    if ((st->framed ? gh_tiffw_put_framed_tile_rows : gh_tiffw_put_level_tile_rows)(tw, st->level, st->tile_row0, st->n_tile_rows,
                                                                                   st->blob, st->offsets + base, st->sizes + base))
        atomic_store(&j->wk->encode_failed, 1);
}

/* the 18 files are independent: their appends run on the I/O threads while the GPU works on the next strips */
static int tile_sink(void *user, const gcn10_tile_strip *st)
{
    worker *wk = user;
    if (open_writers(wk)) {
        atomic_store(&wk->encode_failed, 1);
        return 1;
    }
    sink_job j = { wk, st };
    /* one task per plane: with 16 threads two of 18 planes would wait for a second round, so from nine threads up
     * every plane gets its own helper (they mostly sit in write(2)) */
    const int nt = wk->io_threads >= 9 ? st->n_planes : (wk->io_threads > 0 ? wk->io_threads : 1);
    gh_parallel_for(st->n_planes, nt, sink_plane, &j);
    return atomic_load(&wk->encode_failed) ? 1 : 0;
}

/* option "stats" on the GPU-deflate paths: the histograms the GPU counted while it encoded the block go to the writers,
 * which turn them into the files' statistics on close (after the block's last band, or its one call).  Runs on the
 * thread that called the library, which is also the one whose tile sink opened the writers.  (The host-deflate path
 * needs none: gh_tiffw_write_rows counts the rows it compresses.) */
static void put_gpu_histograms(worker *wk)
{
    if (!wk->opt->stats || !wk->writers_open || atomic_load(&wk->encode_failed))
        return;
    uint64_t hist[NPLANES][256];
    int rc = gcn10_cuda_last_histograms(wk->ctx, hist);
    for (int k = 0; k < NPLANES && !rc; k++)
        rc = gh_tiffw_put_histogram(wk->writers[k], hist[k]);
    if (rc)
        atomic_store(&wk->encode_failed, 1);
}

/* returns 0 ok, 1 = land-cover read failed (recoverable tier) */
static int bands_gpu_deflate(worker *wk, int block_id, const gh_window *we, const uint8_t *hsg, const gh_window *wh,
                             size_t pitch, double *t_read, double *t_gpu)
{
    char msg[1024];
    const int w = we->xcount, h = we->ycount;
    reader_job rj = { wk, we, w, h, pitch, 0.0, "" };
    pthread_t rd;
    wk->encoder_quit = 0;
    wk->bands[0].state = wk->bands[1].state = 0;
    if (pthread_create(&rd, NULL, reader_main, &rj) != 0)
        fatal(wk, "cannot start the reader thread");
    /* a band is one call: cut it into several strips so that its copies and kernels overlap */
    gcn10_cuda_set_option(wk->ctx, "strip_rows", BAND_STRIP_ROWS);
    int turn = 0, failed = 0;
    for (int y0 = 0; y0 < h; y0 += BAND_ROWS, turn ^= 1) {
        band_buf *bb = &wk->bands[turn];
        pthread_mutex_lock(&wk->mu);
        while (bb->state == 0)
            pthread_cond_wait(&wk->cv, &wk->mu);
        int st = bb->state;
        pthread_mutex_unlock(&wk->mu);
        if (st < 0) {
            gh_log_message(wk->log, "ERROR", rj.err, 1);                            /* raster.c:182-186 */
            failed = 1;
            break;
        }
        double t1 = now_s();
        int rc = gcn10_cuda_block_deflate_rows(wk->ctx, bb->esa, w, h, bb->y0, bb->rows, pitch, we->gt, hsg, wh->xcount,
                                               wh->ycount, (size_t)wh->xcount, wh->gt, GCN10_MASK_ALL, tile_sink, wk);
        if (rc && !atomic_load(&wk->encode_failed)) {
            snprintf(msg, sizeof msg, "cuda failure on block %d: %s", block_id, gcn10_cuda_last_error());
            fatal(wk, msg);                         /* CUDA errors are the fatal tier; there is no CPU path */
        }
        *t_gpu += now_s() - t1;
        pthread_mutex_lock(&wk->mu);
        bb->state = 0;
        pthread_cond_broadcast(&wk->cv);
        pthread_mutex_unlock(&wk->mu);
        if (atomic_load(&wk->encode_failed))
            break;
    }
    gcn10_cuda_set_option(wk->ctx, "strip_rows", 2048);
    if (!failed)
        put_gpu_histograms(wk);
    pthread_mutex_lock(&wk->mu);
    wk->encoder_quit = 1;
    pthread_cond_broadcast(&wk->cv);
    pthread_mutex_unlock(&wk->mu);
    pthread_join(rd, NULL);
    *t_read += rj.t_read;
    return failed;
}

/* ---- GPU-inflate path: the land-cover window goes to the device as the DEFLATE tiles of the file(s)
 * (gcn10_cuda_block_parts_deflate): no decode on the host at all.  Returns 0 ok, 1 = tile decode failed
 * (recoverable tier, raster.c:182-186) */
static int block_gpu_tiles(worker *wk, const block_input *in, double *t_gpu)
{
    char msg[1024];
    double t1 = now_s();
    int rc = gcn10_cuda_block_parts_deflate(wk->ctx, in->parts, in->nparts, gh_raster_fill(wk->esa_r), in->we.xcount,
                                            in->we.ycount, in->we.gt, in->hsg, in->wh.xcount, in->wh.ycount,
                                            (size_t)in->wh.xcount, in->wh.gt, GCN10_MASK_ALL, tile_sink, wk);
    *t_gpu += now_s() - t1;
    if (rc == GCN10_EDATA) {
        snprintf(msg, sizeof msg, "gdalrasterio error 3 (%s)", gcn10_cuda_last_error());
        gh_log_message(wk->log, "ERROR", msg, 1);
        return 1;
    }
    if (rc && !atomic_load(&wk->encode_failed)) {
        snprintf(msg, sizeof msg, "cuda failure on block %d: %s", in->block_id, gcn10_cuda_last_error());
        fatal(wk, msg);
    }
    if (!rc)
        put_gpu_histograms(wk);
    return 0;
}

/* ---- --cog with land cover decoded on the host: a COG's levels come first, so the GPU needs the whole block before
 * its first strip -- the window is read into one page-locked buffer (about 1.3 GB for 36001 x 36001) and handed to
 * gcn10_cuda_block_deflate in one call.  Returns 0 ok, 1 = land-cover read failed (recoverable tier) */
static int block_gpu_whole(worker *wk, int block_id, const gh_window *we, const uint8_t *hsg, const gh_window *wh,
                           size_t pitch, double *t_read, double *t_gpu)
{
    char msg[1024], err[GH_ERRLEN] = "";
    const int w = we->xcount, h = we->ycount;
    if (wk->whole_cap < pitch * (size_t)h) {
        gcn10_cuda_host_free(wk->whole);
        wk->whole_cap = pitch * (size_t)h;
        wk->whole = gcn10_cuda_host_alloc(wk->whole_cap);
        if (!wk->whole) {
            wk->whole_cap = 0;
            snprintf(msg, sizeof msg, "pinned allocation failed for block %d: %s", block_id, gcn10_cuda_last_error());
            fatal(wk, msg);
        }
    }
    double t0 = now_s();
    if (read_band(wk, we, 0, h, wk->whole, pitch, err, sizeof err)) {
        gh_log_message(wk->log, "ERROR", err, 1);                                   /* raster.c:182-186 */
        return 1;
    }
    double t1 = now_s();
    int rc = gcn10_cuda_block_deflate(wk->ctx, wk->whole, w, h, pitch, we->gt, hsg, wh->xcount, wh->ycount,
                                      (size_t)wh->xcount, wh->gt, GCN10_MASK_ALL, tile_sink, wk);
    if (rc && !atomic_load(&wk->encode_failed)) {
        snprintf(msg, sizeof msg, "cuda failure on block %d: %s", block_id, gcn10_cuda_last_error());
        fatal(wk, msg);                             /* CUDA errors are the fatal tier; there is no CPU path */
    }
    *t_read += t1 - t0;
    *t_gpu += now_s() - t1;
    if (!rc)
        put_gpu_histograms(wk);
    return 0;
}

/* ---- host-deflate path: raw planes back, zlib thread pool encodes band i while band i+1 is computed ---- */

static int bands_host_deflate(worker *wk, int block_id, const gh_window *we, const uint8_t *hsg, const gh_window *wh,
                              size_t pitch, double *t_read, double *t_gpu)
{
    char msg[1024], err[GH_ERRLEN] = "";
    const int w = we->xcount, h = we->ycount;
    wk->encoder_quit = 0;
    wk->bands[0].state = wk->bands[1].state = 0;
    pthread_t enc;
    if (pthread_create(&enc, NULL, encoder_main, wk) != 0)
        fatal(wk, "cannot start the encoder thread");
    gcn10_cuda_set_option(wk->ctx, "strip_rows", BAND_STRIP_ROWS);
    int turn = 0, failed = 0;
    for (int y0 = 0; y0 < h && !failed; y0 += BAND_ROWS, turn ^= 1) {
        band_buf *bb = &wk->bands[turn];
        int rows = h - y0 < BAND_ROWS ? h - y0 : BAND_ROWS;
        pthread_mutex_lock(&wk->mu);
        while (bb->state != 0)
            pthread_cond_wait(&wk->cv, &wk->mu);
        pthread_mutex_unlock(&wk->mu);
        double t0 = now_s();
        if (read_band(wk, we, y0, rows, bb->esa, pitch, err, sizeof err)) {
            gh_log_message(wk->log, "ERROR", err, 1);                               /* raster.c:182-186 */
            failed = 1;
            break;
        }
        double t1 = now_s();
        int rc = gcn10_cuda_block_rows(wk->ctx, bb->esa, w, h, y0, rows, pitch, we->gt, hsg, wh->xcount, wh->ycount,
                                       (size_t)wh->xcount, wh->gt, GCN10_MASK_ALL, bb->planes, pitch);
        if (rc) {
            snprintf(msg, sizeof msg, "cuda failure on block %d: %s", block_id, gcn10_cuda_last_error());
            fatal(wk, msg);
        }
        *t_read += t1 - t0;
        *t_gpu += now_s() - t1;
        bb->y0 = y0;
        bb->rows = rows;
        pthread_mutex_lock(&wk->mu);
        bb->state = 1;
        pthread_cond_broadcast(&wk->cv);
        pthread_mutex_unlock(&wk->mu);
    }
    gcn10_cuda_set_option(wk->ctx, "strip_rows", 2048);
    pthread_mutex_lock(&wk->mu);
    wk->encoder_quit = 1;
    pthread_cond_broadcast(&wk->cv);
    pthread_mutex_unlock(&wk->mu);
    pthread_join(enc, NULL);
    return failed;
}

/* ---- the loader: everything of process_block() that happens before the first pixel is computed ---------- */

static gh_raster *open_once(worker *wk, gh_raster **slot, const char *path)
{
    char err[GH_ERRLEN] = "";
    if (*slot)
        return *slot;
    if (gh_raster_open(path, slot, err, sizeof err)) {
        gh_log_message(wk->log, "ERROR", err, 1);                                   /* raster.c:121 */
        *slot = NULL;
    }
    else if (strcmp(gh_raster_backend(*slot), "gdal") == 0) {
        char msg[1024];
        snprintf(msg, sizeof msg, "%s opened with gdal: windows are decoded on the host", path);
        gh_log_message(wk->log, "INFO", msg, 0);
    }
    return *slot;
}

/* cn.c:155-203: bbox, land-cover window (+ its compressed tiles when the files allow it), soil window */
static void load_block(worker *wk, block_input *in, int block_id)
{
    char msg[1024], err[GH_ERRLEN] = "";
    double bbox[4], t[6];
    int rw, rh;
    in->block_id = block_id;
    in->failed = 0;
    in->gpu_inflate = 0;
    in->nparts = 0;
    in->prefetched = 0;
    in->t_read = 0;
    if (gh_blocks_bbox(wk->blocks, block_id, bbox)) {
        snprintf(msg, sizeof msg, "block %d not found", block_id);                  /* cn.c:173 */
        gh_log_message(wk->log, "ERROR", msg, 1);
        in->failed = 3;
        return;
    }
    pthread_mutex_lock(&wk->rmu);
    /* land cover window (cn.c:187 -> raster.c:106-189) */
    if (!open_once(wk, &wk->esa_r, wk->opt->cfg.esa_data_path)) {
        in->failed = 1;
        goto out;
    }
    gh_raster_size(wk->esa_r, &rw, &rh);
    gh_raster_geotransform(wk->esa_r, t);
    if (gh_raster_window(rw, rh, t, bbox, &in->we)) {
        snprintf(msg, sizeof msg, "invalid raster bounds for %s", wk->opt->cfg.esa_data_path);   /* raster.c:143 */
        gh_log_message(wk->log, "ERROR", msg, 1);
        in->failed = 1;
        goto out;
    }
    /* soil window (cn.c:195-196) */
    if (!open_once(wk, &wk->hsg_r, wk->opt->cfg.hysogs_data_path)) {
        in->failed = 2;
        goto out;
    }
    gh_raster_size(wk->hsg_r, &rw, &rh);
    gh_raster_geotransform(wk->hsg_r, t);
    if (gh_raster_window(rw, rh, t, bbox, &in->wh)) {
        snprintf(msg, sizeof msg, "invalid raster bounds for %s", wk->opt->cfg.hysogs_data_path);
        gh_log_message(wk->log, "ERROR", msg, 1);
        in->failed = 2;
        goto out;
    }
    const size_t hsg_bytes = (size_t)in->wh.xcount * (size_t)in->wh.ycount;
    if (in->hsg_cap < hsg_bytes) {
        free(in->hsg);
        in->hsg = malloc(hsg_bytes);
        in->hsg_cap = in->hsg ? hsg_bytes : 0;
        if (!in->hsg)
            fatal(wk, "out of memory for raster");                                  /* raster.c:171 */
    }
    double t0 = now_s();
    if (gh_raster_read_window(wk->hsg_r, in->wh.xoff, in->wh.yoff, in->wh.xcount, in->wh.ycount, in->hsg,
                              (size_t)in->wh.xcount, wk->io_threads, err, sizeof err)) {
        gh_log_message(wk->log, "ERROR", err, 1);
        in->failed = 2;
        goto out;
    }

    /* a tiled DEFLATE or LZW land-cover file without predictor (what GDAL writes for COMPRESS=DEFLATE / LZW TILED=YES;
     * the ESA WorldCover files are DEFLATE) is handed to the GPU compressed; anything else is decoded later, band by band */
    const char *hd = getenv("GCN10_HOST_DEFLATE"), *hi = getenv("GCN10_HOST_INFLATE");
    const int host_side = (hd && *hd && *hd != '0') || (hi && *hi && *hi != '0');
    gh_raster_part rp[MAX_PARTS];
    int np = 0;
    int prc = host_side ? 1 : gh_raster_window_parts(wk->esa_r, in->we.xoff, in->we.yoff, in->we.xcount, in->we.ycount, rp,
                                                     MAX_PARTS, &np, err, sizeof err);
    if (prc < 0) {
        gh_log_message(wk->log, "ERROR", err, 1);
        in->failed = 1;
        goto out;
    }
    if (prc == 0) {
        size_t ntiles = 0, bytes = 0;
        for (int k = 0; k < np; k++) {
            ntiles += (size_t)rp[k].plan.tiles_x * (size_t)rp[k].plan.tiles_y;
            bytes += (rp[k].plan.blob_bytes + 15) & ~(size_t)15;
        }
        if (in->blob_cap < bytes + 16) {
            gcn10_cuda_host_free(in->blob);
            in->blob_cap = bytes + bytes / 4 + (1u << 20);
            in->blob = gcn10_cuda_host_alloc(in->blob_cap);
            if (!in->blob) {
                in->blob_cap = 0;
                snprintf(msg, sizeof msg, "pinned allocation failed for block %d: %s", block_id, gcn10_cuda_last_error());
                fatal(wk, msg);
            }
        }
        if (in->tile_cap < ntiles) {
            free(in->tile_off);
            free(in->tile_size);
            in->tile_off = malloc(ntiles * sizeof *in->tile_off);
            in->tile_size = malloc(ntiles * sizeof *in->tile_size);
            if (!in->tile_off || !in->tile_size)
                fatal(wk, "out of memory for raster");
            in->tile_cap = ntiles;
        }
        size_t t_at = 0, b_at = 0;
        for (int k = 0; k < np; k++) {
            if (gh_tiff_window_tiles_read(rp[k].ds, &rp[k].plan, in->blob + b_at, in->tile_off + t_at, in->tile_size + t_at,
                                          wk->io_threads, err, sizeof err)) {
                gh_log_message(wk->log, "ERROR", err, 1);
                in->failed = 1;
                goto out;
            }
            gcn10_tile_part *cp = &in->parts[k];
            cp->tiles.tile_w = rp[k].plan.tile_w;
            cp->tiles.tile_h = rp[k].plan.tile_h;
            cp->tiles.tiles_x = rp[k].plan.tiles_x;
            cp->tiles.tiles_y = rp[k].plan.tiles_y;
            cp->tiles.x_off = rp[k].plan.x_in;
            cp->tiles.y_off = rp[k].plan.y_in;
            cp->tiles.blob = in->blob + b_at;
            cp->tiles.blob_bytes = rp[k].plan.blob_bytes;
            cp->tiles.offsets = in->tile_off + t_at;
            cp->tiles.sizes = in->tile_size + t_at;
            cp->tiles.compression = rp[k].plan.compression;
            cp->dst_x = rp[k].dst_x;
            cp->dst_y = rp[k].dst_y;
            cp->w = rp[k].w;
            cp->h = rp[k].h;
            t_at += (size_t)rp[k].plan.tiles_x * (size_t)rp[k].plan.tiles_y;
            b_at += (rp[k].plan.blob_bytes + 15) & ~(size_t)15;
        }
        in->nparts = np;
        in->gpu_inflate = np > 0;
    }
    in->t_read = now_s() - t0;
out:
    pthread_mutex_unlock(&wk->rmu);
}

static void *loader_main(void *arg)
{
    worker *wk = arg;
    for (int k = 0;; k++) {
        block_input *in = &wk->in[k % LOAD_SLOTS];
        pthread_mutex_lock(&wk->lmu);
        while (in->state != 0)
            pthread_cond_wait(&wk->lcv, &wk->lmu);
        in->state = 1;
        pthread_mutex_unlock(&wk->lmu);
        int i = atomic_fetch_add(wk->next, 1);                  /* replaces i = rank; i += size (main.c:171) */
        int last = i >= wk->n_ids;
        if (!last) {
            char msg[64];
            snprintf(msg, sizeof msg, "processing block %d", wk->ids[i]);          /* main.c:172-173 */
            gh_log_message(wk->log, "INFO", msg, 1);
            load_block(wk, in, wk->ids[i]);
        }
        pthread_mutex_lock(&wk->lmu);
        in->state = last ? 3 : 2;
        pthread_cond_broadcast(&wk->lcv);
        pthread_mutex_unlock(&wk->lmu);
        if (last)
            return NULL;
    }
}

/* cn.c:208-384 for a loaded block */
static int gh_process_block(worker *wk, block_input *in, int total_blocks, double t_start)
{
    char msg[8192];
    const int block_id = in->block_id;
    if (in->failed) {
        if (in->failed != 3) {
            snprintf(msg, sizeof msg, "%s load failed for block %d", in->failed == 2 ? "hysogs" : "esa", block_id);
            gh_log_message(wk->log, "ERROR", msg, 1);                               /* cn.c:189,198-199 */
        }
        return -1;
    }
    const gh_window *we = &in->we, *wh = &in->wh;
    const int w = we->xcount, h = we->ycount;
    const size_t pitch = ((size_t)w + 255) / 256 * 256;
    const char *hd = getenv("GCN10_HOST_DEFLATE");
    const int host_deflate = hd && *hd && *hd != '0';
    if (!in->gpu_inflate && !wk->opt->cog && ensure_bands(wk, pitch, host_deflate)) {
        snprintf(msg, sizeof msg, "pinned allocation failed for block %d: %s", block_id, gcn10_cuda_last_error());
        fatal(wk, msg);
    }
    wk->pitch = pitch;

    /* output directories and file names (cn.c:236-256, 293-360); the files themselves appear with the first rows */
    const char *root = (wk->opt->out_root && *wk->opt->out_root) ? wk->opt->out_root : ".";
    if (mkdir(root, 0755) != 0 && errno != EEXIST) {            /* --outdir may name a directory that does not exist yet */
        snprintf(msg, sizeof msg, "failed to create output directory %s", root);
        fatal(wk, msg);
    }
    for (int c = 0; c < 2; c++) {
        for (int a = 0; a < (wk->opt->aggregate ? 2 : 1); a++) {
            char outdir[PATH_MAX];
            if (a)
                snprintf(outdir, sizeof outdir, "%s/cn_rasters_%s_agg%d", root, k_conds[c], wk->opt->aggregate);
            else
                snprintf(outdir, sizeof outdir, "%s/cn_rasters_%s", root, k_conds[c]);
            if (mkdir(outdir, 0755) != 0 && errno != EEXIST) {
                snprintf(msg, sizeof msg, "failed to create output directory %s", outdir);   /* cn.c:250 */
                fatal(wk, msg);
            }
        }
    }
    for (int k = 0; k < NPLANES; k++) {
        output_path(wk, k / 9, (k % 9) / 3, k % 3, block_id, 0, wk->paths[k], sizeof wk->paths[k]);
        if (wk->opt->aggregate)
            output_path(wk, k / 9, (k % 9) / 3, k % 3, block_id, wk->opt->aggregate, wk->agg_paths[k],
                        sizeof wk->agg_paths[k]);
    }
    wk->writers_open = 0;
    wk->out_w = w;
    wk->out_h = h;
    memcpy(wk->out_gt, we->gt, sizeof wk->out_gt);
    wk->cur_block = block_id;

    atomic_store(&wk->encode_failed, 0);
    double t_read = in->t_read, t_gpu = 0;
    int failed = in->gpu_inflate ? block_gpu_tiles(wk, in, &t_gpu)
                 : host_deflate ? bands_host_deflate(wk, block_id, we, in->hsg, wh, pitch, &t_read, &t_gpu)
                 : wk->opt->cog ? block_gpu_whole(wk, block_id, we, in->hsg, wh, pitch, &t_read, &t_gpu)
                                : bands_gpu_deflate(wk, block_id, we, in->hsg, wh, pitch, &t_read, &t_gpu);

    if (failed || !wk->writers_open) {
        if (wk->writers_open)
            for (int k = 0; k < NPLANES; k++)
                gh_tiffw_abort(wk->writers[k]);
        wk->writers_open = 0;
        abort_agg_writers(wk);
        if (failed) {
            snprintf(msg, sizeof msg, "esa load failed for block %d", block_id);    /* cn.c:189 */
            gh_log_message(wk->log, "ERROR", msg, 1);
        }
        return -1;
    }
    int ok = 1;
    for (int k = 0; k < NPLANES; k++) {
        if (gh_tiffw_close(wk->writers[k]) || atomic_load(&wk->encode_failed)) {
            snprintf(msg, sizeof msg, "write error 3 on %s", wk->paths[k]);         /* raster.c:221 */
            gh_log_message(wk->log, "ERROR", msg, 1);
            ok = 0;
        }
        /* the reference logs each raster and reports it to rank 0 whether or not the write worked
         * (cn.c:363-373) */
        snprintf(msg, sizeof msg, "completed condition for %d: %s/%s/%s", block_id, k_conds[k / 9],
                 k_hcs[(k % 9) / 3], k_arcs[k % 3]);                                /* cn.c:366-369 */
        gh_log_message(wk->log, "INFO", msg, 0);
        snprintf(msg, sizeof msg, "progress: completed block %d / total %d", block_id, total_blocks);
        gh_log_message(wk->log0, "INFO", msg, 0);                                   /* log.c:199-207 */
    }
    /* the mean rasters: complete only if the block is (a failed block leaves none of them behind) */
    for (int k = 0; k < NPLANES && wk->opt->aggregate; k++) {
        if (ok && !atomic_load(&wk->encode_failed)) {
            if (gh_tiffw_close(wk->agg_writers[k])) {
                snprintf(msg, sizeof msg, "write error 3 on %s", wk->agg_paths[k]);
                gh_log_message(wk->log, "ERROR", msg, 1);
                ok = 0;
            }
        }
        else {
            gh_tiffw_abort(wk->agg_writers[k]);
        }
        wk->agg_writers[k] = NULL;
    }
    abort_agg_writers(wk);                      /* (frees the host aggregation; no writer is left to abort) */
    wk->writers_open = 0;
    double dt = now_s() - t_start;
    int lzw = 0;
    for (int k = 0; in->gpu_inflate && k < in->nparts; k++)
        lzw |= in->parts[k].tiles.compression == 5;
    const char *where = !in->gpu_inflate ? ""
                        : lzw ? (in->nparts > 1 ? " [land cover: mosaic parts (LZW) decoded on the gpu]"
                                                : " [land cover: LZW tiles decoded on the gpu]")
                              : (in->nparts > 1 ? " [land cover: mosaic parts inflated on the gpu]"
                                                : " [land cover inflated on the gpu]");
    snprintf(msg, sizeof msg,
             "block %d: %d x %d px, 18 rasters in %.3f s (%.1f Mpx/s; read %.3f s [overlapped], gpu+copies+write %.3f s; %s deflate)%s",
             block_id, w, h, dt, (double)w * h / dt / 1e6, t_read, t_gpu, host_deflate ? "host" : "gpu", where);
    gh_log_message(wk->log, "INFO", msg, 0);
    return ok ? 0 : -1;
}

static void *worker_main(void *arg)
{
    worker *wk = arg;
    char msg[256];
    /* keep this worker (and the loader / reader / encoder threads it spawns, which inherit the mask) on the
     * NUMA node of its GPU so that the pinned buffers are node-local */
    int node = gcn10_cuda_bind_host_thread(wk->device);
    snprintf(msg, sizeof msg, "worker %d on gpu %d, numa node %d", wk->index, wk->device, node);
    gh_log_message(wk->log, "INFO", msg, 0);
    /* ordered strips: a plane's share of a strip is one write; ship kernel: from four GPUs on one host fabric its posted
     * writes beat the copy engine's size read-back + copy (measured on 8 x B200: +4..7 %), below that the copy engine wins */
    if (gcn10_cuda_create(wk->device, &wk->ctx) || gcn10_cuda_set_luts(wk->ctx, wk->tables) ||
        gcn10_cuda_set_option(wk->ctx, "ordered", 1) || gcn10_cuda_set_option(wk->ctx, "ship", wk->n_gpus >= 4) ||
        gcn10_cuda_set_option(wk->ctx, "overviews", wk->opt->overviews) || gcn10_cuda_set_option(wk->ctx, "stats", wk->opt->stats) ||
        gcn10_cuda_set_option(wk->ctx, "aggregate", wk->opt->aggregate) || gcn10_cuda_set_option(wk->ctx, "cog", wk->opt->cog)) {
        snprintf(msg, sizeof msg, "cannot initialise GPU %d: %s", wk->device, gcn10_cuda_last_error());
        fatal(wk, msg);
    }
    pthread_mutex_init(&wk->mu, NULL);
    pthread_cond_init(&wk->cv, NULL);
    pthread_mutex_init(&wk->rmu, NULL);
    pthread_mutex_init(&wk->lmu, NULL);
    pthread_cond_init(&wk->lcv, NULL);
    pthread_t loader;
    if (pthread_create(&loader, NULL, loader_main, wk) != 0)
        fatal(wk, "cannot start the loader thread");
    double t_prev = now_s();
    for (int k = 0;; k++) {
        block_input *in = &wk->in[k % LOAD_SLOTS], *nx = &wk->in[(k + 1) % LOAD_SLOTS];
        pthread_mutex_lock(&wk->lmu);
        while (in->state < 2)
            pthread_cond_wait(&wk->lcv, &wk->lmu);
        const int end = in->state == 3;
        const int next_ready = nx->state == 2;
        pthread_mutex_unlock(&wk->lmu);
        if (end)
            break;
        /* the block after this one is already in memory: its upload + inflate run beside this block's strips */
        if (next_ready && !nx->failed && nx->gpu_inflate && !nx->prefetched && in->gpu_inflate && !in->failed &&
            gcn10_cuda_parts_prefetch(wk->ctx, nx->parts, nx->nparts, gh_raster_fill(wk->esa_r), nx->we.xcount,
                                      nx->we.ycount) == GCN10_OK)
            nx->prefetched = 1;
        if (gh_process_block(wk, in, wk->n_ids, t_prev) == 0)
            atomic_fetch_add(wk->done, 1);
        t_prev = now_s();
        pthread_mutex_lock(&wk->lmu);
        in->state = 0;
        pthread_cond_broadcast(&wk->lcv);
        pthread_mutex_unlock(&wk->lmu);
    }
    pthread_join(loader, NULL);
    for (int b = 0; b < 2; b++) {
        gcn10_cuda_host_free(wk->bands[b].esa);
        for (int k = 0; k < NPLANES; k++)
            gcn10_cuda_host_free(wk->bands[b].planes[k]);
    }
    gcn10_cuda_host_free(wk->whole);
    for (int i = 0; i < LOAD_SLOTS; i++) {
        gcn10_cuda_host_free(wk->in[i].blob);
        free(wk->in[i].tile_off);
        free(wk->in[i].tile_size);
        free(wk->in[i].hsg);
    }
    gh_raster_close(wk->esa_r);
    gh_raster_close(wk->hsg_r);
    gcn10_cuda_destroy(wk->ctx);
    pthread_cond_destroy(&wk->cv);
    pthread_mutex_destroy(&wk->mu);
    pthread_mutex_destroy(&wk->rmu);
    pthread_cond_destroy(&wk->lcv);
    pthread_mutex_destroy(&wk->lmu);
    return NULL;
}

int gh_run_blocks(const gh_run_options *opt, const int *block_ids, int n_blocks)
{
    char err[GH_ERRLEN] = "", msg[1024];
    static int tables[9][256][5];

    int ngpu = gcn10_cuda_device_count();
    if (ngpu <= 0) {
        fprintf(stderr, "gcn10: no usable CUDA device (%s); there is no CPU fallback\n", gcn10_cuda_last_error());
        exit(1);
    }
    /* several workers per GPU keep more than one block in flight on it: the kernels of one block (inflate, then
     * the fused Curve Number + DEFLATE kernel) are latency bound and overlap with the other block's copies */
    const int gpus = opt->n_gpus > 0 && opt->n_gpus < ngpu ? opt->n_gpus : ngpu;
    int nworkers = gpus * (opt->workers_per_gpu > 0 ? opt->workers_per_gpu : 1);
    if (nworkers > n_blocks)
        nworkers = n_blocks > 0 ? n_blocks : 1;

    gh_log *log0 = gh_log_open(opt->cfg.log_dir, 0);
    /* lookup tables once per run (the reference re-reads the CSV 18 times per block, cn.c:261) */
    if (gh_load_lookup_tables(opt->cfg.lookup_table_path, tables, err, sizeof err)) {
        gh_log_message(log0, "ERROR", err, 1);                  /* fatal in the reference: cn.c:25,32,47 */
        exit(1);
    }
    gh_blocks *blocks = NULL;
    if (gh_blocks_open(opt->cfg.blocks_shp_path, &blocks, err, sizeof err)) {
        gh_log_message(log0, "ERROR", err, 1);
        exit(1);
    }
    snprintf(msg, sizeof msg, "processing %d blocks on %d gpu workers (%d gpus)", n_blocks, nworkers,
             gpus < nworkers ? gpus : nworkers);
    gh_log_message(log0, "INFO", msg, 1);

    /* the I/O threads are shared out between the workers */
    int io_each = (opt->io_threads > 0 ? opt->io_threads : 4) / nworkers;
    if (io_each < 1)
        io_each = 1;

    atomic_int next = 0, done = 0;
    worker *wks = calloc((size_t)nworkers, sizeof *wks);
    pthread_t *th = calloc((size_t)nworkers, sizeof *th);
    for (int i = 0; i < nworkers; i++) {
        wks[i].index = i;
        wks[i].device = i % gpus;
        wks[i].n_gpus = gpus;
        wks[i].opt = opt;
        wks[i].io_threads = io_each;
        wks[i].blocks = blocks;
        wks[i].tables = tables;
        wks[i].ids = block_ids;
        wks[i].n_ids = n_blocks;
        wks[i].next = &next;
        wks[i].done = &done;
        wks[i].log0 = log0;
        wks[i].log = i == 0 ? log0 : gh_log_open(opt->cfg.log_dir, i);
        pthread_create(&th[i], NULL, worker_main, &wks[i]);
    }
    for (int i = 0; i < nworkers; i++)
        pthread_join(th[i], NULL);              /* the barrier of main.c:187 */
    snprintf(msg, sizeof msg, "processed %d blocks on %d ranks", n_blocks, nworkers);      /* main.c:191-193 */
    gh_log_message(log0, "INFO", msg, 1);
    for (int i = nworkers - 1; i >= 0; i--)
        gh_log_close(wks[i].log);
    gh_blocks_close(blocks);
    free(wks);
    free(th);
    return atomic_load(&done);
}
