/* gcn10_b200/host/host_tiff.c -- minimal GeoTIFF reader / writer for the gcn10 host program.
 *
 * Stands in for the two GDAL calls on either side of the hot path, neither of which is available
 * in this image (no libgdal):
 *   load_raster()  /root/reference/src/raster.c:106-189  -> gh_tiff_open + gh_tiff_read_window
 *   save_raster()  /root/reference/src/raster.c:192-227  -> gh_tiffw_* / gh_tiff_write
 *
 * Reader: single band, 8 bit, strips or tiles, classic TIFF or BigTIFF, either byte order,
 * compression none (1), LZW (5), DEFLATE (8 / 32946), predictor 1 or 2.
 * Writer: what GDAL's GTiff driver produces for COMPRESS=DEFLATE, TILED=YES with defaults
 * (raster.c:206-207): 256 x 256 tiles, zlib level 6, no predictor, PixelIsArea, EPSG:4326 keys,
 * no NoData tag (gh_tiffw_set_stats adds one, and the band statistics GDAL would compute).  Tiles are compressed in
 * parallel (pthreads) and appended band by band, so a 36000 x 36000 plane never has to be resident in full.
 */
#define _GNU_SOURCE
#include "gcn10_host.h"
#include "host_tiff.h"

#include <errno.h>
#include <math.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <zlib.h>

static void set_err(char *err, size_t errlen, const char *fmt, ...)
{
    if (!err || !errlen)
        return;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(err, errlen, fmt, ap);
    va_end(ap);
}

/* ------------------------------------------------------------------------------- parallel for */

typedef void (*job_fn)(void *arg, int index);

/* Every calling thread (a GPU worker, its loader, its band reader) owns a small pool of helper threads that lives as
 * long as the caller: the tile sinks run a parallel-for per strip, 18 strips per block, and creating the helpers anew
 * each time cost more than the work they did.  A job is "run fn(arg, i) for i in [0, n)"; indices are handed out under
 * the pool's mutex, the caller takes part, and returns when all indices are done. */
typedef struct {
    pthread_mutex_t mu;
    pthread_cond_t work, idle;
    pthread_t *th;
    int nthreads;               /* helpers */
    job_fn fn;
    void *arg;
    int n, next, active, generation, quit;
    int limit;                  /* helpers allowed to join the current job */
} job_pool;

static pthread_key_t g_pool_key;
static pthread_once_t g_pool_once = PTHREAD_ONCE_INIT;

static void *pool_helper(void *p)
{
    job_pool *jp = p;
    int seen = 0;
    pthread_mutex_lock(&jp->mu);
    for (;;) {
        while (!jp->quit && (jp->generation == seen || jp->next >= jp->n || jp->active >= jp->limit))
            pthread_cond_wait(&jp->work, &jp->mu);
        if (jp->quit)
            break;
        seen = jp->generation;
        jp->active++;
        while (jp->next < jp->n) {
            int i = jp->next++;
            pthread_mutex_unlock(&jp->mu);
            jp->fn(jp->arg, i);
            pthread_mutex_lock(&jp->mu);
        }
        jp->active--;
        if (jp->active == 0)
            pthread_cond_signal(&jp->idle);
    }
    pthread_mutex_unlock(&jp->mu);
    return NULL;
}

static void pool_destroy(void *p)
{
    job_pool *jp = p;
    if (!jp)
        return;
    pthread_mutex_lock(&jp->mu);
    jp->quit = 1;
    pthread_cond_broadcast(&jp->work);
    pthread_mutex_unlock(&jp->mu);
    for (int t = 0; t < jp->nthreads; t++)
        pthread_join(jp->th[t], NULL);
    pthread_mutex_destroy(&jp->mu);
    pthread_cond_destroy(&jp->work);
    pthread_cond_destroy(&jp->idle);
    free(jp->th);
    free(jp);
}

static void pool_key_init(void) { pthread_key_create(&g_pool_key, pool_destroy); }

/* the calling thread's pool, grown to at least `helpers` helper threads */
static job_pool *pool_get(int helpers)
{
    pthread_once(&g_pool_once, pool_key_init);
    job_pool *jp = pthread_getspecific(g_pool_key);
    if (!jp) {
        jp = calloc(1, sizeof *jp);
        if (!jp)
            return NULL;
        pthread_mutex_init(&jp->mu, NULL);
        pthread_cond_init(&jp->work, NULL);
        pthread_cond_init(&jp->idle, NULL);
        pthread_setspecific(g_pool_key, jp);
    }
    if (jp->nthreads < helpers) {
        pthread_t *th = realloc(jp->th, sizeof(pthread_t) * (size_t)helpers);
        if (!th)
            return jp;
        jp->th = th;
        while (jp->nthreads < helpers) {
            if (pthread_create(&jp->th[jp->nthreads], NULL, pool_helper, jp) != 0)
                break;
            jp->nthreads++;
        }
    }
    return jp;
}

static void parallel_for(int n, int threads, job_fn fn, void *arg)
{
    if (threads > n)
        threads = n;
    job_pool *jp = threads > 1 ? pool_get(threads - 1) : NULL;
    if (!jp || jp->nthreads == 0) {
        for (int i = 0; i < n; i++)
            fn(arg, i);
        return;
    }
    pthread_mutex_lock(&jp->mu);
    jp->fn = fn;
    jp->arg = arg;
    jp->n = n;
    jp->next = 0;
    jp->limit = threads - 1;
    jp->generation++;
    pthread_cond_broadcast(&jp->work);
    while (jp->next < jp->n) {                 /* the caller works too */
        int i = jp->next++;
        pthread_mutex_unlock(&jp->mu);
        fn(arg, i);
        pthread_mutex_lock(&jp->mu);
    }
    while (jp->active > 0)
        pthread_cond_wait(&jp->idle, &jp->mu);
    jp->n = 0;                                  /* late wakers find nothing to do */
    pthread_mutex_unlock(&jp->mu);
}

void gh_parallel_for(int n, int threads, void (*fn)(void *arg, int index), void *arg)
{
    parallel_for(n, threads, fn, arg);
}

/* ------------------------------------------------------------------------------------- reader */

struct gh_tiff {
    int fd;
    int big, swap;
    int w, h;
    int compression, predictor;
    int tiled, tw, th;          /* tile (or strip: tw = w, th = rows per strip) geometry */
    int tiles_x, tiles_y;
    uint64_t *offsets, *counts;
    uint64_t nchunks;
    uint64_t file_size;
    int has_gt;
    double gt[6];
    /* GeoTIFF georeferencing tags as they lie in the file (34735 key directory, 34736 double params, 34737 ascii
     * params): handed to the outputs verbatim, as the reference copies the source's projection (raster.c:164-165,
     * 212-214) */
    uint16_t *geo_keys;
    size_t n_geo_keys;
    double *geo_doubles;
    size_t n_geo_doubles;
    char *geo_ascii;
    size_t n_geo_ascii;
};

static uint16_t rd16(const gh_tiff *t, const unsigned char *p)
{
    return t->swap ? (uint16_t)(p[0] << 8 | p[1]) : (uint16_t)(p[1] << 8 | p[0]);
}

static uint32_t rd32(const gh_tiff *t, const unsigned char *p)
{
    return t->swap ? ((uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3])
                   : ((uint32_t)p[3] << 24 | (uint32_t)p[2] << 16 | (uint32_t)p[1] << 8 | p[0]);
}

static uint64_t rd64(const gh_tiff *t, const unsigned char *p)
{
    uint64_t v = 0;
    if (t->swap)
        for (int i = 0; i < 8; i++) v = v << 8 | p[i];
    else
        for (int i = 7; i >= 0; i--) v = v << 8 | p[i];
    return v;
}

static int pread_all(int fd, void *buf, size_t n, uint64_t off)
{
    unsigned char *p = buf;
    while (n) {
        ssize_t r = pread(fd, p, n, (off_t)off);
        if (r <= 0)
            return -1;
        p += r;
        n -= (size_t)r;
        off += (uint64_t)r;
    }
    return 0;
}

static size_t type_size(int type)
{
    switch (type) {
    case 1: case 2: case 6: case 7: return 1;
    case 3: case 8: return 2;
    case 4: case 9: case 11: case 13: return 4;
    case 5: case 10: case 12: case 16: case 17: case 18: return 8;
    }
    return 0;
}

/* Fetches the values of one IFD entry as doubles or uint64 (whichever array is non-NULL). */
static int entry_values(gh_tiff *t, int type, uint64_t count, const unsigned char *valfield, size_t valfield_len,
                        uint64_t *u, double *d, uint64_t max)
{
    size_t ts = type_size(type);
    if (!ts || count == 0)
        return -1;
    const int is_inline = count <= valfield_len / ts;            /* decided by the stored count */
    if (count > max)
        count = max;
    /* a table cannot be longer than the file that holds it (a damaged count must not size an allocation) */
    if (!is_inline && count > t->file_size / ts)
        return -1;
    size_t bytes = ts * (size_t)count;
    unsigned char *buf = malloc(bytes);
    if (!buf)
        return -1;
    if (is_inline) {
        memcpy(buf, valfield, bytes);
    }
    else {
        uint64_t off = t->big ? rd64(t, valfield) : rd32(t, valfield);
        if (off > t->file_size || bytes > t->file_size - off || pread_all(t->fd, buf, bytes, off)) {
            free(buf);
            return -1;
        }
    }
    for (uint64_t i = 0; i < count; i++) {
        const unsigned char *p = buf + ts * i;
        uint64_t uv = 0;
        double dv = 0;
        switch (type) {
        case 1: case 2: case 7: uv = p[0]; dv = (double)uv; break;
        case 3: uv = rd16(t, p); dv = (double)uv; break;
        case 4: case 13: uv = rd32(t, p); dv = (double)uv; break;
        case 16: case 18: uv = rd64(t, p); dv = (double)uv; break;
        case 12: { uint64_t b = rd64(t, p); memcpy(&dv, &b, 8); uv = dv >= 0.0 && dv < 1.8e19 ? (uint64_t)dv : 0; break; }
        case 11: { uint32_t b = rd32(t, p); float f; memcpy(&f, &b, 4); dv = f; uv = dv >= 0.0 && dv < 1.8e19 ? (uint64_t)dv : 0; break; }
        default: free(buf); return -1;
        }
        if (u) u[i] = uv;
        if (d) d[i] = dv;
    }
    free(buf);
    return 0;
}

int gh_tiff_open(const char *path, gh_tiff **out, char *err, size_t errlen)
{
    *out = NULL;
    if (err && errlen)
        err[0] = '\0';
    gh_tiff *t = calloc(1, sizeof *t);
    if (!t)
        return -1;
    t->fd = open(path, O_RDONLY);
    unsigned char hdr[16];
    struct stat st;
    if (t->fd < 0 || fstat(t->fd, &st) || st.st_size < 8 || pread_all(t->fd, hdr, 8, 0)) {
        set_err(err, errlen, "gdal open failed: %s", path);                 /* raster.c:121 */
        goto fail;
    }
    t->file_size = (uint64_t)st.st_size;
    if (hdr[0] == 'I' && hdr[1] == 'I') t->swap = 0;
    else if (hdr[0] == 'M' && hdr[1] == 'M') t->swap = 1;
    else { set_err(err, errlen, "gdal open failed: %s (not a TIFF)", path); goto fail; }
    uint16_t magic = rd16(t, hdr + 2);
    uint64_t ifd;
    if (magic == 42) {
        ifd = rd32(t, hdr + 4);
    }
    else if (magic == 43) {
        t->big = 1;
        if (pread_all(t->fd, hdr, 16, 0)) goto fail;
        ifd = rd64(t, hdr + 8);
    }
    else { set_err(err, errlen, "gdal open failed: %s (bad TIFF magic %u)", path, magic); goto fail; }

    unsigned char nb[8];
    if (pread_all(t->fd, nb, t->big ? 8 : 2, ifd)) goto fail;
    uint64_t nent = t->big ? rd64(t, nb) : rd16(t, nb);
    size_t esz = t->big ? 20 : 12;
    if (nent == 0 || nent > 65535 || ifd > t->file_size || esz * nent > t->file_size - ifd) {
        set_err(err, errlen, "gdal open failed: %s (damaged TIFF directory)", path);
        goto fail;
    }
    unsigned char *ents = malloc(esz * (size_t)nent);
    if (!ents || pread_all(t->fd, ents, esz * (size_t)nent, ifd + (t->big ? 8 : 2))) { free(ents); goto fail; }

    int bits = 1, spp = 1, rows_per_strip = 0;
    uint64_t off_tag_count = 0;
    const unsigned char *off_ent = NULL, *cnt_ent = NULL;
    int off_type = 0, cnt_type = 0;
    double scale[3] = { 0 }, tie[6] = { 0 }, xf[16] = { 0 };
    int have_scale = 0, have_tie = 0, have_xf = 0;
    t->compression = 1;
    t->predictor = 1;
    for (uint64_t i = 0; i < nent; i++) {
        const unsigned char *e = ents + esz * i;
        int tag = rd16(t, e), type = rd16(t, e + 2);
        uint64_t count = t->big ? rd64(t, e + 4) : rd32(t, e + 4);
        const unsigned char *val = e + (t->big ? 12 : 8);
        size_t vlen = t->big ? 8 : 4;
        uint64_t u[1] = { 0 };
        switch (tag) {
        case 256: entry_values(t, type, count, val, vlen, u, NULL, 1); t->w = (int)u[0]; break;
        case 257: entry_values(t, type, count, val, vlen, u, NULL, 1); t->h = (int)u[0]; break;
        case 258: entry_values(t, type, count, val, vlen, u, NULL, 1); bits = (int)u[0]; break;
        case 259: entry_values(t, type, count, val, vlen, u, NULL, 1); t->compression = (int)u[0]; break;
        case 277: entry_values(t, type, count, val, vlen, u, NULL, 1); spp = (int)u[0]; break;
        case 278: entry_values(t, type, count, val, vlen, u, NULL, 1); rows_per_strip = (int)(u[0] > 0x7fffffff ? 0x7fffffff : u[0]); break;
        case 317: entry_values(t, type, count, val, vlen, u, NULL, 1); t->predictor = (int)u[0]; break;
        case 322: entry_values(t, type, count, val, vlen, u, NULL, 1); t->tw = (int)u[0]; t->tiled = 1; break;
        case 323: entry_values(t, type, count, val, vlen, u, NULL, 1); t->th = (int)u[0]; t->tiled = 1; break;
        case 273: case 324: off_ent = e; off_type = type; off_tag_count = count; break;
        case 279: case 325: cnt_ent = e; cnt_type = type; break;
        case 33550: have_scale = entry_values(t, type, count, val, vlen, NULL, scale, 3) == 0 && count >= 2; break;
        case 33922: have_tie = entry_values(t, type, count, val, vlen, NULL, tie, 6) == 0 && count >= 6; break;
        case 34264: have_xf = entry_values(t, type, count, val, vlen, NULL, xf, 16) == 0 && count >= 16; break;
        case 34735:
            if (type == 3 && count >= 4 && count < 4096 && !t->geo_keys) {
                uint64_t *tmp = malloc(sizeof(uint64_t) * (size_t)count);
                t->geo_keys = malloc(sizeof(uint16_t) * (size_t)count);
                if (tmp && t->geo_keys && entry_values(t, type, count, val, vlen, tmp, NULL, count) == 0) {
                    for (uint64_t k = 0; k < count; k++)
                        t->geo_keys[k] = (uint16_t)tmp[k];
                    t->n_geo_keys = (size_t)count;
                }
                free(tmp);
            }
            break;
        case 34736:
            if (type == 12 && count > 0 && count < 4096 && !t->geo_doubles) {
                t->geo_doubles = malloc(sizeof(double) * (size_t)count);
                if (t->geo_doubles && entry_values(t, type, count, val, vlen, NULL, t->geo_doubles, count) == 0)
                    t->n_geo_doubles = (size_t)count;
            }
            break;
        case 34737:
            if (type == 2 && count > 0 && count < 65536 && !t->geo_ascii) {
                uint64_t *tmp = malloc(sizeof(uint64_t) * (size_t)count);
                t->geo_ascii = malloc((size_t)count + 1);
                if (tmp && t->geo_ascii && entry_values(t, type, count, val, vlen, tmp, NULL, count) == 0) {
                    for (uint64_t k = 0; k < count; k++)
                        t->geo_ascii[k] = (char)tmp[k];
                    t->geo_ascii[count] = '\0';
                    t->n_geo_ascii = (size_t)count;
                }
                free(tmp);
            }
            break;
        default: break;
        }
    }
    if (t->w <= 0 || t->h <= 0 || bits != 8 || spp != 1 || !off_ent || !cnt_ent) {
        set_err(err, errlen, "gdal open failed: %s (need a single-band 8-bit raster; got %d bits x %d samples)",
                path, bits, spp);
        free(ents);
        goto fail;
    }
    if (t->compression != 1 && t->compression != 5 && t->compression != 8 && t->compression != 32946) {
        set_err(err, errlen, "gdal open failed: %s (unsupported TIFF compression %d)", path, t->compression);
        free(ents);
        goto fail;
    }
    if (!t->tiled) {
        t->tw = t->w;
        t->th = (rows_per_strip <= 0 || rows_per_strip > t->h) ? t->h : rows_per_strip;
    }
    /* tile geometry out of a damaged directory: no division by zero, no tile that cannot be allocated */
    if (t->tw <= 0 || t->th <= 0 || (uint64_t)t->tw * (uint64_t)t->th > (1ull << 33)) {
        set_err(err, errlen, "gdal open failed: %s (bad tile size %d x %d)", path, t->tw, t->th);
        free(ents);
        goto fail;
    }
    t->tiles_x = (int)(((int64_t)t->w + t->tw - 1) / t->tw);
    t->tiles_y = (int)(((int64_t)t->h + t->th - 1) / t->th);
    t->nchunks = (uint64_t)t->tiles_x * (uint64_t)t->tiles_y;
    if (off_tag_count < t->nchunks || t->nchunks > t->file_size) {
        set_err(err, errlen, "gdal open failed: %s (offset table shorter than the tile grid)", path);
        free(ents);
        goto fail;
    }
    t->offsets = malloc(sizeof(uint64_t) * t->nchunks);
    t->counts = malloc(sizeof(uint64_t) * t->nchunks);
    size_t vlen = t->big ? 8 : 4;
    if (!t->offsets || !t->counts ||
        entry_values(t, off_type, off_tag_count, off_ent + (t->big ? 12 : 8), vlen, t->offsets, NULL, t->nchunks) ||
        entry_values(t, cnt_type, off_tag_count, cnt_ent + (t->big ? 12 : 8), vlen, t->counts, NULL, t->nchunks)) {
        set_err(err, errlen, "gdal open failed: %s (cannot read the tile tables)", path);
        free(ents);
        goto fail;
    }
    free(ents);
    if (have_scale && have_tie) {
        /* PixelIsArea north-up: origin = tiepoint world coords minus tiepoint raster coords * scale */
        t->gt[1] = scale[0];
        t->gt[5] = -scale[1];
        t->gt[0] = tie[3] - tie[0] * scale[0];
        t->gt[3] = tie[4] + tie[1] * scale[1];
        t->has_gt = 1;
        /* GTRasterTypeGeoKey (1025) = RasterPixelIsPoint (2): the tiepoint names a pixel CENTRE; GDAL's geotransform
         * is that of the pixel's corner, half a pixel up and to the left */
        for (size_t k = 4; k + 3 < t->n_geo_keys; k += 4)
            if (t->geo_keys[k] == 1025 && t->geo_keys[k + 1] == 0 && t->geo_keys[k + 3] == 2) {
                t->gt[0] -= 0.5 * t->gt[1];
                t->gt[3] -= 0.5 * t->gt[5];
            }
    }
    else if (have_xf) {
        t->gt[0] = xf[3]; t->gt[1] = xf[0]; t->gt[2] = xf[1];
        t->gt[3] = xf[7]; t->gt[4] = xf[4]; t->gt[5] = xf[5];
        t->has_gt = 1;
    }
    else {
        t->gt[1] = 1.0;         /* GDAL's default for an ungeoreferenced raster */
        t->gt[5] = 1.0;
    }
    *out = t;
    return 0;
fail:
    if (err && !*err)
        set_err(err, errlen, "gdal open failed: %s", path);
    gh_tiff_close(t);
    return -1;
}

int gh_tiff_size(const gh_tiff *t, int *w, int *h) { *w = t->w; *h = t->h; return 0; }
int gh_tiff_geotransform(const gh_tiff *t, double gt[6]) { memcpy(gt, t->gt, sizeof t->gt); return t->has_gt ? 0 : 1; }

void gh_tiff_close(gh_tiff *t)
{
    if (!t)
        return;
    if (t->fd >= 0)
        close(t->fd);
    free(t->offsets);
    free(t->counts);
    free(t->geo_keys);
    free(t->geo_doubles);
    free(t->geo_ascii);
    free(t);
}

int gh_tiff_geokeys(const gh_tiff *t, gh_geokeys *out)
{
    memset(out, 0, sizeof *out);
    if (!t->n_geo_keys)
        return 1;
    out->keys = t->geo_keys;
    out->n_keys = t->n_geo_keys;
    out->doubles = t->geo_doubles;
    out->n_doubles = t->n_geo_doubles;
    out->ascii = t->geo_ascii;
    out->n_ascii = t->n_geo_ascii;
    return 0;
}

/* TIFF LZW: MSB-first variable width codes (9..12 bits), 256 = clear, 257 = end of information,
 * width grows one code early ("early change"). */
static int lzw_decode(const unsigned char *src, size_t n, unsigned char *dst, size_t cap)
{
    enum { CLEAR = 256, EOI = 257, FIRST = 258, MAXC = 4096 };
    uint16_t *prefix = malloc(sizeof(uint16_t) * MAXC);
    unsigned char *suffix = malloc(MAXC), *first = malloc(MAXC);
    uint16_t *length = malloc(sizeof(uint16_t) * MAXC);
    if (!prefix || !suffix || !first || !length) { free(prefix); free(suffix); free(first); free(length); return -1; }
    for (int i = 0; i < 256; i++) { prefix[i] = 0xFFFF; suffix[i] = first[i] = (unsigned char)i; length[i] = 1; }
    size_t out = 0, bitpos = 0, nbits = n * 8;
    int width = 9, next = FIRST, prev = -1, rc = 0;
    while (bitpos + (size_t)width <= nbits) {
        uint32_t code = 0;
        for (int b = 0; b < width; b++) {
            size_t bp = bitpos + (size_t)b;
            code = code << 1 | ((src[bp >> 3] >> (7 - (bp & 7))) & 1u);
        }
        bitpos += (size_t)width;
        if (code == EOI)
            break;
        if (code == CLEAR) {
            width = 9;
            next = FIRST;
            prev = -1;
            continue;
        }
        int cur = (int)code;
        if (prev < 0) {
            if (cur >= 256) { rc = -1; break; }
            if (out < cap) dst[out] = (unsigned char)cur;
            out++;
            prev = cur;
            continue;
        }
        int emit;
        if (cur < next) {
            emit = cur;
        }
        else if (cur == next) {
            emit = -1;          /* KwKwK: prev string + its own first byte */
        }
        else { rc = -1; break; }
        /* add table entry prev + first(emit string) */
        unsigned char fb = emit >= 0 ? first[emit] : first[prev];
        if (next < MAXC) {
            prefix[next] = (uint16_t)prev;
            suffix[next] = fb;
            first[next] = first[prev];
            length[next] = (uint16_t)(length[prev] + 1);
            next++;
        }
        int s = emit >= 0 ? emit : next - 1;
        size_t len = length[s];
        if (out + len <= cap) {
            size_t pos = out + len;
            int c = s;
            while (c != 0xFFFF && pos > out) {
                dst[--pos] = suffix[c];
                c = prefix[c];
            }
        }
        out += len;
        prev = cur;
        if (next + 1 >= (1 << width) && width < 12)
            width++;
    }
    free(prefix); free(suffix); free(first); free(length);
    (void)out;
    return rc;
}

typedef struct {
    gh_tiff *t;
    int xoff, yoff, xcount, ycount;
    uint8_t *dst;
    size_t pitch;
    int tx0, ty0, ntx, nty;
    int failed;
} read_job;

static void read_chunk(void *arg, int index)
{
    read_job *j = arg;
    gh_tiff *t = j->t;
    int tx = j->tx0 + index % j->ntx, ty = j->ty0 + index / j->ntx;
    uint64_t ci = (uint64_t)ty * (uint64_t)t->tiles_x + (uint64_t)tx;
    int rows = t->th, cols = t->tw;
    if (!t->tiled && (ty + 1) * t->th > t->h)
        rows = t->h - ty * t->th;           /* the last strip may be short */
    size_t raw = (size_t)rows * (size_t)cols;
    unsigned char *buf = malloc(raw ? raw : 1);
    unsigned char *comp = NULL;
    if (!buf) { j->failed = 1; return; }
    uint64_t n = t->counts[ci];
    if (n == 0) {
        memset(buf, 0, raw);                /* sparse tile: GDAL serves zeros */
    }
    else if (t->compression == 1) {
        size_t take = n < raw ? (size_t)n : raw;
        if (pread_all(t->fd, buf, take, t->offsets[ci])) j->failed = 1;
        if (take < raw) memset(buf + take, 0, raw - take);
    }
    else if (t->offsets[ci] > t->file_size || n > t->file_size - t->offsets[ci]) {
        j->failed = 1;                      /* the tile table points outside the file */
    }
    else {
        comp = malloc((size_t)n);
        if (!comp || pread_all(t->fd, comp, (size_t)n, t->offsets[ci])) {
            j->failed = 1;
        }
        else if (t->compression == 5) {
            memset(buf, 0, raw);
            if (lzw_decode(comp, (size_t)n, buf, raw)) j->failed = 1;
        }
        else {
            uLongf dl = (uLongf)raw;
            int zr = uncompress(buf, &dl, comp, (uLong)n);
            if (zr != Z_OK && zr != Z_BUF_ERROR) j->failed = 1;
            if (dl < raw) memset(buf + dl, 0, raw - dl);
        }
    }
    free(comp);
    if (t->predictor == 2) {
        for (int r = 0; r < rows; r++) {
            unsigned char *p = buf + (size_t)r * cols;
            for (int c = 1; c < cols; c++)
                p[c] = (unsigned char)(p[c] + p[c - 1]);
        }
    }
    /* copy the intersection with the window */
    int cx0 = tx * t->tw, cy0 = ty * t->th;
    int x_lo = cx0 > j->xoff ? cx0 : j->xoff, x_hi = cx0 + cols < j->xoff + j->xcount ? cx0 + cols : j->xoff + j->xcount;
    int y_lo = cy0 > j->yoff ? cy0 : j->yoff, y_hi = cy0 + rows < j->yoff + j->ycount ? cy0 + rows : j->yoff + j->ycount;
    for (int y = y_lo; y < y_hi; y++)
        memcpy(j->dst + (size_t)(y - j->yoff) * j->pitch + (size_t)(x_lo - j->xoff),
               buf + (size_t)(y - cy0) * cols + (size_t)(x_lo - cx0), (size_t)(x_hi - x_lo));
    free(buf);
}

int gh_tiff_read_window(gh_tiff *t, int xoff, int yoff, int xcount, int ycount, uint8_t *dst, size_t pitch,
                        int threads, char *err, size_t errlen)
{
    if (xoff < 0 || yoff < 0 || xcount <= 0 || ycount <= 0 || xoff + xcount > t->w || yoff + ycount > t->h ||
        pitch < (size_t)xcount) {
        set_err(err, errlen, "gdalrasterio error 3 (window %d,%d %dx%d outside %dx%d)", xoff, yoff, xcount, ycount,
                t->w, t->h);
        return -1;
    }
    read_job j = { t, xoff, yoff, xcount, ycount, dst, pitch, 0, 0, 0, 0, 0 };
    j.tx0 = xoff / t->tw;
    j.ty0 = yoff / t->th;
    j.ntx = (xoff + xcount - 1) / t->tw - j.tx0 + 1;
    j.nty = (yoff + ycount - 1) / t->th - j.ty0 + 1;
    parallel_for(j.ntx * j.nty, threads, read_chunk, &j);
    if (j.failed) {
        set_err(err, errlen, "gdalrasterio error 3 (tile decode failed)");
        return -1;
    }
    return 0;
}

/* ---- compressed tiles of a window, untouched (the GPU inflates them) */

int gh_tiff_window_tiles_plan(const gh_tiff *t, int xoff, int yoff, int xcount, int ycount, gh_tile_plan *plan)
{
    if (!t->tiled || (t->compression != 8 && t->compression != 32946 && t->compression != 5) || t->predictor != 1)
        return 1;
    if (xoff < 0 || yoff < 0 || xcount <= 0 || ycount <= 0 || xoff + xcount > t->w || yoff + ycount > t->h)
        return 1;
    plan->tile_w = t->tw;
    plan->tile_h = t->th;
    plan->tx0 = xoff / t->tw;
    plan->ty0 = yoff / t->th;
    plan->tiles_x = (xoff + xcount - 1) / t->tw - plan->tx0 + 1;
    plan->tiles_y = (yoff + ycount - 1) / t->th - plan->ty0 + 1;
    plan->x_in = xoff - plan->tx0 * t->tw;
    plan->y_in = yoff - plan->ty0 * t->th;
    size_t total = 0;
    for (int ty = 0; ty < plan->tiles_y; ty++)
        for (int tx = 0; tx < plan->tiles_x; tx++) {
            const uint64_t ci = (uint64_t)(plan->ty0 + ty) * (uint64_t)t->tiles_x + (uint64_t)(plan->tx0 + tx);
            uint64_t n = t->counts[ci];
            /* a tile the file cannot hold: leave it to the host path, whose read fails like GDAL's would */
            if (n > 0xFFFFFFFFull || t->offsets[ci] > t->file_size || n > t->file_size - t->offsets[ci])
                return 1;
            total += (size_t)n;
        }
    plan->blob_bytes = total;
    plan->compression = t->compression;
    return 0;
}

typedef struct {
    gh_tiff *t;
    const gh_tile_plan *plan;
    uint8_t *blob;
    const uint64_t *offsets;
    int failed;
} tiles_job;

/* one job = one tile row of the window: runs of tiles that are adjacent in the file become one pread */
static void read_tile_row(void *arg, int ty)
{
    tiles_job *j = arg;
    const gh_tile_plan *p = j->plan;
    const gh_tiff *t = j->t;
    int tx = 0;
    while (tx < p->tiles_x) {
        uint64_t ci = (uint64_t)(p->ty0 + ty) * (uint64_t)t->tiles_x + (uint64_t)(p->tx0 + tx);
        uint64_t start = t->offsets[ci], len = t->counts[ci];
        int run = 1;
        while (tx + run < p->tiles_x && t->counts[ci + run] > 0 && t->offsets[ci + run] == start + len) {
            len += t->counts[ci + run];
            run++;
        }
        if (len && pread_all(t->fd, j->blob + j->offsets[(size_t)ty * p->tiles_x + tx], (size_t)len, start))
            j->failed = 1;
        tx += run;
    }
}

int gh_tiff_window_tiles_read(gh_tiff *t, const gh_tile_plan *plan, uint8_t *blob, uint64_t *offsets, uint32_t *sizes,
                              int threads, char *err, size_t errlen)
{
    uint64_t pos = 0;
    for (int ty = 0; ty < plan->tiles_y; ty++)
        for (int tx = 0; tx < plan->tiles_x; tx++) {
            uint64_t n = t->counts[(uint64_t)(plan->ty0 + ty) * (uint64_t)t->tiles_x + (uint64_t)(plan->tx0 + tx)];
            offsets[(size_t)ty * plan->tiles_x + tx] = pos;
            sizes[(size_t)ty * plan->tiles_x + tx] = (uint32_t)n;
            pos += n;
        }
    tiles_job j = { t, plan, blob, offsets, 0 };
    parallel_for(plan->tiles_y, threads, read_tile_row, &j);
    if (j.failed) {
        set_err(err, errlen, "gdalrasterio error 3 (tile read failed)");
        return -1;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------- writer */

enum { TILE = 256 };

static void put16(unsigned char **p, uint16_t v) { (*p)[0] = (unsigned char)v; (*p)[1] = (unsigned char)(v >> 8); *p += 2; }
static void put32(unsigned char **p, uint32_t v) { for (int i = 0; i < 4; i++) (*p)[i] = (unsigned char)(v >> (8 * i)); *p += 4; }
static void put_f64(unsigned char **p, double d) { uint64_t v; memcpy(&v, &d, 8); for (int i = 0; i < 8; i++) (*p)[i] = (unsigned char)(v >> (8 * i)); *p += 8; }

/* the tile grid of one level of the file: level 0 = the full-resolution raster, k >= 1 = overview level k */
typedef struct {
    int w, h;
    int tiles_x, tiles_y;
    uint32_t *offsets, *counts;
    int next_tile_row;
    uint8_t *band;              /* gh_tiffw_write_rows, levels >= 1: the level's tile row being sampled, TILE x w */
} tw_grid;

struct gh_tiffw {
    FILE *fp;
    char *path, *tmp;           /* written as <path>.part, renamed on a successful close, removed otherwise */
    uint16_t *geo_keys;         /* georeferencing tags copied from the land-cover source, or NULL = EPSG:4326 */
    size_t n_geo_keys;
    double *geo_doubles;
    size_t n_geo_doubles;
    char *geo_ascii;
    size_t n_geo_ascii;
    double gt[6];
    uint64_t pos;
    int nlev;                   /* overview levels (gh_tiffw_set_overviews) */
    tw_grid g[1 + GCN10_MAX_OVERVIEWS];
    int stats;                  /* gh_tiffw_set_stats: NoData tag + GDAL_METADATA statistics from hist */
    uint64_t hist[256];         /* full-resolution pixels per value */
    int nodata;                 /* gh_tiffw_set_nodata: NoData tag without statistics */
    int cog;                    /* gh_tiffw_set_cog: Cloud Optimized GeoTIFF layout */
    int cog_level;              /* ... the level whose tiles come next (nlev .. 0) */
    uint64_t cog_data;          /* ... the first byte after the header region */
    int level;                  /* zlib level */
    int failed;
};

typedef struct {
    gh_tiffw *tw;
    const tw_grid *g;
    const uint8_t *data;        /* first row of this band */
    size_t pitch;
    int rows;                   /* rows available in the band */
    int tile_row0;
    unsigned char **comp;
    uLongf *comp_len;
    uint32_t (*hist)[256];      /* per tile: its pixels per value (NULL: not counted) */
} write_job;

static void compress_tile(void *arg, int index)
{
    write_job *j = arg;
    gh_tiffw *tw = j->tw;
    int tx = index % j->g->tiles_x, tr = index / j->g->tiles_x;
    unsigned char tile[TILE * TILE];
    int x0 = tx * TILE, y0 = tr * TILE;
    int cols = j->g->w - x0 < TILE ? j->g->w - x0 : TILE;
    int rows = j->rows - y0 < TILE ? j->rows - y0 : TILE;
    if (cols < TILE || rows < TILE)
        memset(tile, 0, sizeof tile);       /* edge tiles are padded with zeros */
    for (int r = 0; r < rows; r++)
        memcpy(tile + r * TILE, j->data + (size_t)(y0 + r) * j->pitch + x0, (size_t)cols);
    if (j->hist) {
        uint32_t *hc = j->hist[index];
        memset(hc, 0, sizeof j->hist[index]);
        for (int r = 0; r < rows; r++)
            for (int x = 0; x < cols; x++)
                hc[tile[r * TILE + x]]++;
    }
    uLongf cap = compressBound(sizeof tile);
    unsigned char *out = malloc(cap);
    if (!out || compress2(out, &cap, tile, sizeof tile, tw->level) != Z_OK) {
        free(out);
        out = NULL;
        cap = 0;
        tw->failed = 1;
    }
    j->comp[index] = out;
    j->comp_len[index] = cap;
}

/* Appends one compressed tile as tile ti of grid g.  In a COG it is framed: its byte count as a uint32 LE before it,
 * its last 4 bytes repeated after it (GDAL's BLOCK_LEADER=SIZE_AS_UINT4, BLOCK_TRAILER=LAST_4_BYTES_REPEATED); the
 * tile's offset and byte count are those of the stream itself. */
static int put_tile(gh_tiffw *tw, tw_grid *g, size_t ti, const uint8_t *z, uint32_t n)
{
    const uint32_t frame = tw->cog ? 8 : 0;
    if (tw->pos + n + frame > 0xFFFFFFF0ull || (tw->cog && n < 4)) {
        tw->failed = 1;
        return -1;
    }
    unsigned char lead[4], *q = lead;
    put32(&q, n);
    if ((tw->cog && fwrite(lead, 1, 4, tw->fp) != 4) || fwrite(z, 1, n, tw->fp) != n ||
        (tw->cog && fwrite(z + n - 4, 1, 4, tw->fp) != 4))
        tw->failed = 1;
    g->offsets[ti] = (uint32_t)(tw->pos + frame / 2);
    g->counts[ti] = n;
    tw->pos += n + frame;
    return tw->failed ? -1 : 0;
}

static int grid_init(tw_grid *g, int w, int h)
{
    g->w = w;
    g->h = h;
    g->tiles_x = (w + TILE - 1) / TILE;
    g->tiles_y = (h + TILE - 1) / TILE;
    size_t nt = (size_t)g->tiles_x * (size_t)g->tiles_y;
    g->offsets = calloc(nt, sizeof(uint32_t));
    g->counts = calloc(nt, sizeof(uint32_t));
    return g->offsets && g->counts ? 0 : -1;
}

static void free_grids(gh_tiffw *tw)
{
    for (int k = 0; k <= tw->nlev; k++) {
        free(tw->g[k].offsets);
        free(tw->g[k].counts);
        free(tw->g[k].band);
    }
}

int gh_tiffw_open(const char *path, int w, int h, const double gt[6], gh_tiffw **out, char *err, size_t errlen)
{
    *out = NULL;
    if (w <= 0 || h <= 0) {
        set_err(err, errlen, "write error 3 on %s (empty raster)", path);
        return -1;
    }
    gh_tiffw *tw = calloc(1, sizeof *tw);
    if (!tw)
        return -1;
    /* A block that fails half way (read error, damaged tile, full disk) must not leave a truncated file under the
     * reference's output name: with overwrite off a re-run would keep it and write beside it (cn.c:320-360). */
    tw->path = strdup(path);
    tw->tmp = malloc(strlen(path) + 6);
    if (tw->path && tw->tmp) {
        sprintf(tw->tmp, "%s.part", path);
        tw->fp = fopen(tw->tmp, "wb");
    }
    if (!tw->fp) {
        set_err(err, errlen, "write error 3 on %s (%s)", path, strerror(errno));     /* raster.c:221 */
        free(tw->path);
        free(tw->tmp);
        free(tw);
        return -1;
    }
    setvbuf(tw->fp, NULL, _IOFBF, 1 << 20);     /* tiles arrive as ~1.5 KB pieces: one write(2) per MB, not per tile */
    tw->level = 6;              /* GDAL's default ZLEVEL */
    memcpy(tw->gt, gt, sizeof tw->gt);
    unsigned char hdr[8] = { 'I', 'I', 42, 0, 0, 0, 0, 0 };      /* IFD offset patched on close */
    if (grid_init(&tw->g[0], w, h) || fwrite(hdr, 1, 8, tw->fp) != 8) {
        set_err(err, errlen, "write error 3 on %s", path);
        gh_tiffw_abort(tw);
        return -1;
    }
    tw->pos = 8;
    *out = tw;
    return 0;
}

int gh_tiffw_set_geokeys(gh_tiffw *tw, const gh_geokeys *gk)
{
    if (!tw || !gk || !gk->keys || gk->n_keys < 4 || tw->cog)
        return -1;
    free(tw->geo_keys);
    free(tw->geo_doubles);
    free(tw->geo_ascii);
    tw->geo_keys = malloc(sizeof(uint16_t) * gk->n_keys);
    tw->geo_doubles = gk->n_doubles ? malloc(sizeof(double) * gk->n_doubles) : NULL;
    tw->geo_ascii = gk->n_ascii ? malloc(gk->n_ascii) : NULL;
    if (!tw->geo_keys || (gk->n_doubles && !tw->geo_doubles) || (gk->n_ascii && !tw->geo_ascii)) {
        free(tw->geo_keys);
        free(tw->geo_doubles);
        free(tw->geo_ascii);
        tw->geo_keys = NULL;
        tw->geo_doubles = NULL;
        tw->geo_ascii = NULL;
        tw->n_geo_keys = tw->n_geo_doubles = tw->n_geo_ascii = 0;
        return -1;
    }
    memcpy(tw->geo_keys, gk->keys, sizeof(uint16_t) * gk->n_keys);
    tw->n_geo_keys = gk->n_keys;
    if (gk->n_doubles)
        memcpy(tw->geo_doubles, gk->doubles, sizeof(double) * gk->n_doubles);
    tw->n_geo_doubles = gk->n_doubles;
    if (gk->n_ascii)
        memcpy(tw->geo_ascii, gk->ascii, gk->n_ascii);
    tw->n_geo_ascii = gk->n_ascii;
    /* the outputs' tiepoint is the corner of pixel (0, 0): whatever the source said, they are PixelIsArea */
    for (size_t k = 4; k + 3 < tw->n_geo_keys; k += 4)
        if (tw->geo_keys[k] == 1025 && tw->geo_keys[k + 1] == 0)
            tw->geo_keys[k + 3] = 1;
    return 0;
}

int gh_tiffw_set_overviews(gh_tiffw *tw, int n)
{
    if (!tw || tw->failed || n < 0 || n > GCN10_MAX_OVERVIEWS || tw->nlev || tw->pos != 8 || tw->g[0].next_tile_row)
        return -1;
    const int nlev = gcn10_overview_levels(tw->g[0].w, tw->g[0].h, n);
    for (int k = 1; k <= nlev; k++) {
        tw->nlev = k;
        if (grid_init(&tw->g[k], gcn10_overview_dim(tw->g[0].w, k), gcn10_overview_dim(tw->g[0].h, k))) {
            tw->failed = 1;
            return -1;
        }
    }
    return 0;
}

int gh_tiffw_levels(const gh_tiffw *tw) { return tw ? tw->nlev : -1; }

int gh_tiffw_set_stats(gh_tiffw *tw, int on)
{
    if (!tw || tw->failed || (on != 0 && on != 1) || tw->pos != 8 || tw->g[0].next_tile_row)
        return -1;
    tw->stats = on;
    return 0;
}

int gh_tiffw_set_nodata(gh_tiffw *tw, int on)
{
    if (!tw || tw->failed || (on != 0 && on != 1) || tw->cog)
        return -1;
    tw->nodata = on;
    return 0;
}

int gh_tiffw_put_histogram(gh_tiffw *tw, const uint64_t hist[256])
{
    if (!tw || !hist || !tw->stats)
        return -1;
    for (int v = 0; v < 256; v++)
        tw->hist[v] += hist[v];
    return 0;
}

/* The band statistics GDAL computes for a file whose NoData value is 255, as GDAL stores them in GDAL_METADATA: only
 * pixels other than 255 count, the standard deviation is the population one, VALID_PERCENT = 100 * valid / pixels.  A
 * plane without a valid pixel gets VALID_PERCENT 0 and nothing else.  The sums are exact integers: N * sum(v^2) needs
 * more than 64 bits at 36001 x 36001.  Returns the length of the NUL-terminated text, or -1 if cap is too small. */
static const char k_stats_none[] =
    "<GDALMetadata>\n  <Item name=\"STATISTICS_VALID_PERCENT\" sample=\"0\">%.17g</Item>\n</GDALMetadata>\n";
static const char k_stats_all[] =
    "<GDALMetadata>\n"
    "  <Item name=\"STATISTICS_MAXIMUM\" sample=\"0\">%.17g</Item>\n"
    "  <Item name=\"STATISTICS_MEAN\" sample=\"0\">%.17g</Item>\n"
    "  <Item name=\"STATISTICS_MINIMUM\" sample=\"0\">%.17g</Item>\n"
    "  <Item name=\"STATISTICS_STDDEV\" sample=\"0\">%.17g</Item>\n"
    "  <Item name=\"STATISTICS_VALID_PERCENT\" sample=\"0\">%.17g</Item>\n"
    "</GDALMetadata>\n";

static int stats_metadata(const uint64_t hist[256], uint64_t pixels, char *out, size_t cap)
{
    uint64_t valid = 0, sum = 0;
    unsigned __int128 sum2 = 0;
    int lo = -1, hi = -1;
    for (int v = 0; v < GCN10_NODATA; v++) {
        if (!hist[v])
            continue;
        if (lo < 0)
            lo = v;
        hi = v;
        valid += hist[v];
        sum += hist[v] * (uint64_t)v;
        sum2 += (unsigned __int128)hist[v] * (unsigned)(v * v);
    }
    const double pct = pixels ? 100.0 * (double)valid / (double)pixels : 0.0;
    int n;
    if (!valid) {
        n = snprintf(out, cap, k_stats_none, pct);
    }
    else {
        const unsigned __int128 var_n2 = (unsigned __int128)valid * sum2 - (unsigned __int128)sum * sum;   /* N^2 var */
        const double mean = (double)sum / (double)valid, sd = sqrt((double)var_n2) / (double)valid;
        n = snprintf(out, cap, k_stats_all, (double)hi, mean, (double)lo, sd, pct);
    }
    return n < 0 || (size_t)n >= cap ? -1 : n;
}

/* The most bytes stats_metadata can produce, its NUL included: every number at the longest %.17g prints (24
 * characters: sign, 17 digits, point, a three-digit exponent).  A COG reserves this much before the data, because the
 * statistics are only known at close. */
static size_t stats_metadata_cap(void)
{
    const double x = -1.2345678901234567e-300;
    return (size_t)snprintf(NULL, 0, k_stats_all, x, x, x, x, x) + 1;
}

/* Compresses the tile rows [0, rows) held in data (pitch bytes apart) as the next tile rows of grid g; with `count`
 * their pixels are added to the file's histogram. */
static int append_tile_rows(gh_tiffw *tw, tw_grid *g, const uint8_t *data, size_t pitch, int rows, int threads, int count)
{
    int tile_rows = (rows + TILE - 1) / TILE;
    int n = tile_rows * g->tiles_x;
    write_job j = { tw, g, data, pitch, rows, g->next_tile_row, NULL, NULL, NULL };
    j.comp = calloc((size_t)n, sizeof(unsigned char *));
    j.comp_len = calloc((size_t)n, sizeof(uLongf));
    if (count)
        j.hist = malloc((size_t)n * sizeof *j.hist);
    if (!j.comp || !j.comp_len || (count && !j.hist)) {
        free(j.comp);
        free(j.comp_len);
        free(j.hist);
        tw->failed = 1;
        return -1;
    }
    parallel_for(n, threads, compress_tile, &j);
    for (int i = 0; count && i < n; i++)
        for (int v = 0; v < 256; v++)
            tw->hist[v] += j.hist[i][v];
    free(j.hist);
    for (int i = 0; i < n; i++) {
        size_t ti = (size_t)(g->next_tile_row + i / g->tiles_x) * (size_t)g->tiles_x + (size_t)(i % g->tiles_x);
        if (!tw->failed && j.comp[i])
            put_tile(tw, g, ti, j.comp[i], (uint32_t)j.comp_len[i]);
        free(j.comp[i]);
    }
    free(j.comp);
    free(j.comp_len);
    g->next_tile_row += tile_rows;
    return tw->failed ? -1 : 0;
}

int gh_tiffw_write_rows(gh_tiffw *tw, const uint8_t *data, size_t pitch, int y0, int nrows, int threads)
{
    tw_grid *g0 = &tw->g[0];
    if (tw->failed || tw->cog || y0 != g0->next_tile_row * TILE || y0 + nrows > g0->h ||
        (nrows % TILE != 0 && y0 + nrows != g0->h))
        return -1;
    if (append_tile_rows(tw, g0, data, pitch, nrows, threads, tw->stats))
        return -1;
    /* the overview levels, sampled from this band by the rule of gcn10_overview_src: each level keeps one tile row
     * and appends it compressed when it is full, so the levels cost a few MB, not a third of the raster */
    for (int k = 1; k <= tw->nlev; k++) {
        tw_grid *g = &tw->g[k];
        if (!g->band && !(g->band = malloc((size_t)TILE * (size_t)g->w))) {
            tw->failed = 1;
            return -1;
        }
        for (int i = g->next_tile_row * TILE; i < g->h; i++) {
            const int src = gcn10_overview_src(i, k, g0->h);
            if (src < y0)
                continue;       /* (a band boundary inside a tile row: rows before it were sampled already) */
            if (src >= y0 + nrows)
                break;
            const uint8_t *row = data + (size_t)(src - y0) * pitch;
            uint8_t *dst = g->band + (size_t)(i % TILE) * (size_t)g->w;
            for (int x = 0; x < g->w; x++)
                dst[x] = row[gcn10_overview_src(x, k, g0->w)];
            if (i % TILE == TILE - 1 || i == g->h - 1) {
                if (append_tile_rows(tw, g, g->band, (size_t)g->w, i % TILE + 1, threads, 0))
                    return -1;
            }
        }
    }
    return 0;
}

static int put_grid_tile_row(gh_tiffw *tw, tw_grid *g, int tile_row, const uint8_t *blob, const uint64_t *offsets,
                             const uint32_t *sizes)
{
    if (tw->failed || tile_row != g->next_tile_row || tile_row >= g->tiles_y)
        return -1;
    for (int tx = 0; tx < g->tiles_x; tx++)
        if (put_tile(tw, g, (size_t)tile_row * (size_t)g->tiles_x + (size_t)tx, blob + offsets[tx], sizes[tx]))
            return -1;
    g->next_tile_row++;
    return 0;
}

/* COG: the levels come smallest first (nlev .. 1), then the full resolution; anything else fails the file */
static int cog_accepts(gh_tiffw *tw, int level)
{
    if (!tw->cog)
        return 1;
    while (tw->cog_level > 0 && tw->g[tw->cog_level].next_tile_row == tw->g[tw->cog_level].tiles_y)
        tw->cog_level--;
    if (level == tw->cog_level)
        return 1;
    tw->failed = 1;
    return 0;
}

int gh_tiffw_put_tile_row(gh_tiffw *tw, int tile_row, const uint8_t *blob, const uint64_t *offsets,
                          const uint32_t *sizes)
{
    if (!cog_accepts(tw, 0))
        return -1;
    return put_grid_tile_row(tw, &tw->g[0], tile_row, blob, offsets, sizes);
}

int gh_tiffw_put_tile_rows(gh_tiffw *tw, int tile_row0, int nrows, const uint8_t *blob, const uint64_t *offsets,
                           const uint32_t *sizes)
{
    return gh_tiffw_put_level_tile_rows(tw, 0, tile_row0, nrows, blob, offsets, sizes);
}

int gh_tiffw_put_level_tile_rows(gh_tiffw *tw, int level, int tile_row0, int nrows, const uint8_t *blob,
                                 const uint64_t *offsets, const uint32_t *sizes)
{
    if (!tw || level < 0 || level > tw->nlev)
        return -1;
    tw_grid *g = &tw->g[level];
    if (tw->failed || tile_row0 != g->next_tile_row || nrows < 1 || tile_row0 + nrows > g->tiles_y || !cog_accepts(tw, level))
        return -1;
    const size_t n = (size_t)nrows * (size_t)g->tiles_x;
    /* laid out in table order with small gaps (the library's "ordered" strips)?  Then the whole share is one write;
     * the gaps (< 16 bytes per tile, alignment padding) go into the file as unused bytes, which TIFF allows.  (A COG's
     * tiles need their framing between them: the writer adds it tile by tile.) */
    int ordered = !tw->cog;
    for (size_t i = 0; i + 1 < n && ordered; i++)
        ordered = offsets[i + 1] >= offsets[i] + sizes[i] && offsets[i + 1] - (offsets[i] + sizes[i]) < 64;
    if (!ordered) {
        for (int r = 0; r < nrows; r++)
            if (put_grid_tile_row(tw, g, tile_row0 + r, blob, offsets + (size_t)r * g->tiles_x, sizes + (size_t)r * g->tiles_x))
                return -1;
        return 0;
    }
    const uint64_t first = offsets[0], bytes = offsets[n - 1] + sizes[n - 1] - first;
    if (tw->pos + bytes > 0xFFFFFFF0ull || fwrite(blob + first, 1, (size_t)bytes, tw->fp) != (size_t)bytes) {
        tw->failed = 1;
        return -1;
    }
    for (size_t i = 0; i < n; i++) {
        const size_t ti = (size_t)tile_row0 * (size_t)g->tiles_x + i;
        g->offsets[ti] = (uint32_t)(tw->pos + (offsets[i] - first));
        g->counts[ti] = sizes[i];
    }
    tw->pos += bytes;
    g->next_tile_row += nrows;
    return 0;
}

int gh_tiffw_put_framed_tile_rows(gh_tiffw *tw, int level, int tile_row0, int nrows, const uint8_t *blob,
                                  const uint64_t *offsets, const uint32_t *sizes)
{
    if (!tw || !tw->cog || level < 0 || level > tw->nlev)
        return -1;
    tw_grid *g = &tw->g[level];
    if (tw->failed || tile_row0 != g->next_tile_row || nrows < 1 || tile_row0 + nrows > g->tiles_y || !cog_accepts(tw, level))
        return -1;
    const size_t n = (size_t)nrows * (size_t)g->tiles_x;
    /* every tile framed in place, in table order, with at most alignment padding between one trailer and the next
     * leader: then the share from the first leader to the last trailer is one write */
    for (size_t i = 0; i < n; i++) {
        const uint8_t *z = blob + offsets[i];
        if (offsets[i] < 4 || sizes[i] < 4 ||
            ((uint32_t)z[-4] | (uint32_t)z[-3] << 8 | (uint32_t)z[-2] << 16 | (uint32_t)z[-1] << 24) != sizes[i] ||
            memcmp(z + sizes[i], z + sizes[i] - 4, 4) != 0 ||
            (i + 1 < n && (offsets[i + 1] < offsets[i] + sizes[i] + 8 || offsets[i + 1] - (offsets[i] + sizes[i]) >= 64))) {
            tw->failed = 1;
            return -1;
        }
    }
    const uint64_t first = offsets[0] - 4, bytes = offsets[n - 1] + sizes[n - 1] + 4 - first;
    if (tw->pos + bytes > 0xFFFFFFF0ull || fwrite(blob + first, 1, (size_t)bytes, tw->fp) != (size_t)bytes) {
        tw->failed = 1;
        return -1;
    }
    for (size_t i = 0; i < n; i++) {
        const size_t ti = (size_t)tile_row0 * (size_t)g->tiles_x + i;
        g->offsets[ti] = (uint32_t)(tw->pos + (offsets[i] - first));
        g->counts[ti] = sizes[i];
    }
    tw->pos += bytes;
    g->next_tile_row += nrows;
    return 0;
}

static void put_entry(unsigned char **p, uint16_t tag, uint16_t type, uint32_t count, uint32_t value)
{
    put16(p, tag);
    put16(p, type);
    put32(p, count);
    if (type == 3 && count == 1) { put16(p, (uint16_t)value); put16(p, 0); }
    else put32(p, value);
}

/* What IFD0 and the level IFDs hold besides the tile tables: the georeferencing (the land cover's GeoKeys, or
 * EPSG:4326) and the NoData / statistics tags */
typedef struct {
    const uint16_t *keys;
    size_t nkeys;
    const char *ascii;
    size_t nascii, ndbl;
    int tag_nodata;             /* GDAL_NODATA in every IFD */
    int nent, level_entries;    /* entries of IFD0 and of a level's IFD */
} tw_tags;

static void tags_of(const gh_tiffw *tw, tw_tags *t)
{
    static const uint16_t geokeys[] = {
        1, 1, 0, 4,
        1024, 0, 1, 2,          /* GTModelTypeGeoKey      = ModelTypeGeographic */
        1025, 0, 1, 1,          /* GTRasterTypeGeoKey     = RasterPixelIsArea   */
        2048, 0, 1, 4326,       /* GeographicTypeGeoKey   = WGS 84              */
        2054, 0, 1, 9102,       /* GeogAngularUnitsGeoKey = degree              */
    };
    static const char ascii_default[] = "WGS 84|";
    t->keys = tw->geo_keys ? tw->geo_keys : geokeys;
    t->nkeys = tw->geo_keys ? tw->n_geo_keys : sizeof geokeys / 2;
    t->ascii = tw->geo_keys ? tw->geo_ascii : ascii_default;
    t->nascii = tw->geo_keys ? tw->n_geo_ascii : sizeof ascii_default;
    t->ndbl = tw->geo_keys ? tw->n_geo_doubles : 0;
    t->tag_nodata = tw->stats || tw->nodata;
    t->nent = 14 + 1 + (t->ndbl ? 1 : 0) + (t->nascii ? 1 : 0) + (tw->stats ? 1 : 0) + t->tag_nodata;
    t->level_entries = 13 + t->tag_nodata;
}

/* File offsets of everything the IFDs hold or point to.  end = the first byte after all of it. */
typedef struct {
    uint64_t offsets, counts, scale, tie, keys, dbl, ascii, meta, ifd0;
    uint64_t lv_tables[1 + GCN10_MAX_OVERVIEWS];        /* a level's tile offsets, then its byte counts */
    uint64_t lv_ifd[1 + GCN10_MAX_OVERVIEWS];
    uint64_t end;
} tw_layout;

/* IFD0's arrays and IFD0 at the current (even) end of the data, then per overview level its tables and IFD */
static void trailing_layout(const gh_tiffw *tw, const tw_tags *t, size_t nmeta, tw_layout *L)
{
    const uint64_t nt = (uint64_t)tw->g[0].tiles_x * (uint64_t)tw->g[0].tiles_y;
    L->offsets = tw->pos;
    L->counts = L->offsets + 4 * nt;
    L->scale = L->counts + 4 * nt;
    L->tie = L->scale + 24;
    L->keys = L->tie + 48;
    L->dbl = L->keys + 2 * t->nkeys;
    L->ascii = L->dbl + 8 * t->ndbl;
    L->meta = (L->ascii + t->nascii + 1) & ~(uint64_t)1;     /* word aligned */
    L->ifd0 = (L->meta + nmeta + 1) & ~(uint64_t)1;
    L->end = L->ifd0 + 2 + (uint64_t)t->nent * 12 + 4;
    /* behind IFD0, per overview level: its tile offsets, byte counts and IFD (reduced-resolution image, no geo tags:
     * readers derive the level's georeferencing from the size ratio) */
    for (int k = 1; k <= tw->nlev; k++) {
        L->lv_tables[k] = L->end;
        L->lv_ifd[k] = L->end + 8 * (uint64_t)tw->g[k].tiles_x * (uint64_t)tw->g[k].tiles_y;
        L->end = L->lv_ifd[k] + 2 + (uint64_t)t->level_entries * 12 + 4;
    }
}

/* GDAL's ghost area of a COG (its COG driver writes it; its validator reads it): the layout promises a reader that the
 * IFDs come before the data, tiles in row-major order, each framed by its size and its last 4 bytes */
static const char k_cog_ghost[] = "LAYOUT=IFDS_BEFORE_DATA\n"
                                  "BLOCK_ORDER=ROW_MAJOR\n"
                                  "BLOCK_LEADER=SIZE_AS_UINT4\n"
                                  "BLOCK_TRAILER=LAST_4_BYTES_REPEATED\n"
                                  "KNOWN_INCOMPATIBLE_EDITION=NO\n ";

/* A COG's header region: the TIFF header and the ghost area, IFD0 at the next even offset, the level IFDs from the
 * largest level to the smallest, then every array they point to -- the GDAL_METADATA slot sized for the longest
 * statistics text -- and the data after it.  Known as soon as the tile grids, the georeferencing and the tags are. */
static void cog_layout(const gh_tiffw *tw, const tw_tags *t, tw_layout *L)
{
    const uint64_t ghost = 8 + strlen("GDAL_STRUCTURAL_METADATA_SIZE=000000 bytes\n") + (sizeof k_cog_ghost - 1);
    L->ifd0 = (ghost + 1) & ~(uint64_t)1;
    uint64_t at = L->ifd0 + 2 + (uint64_t)t->nent * 12 + 4;
    for (int k = 1; k <= tw->nlev; k++) {
        L->lv_ifd[k] = at;
        at += 2 + (uint64_t)t->level_entries * 12 + 4;
    }
    const uint64_t nt = (uint64_t)tw->g[0].tiles_x * (uint64_t)tw->g[0].tiles_y;
    L->offsets = at;
    L->counts = L->offsets + 4 * nt;
    at = L->counts + 4 * nt;
    for (int k = 1; k <= tw->nlev; k++) {
        L->lv_tables[k] = at;
        at += 8 * (uint64_t)tw->g[k].tiles_x * (uint64_t)tw->g[k].tiles_y;
    }
    L->scale = at;
    L->tie = L->scale + 24;
    L->keys = L->tie + 48;
    L->dbl = L->keys + 2 * t->nkeys;
    L->ascii = L->dbl + 8 * t->ndbl;
    L->meta = (L->ascii + t->nascii + 1) & ~(uint64_t)1;
    L->end = (L->meta + (tw->stats ? stats_metadata_cap() : 0) + 1) & ~(uint64_t)1;
}

int gh_tiffw_set_cog(gh_tiffw *tw, int on)
{
    if (!tw || tw->failed || (on != 0 && on != 1) || tw->cog || tw->pos != 8)
        return -1;
    for (int k = 0; k <= tw->nlev; k++)
        if (tw->g[k].next_tile_row)
            return -1;
    if (!on)
        return 0;
    tw_tags t;
    tw_layout L;
    tw->cog = 1;
    tags_of(tw, &t);
    cog_layout(tw, &t, &L);
    /* the header region is filled in on close; the tiles follow it */
    unsigned char *zero = calloc(1, (size_t)(L.end - 8));
    if (!zero || fwrite(zero, 1, (size_t)(L.end - 8), tw->fp) != (size_t)(L.end - 8) || L.end + 256 >= 0xFFFFFFF0ull) {
        free(zero);
        tw->failed = 1;
        return -1;
    }
    free(zero);
    tw->pos = tw->cog_data = L.end;
    tw->cog_level = tw->nlev;
    return 0;
}

int gh_tiffw_close(gh_tiffw *tw)
{
    if (!tw)
        return -1;
    int rc = -1;
    const tw_grid *g0 = &tw->g[0];
    size_t nt = (size_t)g0->tiles_x * (size_t)g0->tiles_y;
    int complete = !tw->failed;
    for (int k = 0; k <= tw->nlev; k++)
        complete = complete && tw->g[k].next_tile_row == tw->g[k].tiles_y;
    /* statistics: GDAL_METADATA (42112) in IFD0 and GDAL_NODATA (42113) "255" in every IFD; a histogram that does not
     * count every pixel exactly once (never handed over, or not this raster's) would publish wrong numbers */
    char meta[1024];
    size_t nmeta = 0;
    if (complete && tw->stats) {
        uint64_t total = 0;
        for (int v = 0; v < 256; v++)
            total += tw->hist[v];
        const int n = total == (uint64_t)g0->w * (uint64_t)g0->h ? stats_metadata(tw->hist, total, meta, sizeof meta) : -1;
        complete = n > 0;
        nmeta = n > 0 ? (size_t)n + 1 : 0;
    }
    const uint32_t nodata_ascii = '2' | '5' << 8 | '5' << 16;     /* "255\0", held in the entry itself */
    if (complete) {
        tw_tags t;
        tw_layout L;
        tags_of(tw, &t);
        uint64_t at;            /* buf holds the file's bytes [at, L.end) */
        if (tw->cog) {
            if (nmeta > stats_metadata_cap())
                complete = 0;
            cog_layout(tw, &t, &L);
            at = 0;
        }
        else {
            if (tw->pos & 1) { fputc(0, tw->fp); tw->pos++; }
            trailing_layout(tw, &t, nmeta, &L);
            at = tw->pos;
        }
        size_t tail = (size_t)(L.end - at);
        unsigned char *buf = complete ? calloc(1, tail) : NULL, *p = buf;
        if (buf && L.end + 256 < 0xFFFFFFF0ull) {
            p = buf + (L.offsets - at);
            for (size_t i = 0; i < nt; i++) put32(&p, g0->offsets[i]);
            for (size_t i = 0; i < nt; i++) put32(&p, g0->counts[i]);
            p = buf + (L.scale - at);
            put_f64(&p, tw->gt[1]); put_f64(&p, -tw->gt[5]); put_f64(&p, 0.0);
            put_f64(&p, 0.0); put_f64(&p, 0.0); put_f64(&p, 0.0);
            put_f64(&p, tw->gt[0]); put_f64(&p, tw->gt[3]); put_f64(&p, 0.0);
            for (size_t i = 0; i < t.nkeys; i++) put16(&p, t.keys[i]);
            for (size_t i = 0; i < t.ndbl; i++) put_f64(&p, tw->geo_doubles[i]);
            if (t.nascii)
                memcpy(p, t.ascii, t.nascii);
            if (nmeta)
                memcpy(buf + (L.meta - at), meta, nmeta);
            p = buf + (L.ifd0 - at);
            put16(&p, (uint16_t)t.nent);
            put_entry(&p, 256, 4, 1, (uint32_t)g0->w);
            put_entry(&p, 257, 4, 1, (uint32_t)g0->h);
            put_entry(&p, 258, 3, 1, 8);
            put_entry(&p, 259, 3, 1, 8);                /* Adobe DEFLATE, what GDAL writes */
            put_entry(&p, 262, 3, 1, 1);                /* BlackIsZero */
            put_entry(&p, 277, 3, 1, 1);
            put_entry(&p, 284, 3, 1, 1);
            put_entry(&p, 322, 3, 1, TILE);
            put_entry(&p, 323, 3, 1, TILE);
            put_entry(&p, 324, 4, (uint32_t)nt, nt == 1 ? g0->offsets[0] : (uint32_t)L.offsets);
            put_entry(&p, 325, 4, (uint32_t)nt, nt == 1 ? g0->counts[0] : (uint32_t)L.counts);
            put_entry(&p, 339, 3, 1, 1);                /* SampleFormat = unsigned */
            put_entry(&p, 33550, 12, 3, (uint32_t)L.scale);
            put_entry(&p, 33922, 12, 6, (uint32_t)L.tie);
            put_entry(&p, 34735, 3, (uint32_t)t.nkeys, (uint32_t)L.keys);
            if (t.ndbl)
                put_entry(&p, 34736, 12, (uint32_t)t.ndbl, (uint32_t)L.dbl);
            if (t.nascii)
                put_entry(&p, 34737, 2, (uint32_t)t.nascii, (uint32_t)L.ascii);
            if (tw->stats)
                put_entry(&p, 42112, 2, (uint32_t)nmeta, (uint32_t)L.meta);
            if (t.tag_nodata)
                put_entry(&p, 42113, 2, 4, nodata_ascii);
            put32(&p, tw->nlev ? (uint32_t)L.lv_ifd[1] : 0);
            for (int k = 1; k <= tw->nlev; k++) {
                const tw_grid *g = &tw->g[k];
                const size_t n = (size_t)g->tiles_x * (size_t)g->tiles_y;
                p = buf + (L.lv_tables[k] - at);
                for (size_t i = 0; i < n; i++) put32(&p, g->offsets[i]);
                for (size_t i = 0; i < n; i++) put32(&p, g->counts[i]);
                p = buf + (L.lv_ifd[k] - at);
                put16(&p, (uint16_t)t.level_entries);
                put_entry(&p, 254, 4, 1, 1);            /* NewSubfileType = reduced-resolution version */
                put_entry(&p, 256, 4, 1, (uint32_t)g->w);
                put_entry(&p, 257, 4, 1, (uint32_t)g->h);
                put_entry(&p, 258, 3, 1, 8);
                put_entry(&p, 259, 3, 1, 8);
                put_entry(&p, 262, 3, 1, 1);
                put_entry(&p, 277, 3, 1, 1);
                put_entry(&p, 284, 3, 1, 1);
                put_entry(&p, 322, 3, 1, TILE);
                put_entry(&p, 323, 3, 1, TILE);
                put_entry(&p, 324, 4, (uint32_t)n, n == 1 ? g->offsets[0] : (uint32_t)L.lv_tables[k]);
                put_entry(&p, 325, 4, (uint32_t)n, n == 1 ? g->counts[0] : (uint32_t)(L.lv_tables[k] + 4 * n));
                put_entry(&p, 339, 3, 1, 1);
                if (t.tag_nodata)
                    put_entry(&p, 42113, 2, 4, nodata_ascii);
                put32(&p, k < tw->nlev ? (uint32_t)L.lv_ifd[k + 1] : 0);
            }
            if (tw->cog) {
                /* the header region: TIFF header, GDAL's ghost area, then everything above, in place before the data */
                p = buf;
                put16(&p, 'I' | 'I' << 8);
                put16(&p, 42);
                put32(&p, (uint32_t)L.ifd0);
                snprintf((char *)buf + 8, L.ifd0 - 8, "GDAL_STRUCTURAL_METADATA_SIZE=%06d bytes\n%s",
                         (int)(sizeof k_cog_ghost - 1), k_cog_ghost);
                if (L.end == tw->cog_data && fseek(tw->fp, 0, SEEK_SET) == 0 && fwrite(buf, 1, tail, tw->fp) == tail)
                    rc = 0;
            }
            else if (fwrite(buf, 1, tail, tw->fp) == tail && fseek(tw->fp, 4, SEEK_SET) == 0) {
                unsigned char o[4], *q = o;
                put32(&q, (uint32_t)L.ifd0);
                if (fwrite(o, 1, 4, tw->fp) == 4)
                    rc = 0;
            }
        }
        free(buf);
    }
    if (fclose(tw->fp) != 0)
        rc = -1;
    if (rc == 0 && rename(tw->tmp, tw->path) != 0)
        rc = -1;
    if (rc != 0)
        unlink(tw->tmp);
    free(tw->geo_keys);
    free(tw->geo_doubles);
    free(tw->geo_ascii);
    free(tw->path);
    free(tw->tmp);
    free_grids(tw);
    free(tw);
    return rc;
}

void gh_tiffw_abort(gh_tiffw *tw)
{
    if (!tw)
        return;
    if (tw->fp)
        fclose(tw->fp);
    if (tw->tmp)
        unlink(tw->tmp);
    free(tw->geo_keys);
    free(tw->geo_doubles);
    free(tw->geo_ascii);
    free(tw->path);
    free(tw->tmp);
    free_grids(tw);
    free(tw);
}

int gh_tiff_write(const char *path, const uint8_t *data, int w, int h, size_t pitch, const double gt[6],
                  int threads, char *err, size_t errlen)
{
    gh_tiffw *tw;
    if (gh_tiffw_open(path, w, h, gt, &tw, err, errlen))
        return -1;
    /* bands of 16 tile rows keep the compressed scratch small */
    for (int y0 = 0; y0 < h; y0 += 16 * TILE) {
        int rows = h - y0 < 16 * TILE ? h - y0 : 16 * TILE;
        if (gh_tiffw_write_rows(tw, data + (size_t)y0 * pitch, pitch, y0, rows, threads)) {
            set_err(err, errlen, "write error 3 on %s", path);
            gh_tiffw_abort(tw);
            return -1;
        }
    }
    if (gh_tiffw_close(tw)) {
        set_err(err, errlen, "write error 3 on %s", path);
        return -1;
    }
    return 0;
}

int gh_tiff_write_cog(const char *path, const uint8_t *data, int w, int h, size_t pitch, const double gt[6], int overviews,
                      int threads, char *err, size_t errlen)
{
    gh_tiffw *tw;
    if (gh_tiffw_open(path, w, h, gt, &tw, err, errlen))
        return -1;
    int rc = gh_tiffw_set_overviews(tw, overviews) || gh_tiffw_set_cog(tw, 1);
    /* the levels first, the smallest first, each sampled whole (a level is at most a quarter of the raster); then the
     * full resolution, in bands of 16 tile rows */
    for (int k = tw->nlev; k >= 0 && !rc; k--) {
        tw_grid *g = &tw->g[k];
        uint8_t *lv = k ? malloc((size_t)g->w * (size_t)g->h) : NULL;
        if (k && !lv) {
            rc = -1;
            break;
        }
        for (int i = 0; k && i < g->h; i++) {
            const uint8_t *row = data + (size_t)gcn10_overview_src(i, k, h) * pitch;
            for (int x = 0; x < g->w; x++)
                lv[(size_t)i * g->w + x] = row[gcn10_overview_src(x, k, w)];
        }
        const uint8_t *src = k ? lv : data;
        const size_t sp = k ? (size_t)g->w : pitch;
        for (int y0 = 0; y0 < g->h && !rc; y0 += 16 * TILE)
            rc = append_tile_rows(tw, g, src + (size_t)y0 * sp, sp, g->h - y0 < 16 * TILE ? g->h - y0 : 16 * TILE, threads, 0);
        free(lv);
    }
    if (rc) {
        set_err(err, errlen, "write error 3 on %s", path);
        gh_tiffw_abort(tw);
        return -1;
    }
    if (gh_tiffw_close(tw)) {
        set_err(err, errlen, "write error 3 on %s", path);
        return -1;
    }
    return 0;
}

/* ---- mean rasters on the host (gh_aggregate_*) ---- */

struct gh_aggregate {
    int w, h, f, cw, ch;
    uint32_t *sum, *cnt;        /* the cell row in progress */
    int next_y, next_cell;      /* the next plane row and cell row */
    uint8_t *buf;               /* completed cell rows not yet written: rows buf_row0 .. + buf_rows */
    int buf_rows, buf_cap, buf_row0;
};

gh_aggregate *gh_aggregate_new(int w, int h, int f)
{
    if (w <= 0 || h <= 0 || f < 2 || f > GCN10_MAX_AGGREGATE)
        return NULL;
    gh_aggregate *a = calloc(1, sizeof *a);
    if (!a)
        return NULL;
    a->w = w;
    a->h = h;
    a->f = f;
    a->cw = gcn10_aggregate_dim(w, f);
    a->ch = gcn10_aggregate_dim(h, f);
    a->sum = calloc((size_t)a->cw, sizeof *a->sum);
    a->cnt = calloc((size_t)a->cw, sizeof *a->cnt);
    if (!a->sum || !a->cnt) {
        gh_aggregate_free(a);
        return NULL;
    }
    return a;
}

void gh_aggregate_free(gh_aggregate *a)
{
    if (!a)
        return;
    free(a->sum);
    free(a->cnt);
    free(a->buf);
    free(a);
}

int gh_aggregate_rows(gh_aggregate *a, const uint8_t *data, size_t pitch, int y0, int nrows, uint8_t *out, size_t out_pitch,
                      int *row0)
{
    if (!a || !data || !out || nrows < 0 || y0 != a->next_y || nrows > a->h - y0 || out_pitch < (size_t)a->cw)
        return -1;
    if (row0)
        *row0 = a->next_cell;
    int n = 0;
    for (int y = y0; y < y0 + nrows; y++) {
        const uint8_t *row = data + (size_t)(y - y0) * pitch;
        for (int cx = 0, x = 0; cx < a->cw; cx++) {
            const int xe = x + a->f < a->w ? x + a->f : a->w;
            uint32_t s = 0, c = 0;
            for (; x < xe; x++)
                if (row[x] != GCN10_NODATA) {
                    s += row[x];
                    c++;
                }
            a->sum[cx] += s;
            a->cnt[cx] += c;
        }
        if ((y + 1) % a->f == 0 || y + 1 == a->h) {
            uint8_t *o = out + (size_t)n * out_pitch;
            for (int cx = 0; cx < a->cw; cx++)
                o[cx] = gcn10_aggregate_value(a->sum[cx], a->cnt[cx]);
            memset(a->sum, 0, (size_t)a->cw * sizeof *a->sum);
            memset(a->cnt, 0, (size_t)a->cw * sizeof *a->cnt);
            n++;
        }
    }
    a->next_y = y0 + nrows;
    a->next_cell += n;
    return n;
}

int gh_aggregate_write_rows(gh_aggregate *a, gh_tiffw *tw, const uint8_t *data, size_t pitch, int y0, int nrows, int threads)
{
    if (!a || !tw)
        return -1;
    const int most = nrows / a->f + 2;                  /* cell rows this band can complete (the last one short) */
    if (a->buf_rows + most > a->buf_cap) {
        const int cap = a->buf_rows + most + TILE;
        uint8_t *b = realloc(a->buf, (size_t)cap * (size_t)a->cw);
        if (!b)
            return -1;
        a->buf = b;
        a->buf_cap = cap;
    }
    if (a->buf_rows == 0)
        a->buf_row0 = a->next_cell;
    const int n = gh_aggregate_rows(a, data, pitch, y0, nrows, a->buf + (size_t)a->buf_rows * a->cw, (size_t)a->cw, NULL);
    if (n < 0)
        return -1;
    a->buf_rows += n;
    const int done = a->buf_row0 + a->buf_rows == a->ch;
    const int put = done ? a->buf_rows : a->buf_rows / TILE * TILE;
    if (put > 0) {
        if (gh_tiffw_write_rows(tw, a->buf, (size_t)a->cw, a->buf_row0, put, threads))
            return -1;
        memmove(a->buf, a->buf + (size_t)put * a->cw, (size_t)(a->buf_rows - put) * a->cw);
        a->buf_rows -= put;
        a->buf_row0 += put;
    }
    return 0;
}
