/* gcn10_b200/host/gcn10_main.c -- command line of the B200 Curve Number generator.
 *
 * Keeps the reference's CLI surface (/root/reference/src/main.c:16-36, 85-98): --config/-c,
 * --blocks/-l (the usage text also advertises -b, accepted here too), --overwrite/-o, --help/-h,
 * --version/-v, the same config file and block list formats, outputs under
 * ./cn_rasters_{drained,undrained}/ and logs under <log_dir>/rank_<n>.log.  It is launched
 * directly (no mpirun): the ranks of the reference become one worker thread per visible B200.
 * Extra flags: --gpus N (default: all), --io-threads N (per worker), --outdir DIR (default: CWD).
 */
#include "gcn10_host.h"
#include "../../include/gcn10_cuda.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#ifndef GCN10_VERSION
#define GCN10_VERSION "0.1.0"       /* main.c:12-14 */
#endif

static void usage(FILE *fp)
{
    fprintf(fp,
            "gcn10 - high-resolution curve number generator (B200 / CUDA build)\n"
            "usage:\n"
            "  gcn10 --config <config.txt> [--blocks <blocks.txt>] [--overwrite] [--gpus <n>]\n"
            "  gcn10 --help | -h | --version | -v\n"
            "\n"
            "options:\n"
            "  --config, -c <file>	path to config file (required)\n"
            "  --blocks, -l, -b <file>	optional list of block ids to process\n"
            "  --overwrite, -o	overwrite existing outputs if present (optional)\n"
            "  --gpus <n>		number of GPU workers (default: every visible GPU)\n"
            "  --io-threads <n>	decode/encode threads per worker (default: cores / workers)\n"
            "  --workers-per-gpu <n>	blocks in flight per GPU, each with its own context (default: 1)\n"
            "  --outdir <dir>	where cn_rasters_<condition>/ are created (default: .)\n"
            "  --overviews		also write reduced-resolution overview levels into every output\n"
            "			(nearest neighbour, halving until a level fits one 256 x 256 tile)\n"
            "  --stats		tag every output with NoData 255 and its band statistics (minimum, maximum,\n"
            "			mean, standard deviation, valid percent), counted on the GPU\n"
            "  --aggregate <f>	also write the f x f mean of every output (the composite Curve Number of\n"
            "			cells of f x f pixels, nodata 255 left out; f = 2..1024, 25 = the 250 m soil\n"
            "			grid) to cn_rasters_<condition>_agg<f>/, computed on the GPU\n"
            "  --cog		write every output as a Cloud Optimized GeoTIFF: header first, overview\n"
            "			levels before the full resolution (turns --overviews on), tiles framed as\n"
            "			GDAL's COG driver frames them; with --aggregate the mean rasters too\n"
            "  --help, -h		show this help and exit\n"
            "  --version, -v	print version and exit\n"
            "\n"
            "notes:\n"
            "  one worker thread per GPU takes the place of one mpi rank; blocks are handed out\n"
            "  from a shared queue instead of round-robin, nothing else about a run changes.\n");
}

int main(int argc, char **argv)
{
    /* meta flags first, before anything touches CUDA (main.c:39-56,67) */
    for (int i = 1; i < argc; i++) {
        if (!strcmp(argv[i], "--help") || !strcmp(argv[i], "-h")) {
            usage(stdout);
            return 0;
        }
        if (!strcmp(argv[i], "--version") || !strcmp(argv[i], "-v")) {
            printf("gcn10 %s\n", GCN10_VERSION);                /* main.c:51 */
            return 0;
        }
    }

    const char *conf = NULL, *list = NULL;
    gh_run_options opt;
    memset(&opt, 0, sizeof opt);
    for (int i = 1; i < argc; i++) {                            /* main.c:85-98 */
        if ((!strcmp(argv[i], "-c") || !strcmp(argv[i], "--config")) && i + 1 < argc)
            conf = argv[++i];
        else if ((!strcmp(argv[i], "-l") || !strcmp(argv[i], "-b") || !strcmp(argv[i], "--blocks")) && i + 1 < argc)
            list = argv[++i];
        else if (!strcmp(argv[i], "-o") || !strcmp(argv[i], "--overwrite"))
            opt.overwrite = 1;
        else if (!strcmp(argv[i], "--gpus") && i + 1 < argc)
            opt.n_gpus = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--io-threads") && i + 1 < argc)
            opt.io_threads = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--workers-per-gpu") && i + 1 < argc)
            opt.workers_per_gpu = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--outdir") && i + 1 < argc)
            opt.out_root = argv[++i];
        else if (!strcmp(argv[i], "--overviews"))
            opt.overviews = GCN10_MAX_OVERVIEWS;
        else if (!strcmp(argv[i], "--stats"))
            opt.stats = 1;
        else if (!strcmp(argv[i], "--cog"))
            opt.cog = 1;
        else if (!strcmp(argv[i], "--aggregate") && i + 1 < argc) {
            char *end = NULL;
            const long f = strtol(argv[++i], &end, 10);
            if (!end || *end || f < 2 || f > GCN10_MAX_AGGREGATE) {
                fprintf(stderr, "[rank 0] --aggregate takes a factor from 2 to %d, not '%s'\n", GCN10_MAX_AGGREGATE, argv[i]);
                return 1;
            }
            opt.aggregate = (int)f;
        }
    }
    if (!conf) {
        fprintf(stderr, "[rank 0] missing -c/--config <file>; see 'gcn10 -h' for usage.\n");    /* main.c:103-107 */
        return 1;
    }
    /* a COG's levels come before its full resolution: the GPU makes them from the whole block first */
    if (opt.cog)
        opt.overviews = GCN10_MAX_OVERVIEWS;
    char err[GH_ERRLEN] = "";
    if (gh_config_parse(conf, &opt.cfg, err, sizeof err)) {
        fprintf(stderr, "%s\n", err);                           /* config.c:52,108-111 */
        return 1;
    }
    fprintf(stderr,
            "config loaded:\n"
            "  hysogs_data_path   = %s\n"
            "  esa_data_path      = %s\n"
            "  blocks_shp_path    = %s\n"
            "  lookup_table_path  = %s\n"
            "  log_dir            = %s\n",                      /* main.c:114-125 */
            opt.cfg.hysogs_data_path, opt.cfg.esa_data_path, opt.cfg.blocks_shp_path,
            opt.cfg.lookup_table_path, opt.cfg.log_dir);

    int *ids = NULL, n = 0;
    if (list) {
        if (gh_read_block_list(list, &ids, &n) || n == 0) {
            fprintf(stderr, "no ids found in %s\n", list);      /* main.c:134-137 */
            return 1;
        }
    }
    else {
        /* every block of the shapefile (get_all_blocks, raster.c:68-103; the reference's version
         * increments the wrong thing at raster.c:97 -- here the ids are simply collected) */
        gh_blocks *b = NULL;
        if (gh_blocks_open(opt.cfg.blocks_shp_path, &b, err, sizeof err)) {
            fprintf(stderr, "failed to read shapefile %s\n", opt.cfg.blocks_shp_path);   /* main.c:143-146 */
            return 1;
        }
        n = gh_blocks_count(b);
        ids = malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
        for (int i = 0; i < n; i++)
            ids[i] = gh_blocks_id(b, i);
        gh_blocks_close(b);
        if (n == 0) {
            fprintf(stderr, "no blocks found in %s\n", opt.cfg.blocks_shp_path);         /* main.c:148-151 */
            return 1;
        }
    }
    if (opt.io_threads <= 0) {
        long cores = sysconf(_SC_NPROCESSORS_ONLN);
        opt.io_threads = (int)(cores > 0 ? cores : 4);          /* split between workers in gh_run_blocks */
    }
    fprintf(stderr, "processing %d blocks %s\n", n, list ? "from list file" : "from shapefile");   /* main.c:165-167 */
    int done = gh_run_blocks(&opt, ids, n);
    fprintf(stderr, "%d of %d blocks produced all 18 rasters\n", done, n);
    free(ids);
    gh_config_free(&opt.cfg);
    return 0;                                                   /* main.c:202: EXIT_SUCCESS even if blocks were skipped */
}
