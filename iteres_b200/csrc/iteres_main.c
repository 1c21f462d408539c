/* iteres_main.c -- the `iteres` command line tool on top of libiteres_gpu.so.
 *
 * Same sub-commands, option letters, defaults, positional arguments and output file names as the
 * reference drivers (iteres.c:17-29, stat.c:30-186, filter.c:30-161, cpgstat.c:16-95,
 * cpgfilter.c:19-110), so it is a drop-in for `iteres stat | filter | cpgstat | cpgfilter`.
 * nameStat / subfamStat are aliases (BASELINE.json's names): nameStat == filter, subfamStat == stat.
 * The scan itself runs on the CUDA device through the C ABI of include/iteres_gpu.h; failures keep
 * the reference's convention: message on stderr, exit status 255 (cuskent/errabort.c:166-181).
 *
 * Every option of the reference drivers is accepted.
 */
#define _GNU_SOURCE
#include <getopt.h>
#include <libgen.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <pthread.h>
#include <unistd.h>
#include "../../include/iteres_gpu.h"

#define REF_VERSION "0.3.3-r123"

static void die(const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap);
    fputc('\n', stderr);
    exit(-1);
}
static char *fmt_alloc(const char *fmt, ...) {
    char *s = NULL; va_list ap; va_start(ap, fmt);
    if (vasprintf(&s, fmt, ap) < 0) die("Mem Error.");
    va_end(ap);
    return s;
}
/* basename without its last extension (generic.c:7-15) */
static char *stem(const char *path) {
    char *tmp = strdup(path), *b = strdup(basename(tmp));
    char *dot = strrchr(b, '.');
    if (dot && dot != b) *dot = 0;
    free(tmp);
    return b;
}
static unsigned int uarg(const char *s) { return (unsigned int)strtol(s, 0, 0); }

typedef struct { const char *flag, *text; } optline;
static int print_usage(const char *what, const char *synopsis, const optline *o) {
    fprintf(stderr, "\n%s\n\nUsage:   %s\n\n", what, synopsis);
    for (int i = 0; o[i].flag; i++) fprintf(stderr, "%s -%s       %s\n", i ? "        " : "Options:", o[i].flag, o[i].text);
    fprintf(stderr, "\n");
    return 1;
}

static const optline STAT_OPTS[] = {
    {"S", "input is SAM [off]"}, {"Q", "unique reads mapping Quality threshold [10]"}, {"c", "coverage threshold for overlapping [0.0001]"},
    {"x", "discard multi-reads if mapped to different subfamily [on]"},
    {"N", "normalized by number of (0: reads in repeats, 1: non-redundant reads, 2: mapped reads, 3: total reads) [0])"},
    {"U", "unique reads normalized by number of (0: unique mapped reads in repeats, 1: unique mapped reads, 2: total reads) [0])"},
    {"R", "remove redundant reads [off]"}, {"T", "treat 1 paired-end read as 2 single-end reads [off]"},
    {"D", "discard if only one end mapped in a paired end reads [off]"}, {"w", "keep the wiggle file [off]"},
    {"B", "output bed file of mapped reads [off]"}, {"V", "output bed file of unique mapped reads [off]"},
    {"C", "Add 'chr' string as prefix of reference sequence [off]"}, {"E", "extend reads to represent fragment [150], specify 0 if want no extension"},
    {"I", "Insert length threshold [500]"}, {"o", "output prefix [basename of input without extension]"}, {"h", "help message"}, {"?", "help message"}, {0, 0}};
static const optline FILTER_OPTS[] = {
    {"S", "input is SAM [off]"}, {"Q", "unique reads mapping Quality threshold [10]"}, {"g", "coverage threshold for overlapping [0.0001]"},
    {"N", "normalized by number of (0: unique reads, 1: non-redundant reads, 2: mapped reads, 3: used read ends) [0]"},
    {"n", "repName filter"}, {"c", "repClass filter"}, {"f", "repFamily filter"}, {"t", "only output repeats with at least this many reads [1]"},
    {"r", "output the list of reads of each repeat [off]"}, {"R", "remove redundant reads [off]"},
    {"T", "treat 1 paired-end read as 2 single-end reads [off]"}, {"D", "discard if only one end mapped in a paired end reads [off]"},
    {"C", "Add 'chr' string as prefix of reference sequence [off]"}, {"E", "extend reads to represent fragment [150], specify 0 if want no extension"},
    {"I", "Insert length threshold [500]"}, {"o", "output prefix [basename of input without extension]"}, {"h", "help message"}, {"?", "help message"}, {0, 0}};
static const optline CPGSTAT_OPTS[] = {{"w", "keep the wiggle file [off]"}, {"o", "output prefix [basename of input without extension]"}, {"h", "help message"}, {"?", "help message"}, {0, 0}};
static const optline CPGFILTER_OPTS[] = {{"n", "repName filter"}, {"c", "repClass filter"}, {"f", "repFamily filter"}, {"t", "CpG score threshold [0]"},
    {"o", "output prefix [basename of input without extension]"}, {"h", "help message"}, {"?", "help message"}, {0, 0}};

static int stat_usage(void) { return print_usage("Obtain alignment statistics for each repeat subfamily, family and class.",
    "iteres stat [options] <chromosome size file> <repeat size file> <rmsk.txt> <bam/sam alignment file1,file2,file3...>", STAT_OPTS); }
static int filter_usage(void) { return print_usage("Filter alignment statistics on repName, repClass or repFamily; one row per repeat locus.",
    "iteres filter [options] <chromosome size file> <repeat size file> <rmsk.txt> <bam/sam alignment file>", FILTER_OPTS); }
static int cpgstat_usage(void) { return print_usage("Obtain CpG statistics for each repeat subfamily, family and class.",
    "iteres cpgstat [options] <chromosome size file> <repeat size file> <rmsk.txt> <CpG bedGraph file>", CPGSTAT_OPTS); }
static int cpgfilter_usage(void) { return print_usage("Filter CpG statistics on repName, repClass or repFamily; one row per repeat locus.",
    "iteres cpgfilter [options] <chromosome size file> <repeat size file> <rmsk.txt> <CpG bedGraph file>", CPGFILTER_OPTS); }

static void use_device(void) {
    /* the device itself is first touched by itx_index_build (which fails with "no usable CUDA device" when there is none) */
    const char *d = getenv("ITERES_DEVICE");
    if (d && itx_set_device(atoi(d)) != ITX_OK) die("cannot use CUDA device %s", d);
}
/* ITERES_GPUS=N: the job is split over N devices (ITERES_DEVICE, ITERES_DEVICE + 1, ...), one host thread and one index per device.
 * Alignments: ONE file list, every rank scans its BGZF block range of every file (itx_scan_alignments_shard); CpG: every rank its part of
 * the bedGraph's lines; then ONE allreduce of the counter block, and rank 0 writes the tables -- the same bytes as a single device writes
 * (integer sums; CpG score sums within 1e-9 relative).  -R exchanges the duplicate keys of every part between the devices
 * (itx_scan_alignments_shard); the side outputs that follow the reads in file order (-B, -V, -r) and SAM text run on one device. */
typedef struct {
    int rank, n, dev0; const char *cs, *rs, *rm; int field; const char *fname; const uint8_t *uid;
    int cpg, cpg_filter; const char *input; const itx_scan_opts *o;
    itx_index *ix; uint64_t cnt[13]; int rc; char err[ITX_ERRLEN];
} gpu_rank;
static void *gpu_rank_main(void *arg) {
    gpu_rank *g = (gpu_rank *)arg;
    g->rc = ITX_OK; g->err[0] = 0;
    g->ix = itx_index_build_on(g->dev0 + g->rank, g->cs, g->rs, g->rm, g->field, g->fname, g->err);
    if (!g->ix) { g->rc = ITX_EFORMAT; return NULL; }
    if ((g->rc = itx_comm_init(g->ix, g->uid, g->rank, g->n, g->err))) return NULL;
    if (g->cpg) { uint32_t a = 0, b = 0; g->rc = itx_scan_cpg_shard(g->ix, g->input, g->cpg_filter, g->rank, g->n, &a, &b, g->err); }
    else g->rc = itx_scan_alignments_shard(g->ix, g->input, g->o, g->cnt, g->err);
    if (g->rc) return NULL;
    g->rc = itx_comm_allreduce_counts(g->ix, g->err);
    if (g->rc == ITX_OK) itx_get_counters(g->ix, g->cnt);
    return NULL;
}
static int n_gpus_wanted(void) {
    const char *v = getenv("ITERES_GPUS");
    int n = v ? atoi(v) : 1;
    if (n < 1) n = 1;
    if (n > 64) n = 64;
    return n;
}
/* the whole multi-device run; returns rank 0's index, holding the job's counters (cnt filled for alignment scans) */
static itx_index *run_on_gpus(int n, const char *cs, const char *rs, const char *rm, int field, const char *fname, int cpg, int cpg_filter,
                              const char *input, const itx_scan_opts *o, uint64_t cnt[13]) {
    static uint8_t uid[ITX_NCCL_ID_BYTES];
    char err[ITX_ERRLEN];
    if (itx_device_count() < n) die("ITERES_GPUS=%d, but only %d CUDA device(s) are visible", n, itx_device_count());
    if (itx_comm_unique_id(uid, err) != ITX_OK) die("%s", err);
    const char *d0 = getenv("ITERES_DEVICE");
    gpu_rank *g = (gpu_rank *)calloc((size_t)n, sizeof(gpu_rank));
    pthread_t *th = (pthread_t *)calloc((size_t)n, sizeof(pthread_t));
    for (int r = 0; r < n; r++) {
        g[r].rank = r; g[r].n = n; g[r].dev0 = d0 ? atoi(d0) : 0; g[r].cs = cs; g[r].rs = rs; g[r].rm = rm; g[r].field = field; g[r].fname = fname; g[r].uid = uid;
        g[r].cpg = cpg; g[r].cpg_filter = cpg_filter; g[r].input = input; g[r].o = o;
        if (pthread_create(&th[r], NULL, gpu_rank_main, &g[r]) != 0) die("cannot start the thread of device %d", r);
    }
    for (int r = 0; r < n; r++) pthread_join(th[r], NULL);
    for (int r = 0; r < n; r++) if (g[r].rc != ITX_OK) die("%s", g[r].err[0] ? g[r].err : "a device failed");
    if (cnt) memcpy(cnt, g[0].cnt, sizeof g[0].cnt);
    itx_index *ix = g[0].ix;
    for (int r = 1; r < n; r++) itx_index_free(g[r].ix);
    free(th); free(g);
    return ix;
}

static void done_in(time_t t0) { fprintf(stderr, "* Done, time used %.0f seconds.\n", difftime(time(NULL), t0)); }

/* which of -n / -c / -f was given -> (rmsk column, name) as filter.c:93-113 */
static int pick_filter(char *name, char *cls, char *fam, char **subfam) {
    int field = 0;
    if ((name && cls) || (name && fam) || (cls && fam)) die("Please specify only one filter, either -n, -c or -f.");
    *subfam = strdup("ALL");
    if (name) { *subfam = name; field = 10; } else if (cls) { *subfam = cls; field = 11; } else if (fam) { *subfam = fam; field = 12; }
    if (strcmp(*subfam, "ALL") == 0) { fprintf(stderr, "* You didn't specify any filter, will output all repeats\n"); field = 0; }
    return field;
}

static double lap_ms(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec * 1e3 + t.tv_nsec * 1e-6; }
static double g_t0;
#define LAP(what) do { if (getenv("ITX_TIMING")) fprintf(stderr, "[itx timing] cli: %s at %.0f ms\n", what, lap_ms() - g_t0); } while (0)

typedef struct { const char *wig, *sizes, *out; int rc; char err[ITX_ERRLEN]; } bw_job;
static void *bw_run(void *arg) { bw_job *j = (bw_job *)arg; j->rc = itx_wig_to_bigwig(j->wig, j->sizes, j->out, j->err); return NULL; }

static int main_stat(int argc, char **argv) {
    g_t0 = lap_ms();
    itx_scan_opts o; itx_scan_opts_default(&o);
    int c, keep_wig = 0, sam = 0, bed = 0, bedu = 0; unsigned int norm = 0, norm2 = 0; char *prefix = NULL;
    time_t t0 = time(NULL);
    while ((c = getopt(argc, argv, "SQ:c:xN:U:RTDwBVCo:E:I:h?")) >= 0) {
        switch (c) {
            case 'S': sam = 1; break;
            case 'Q': o.mapQ = uarg(optarg); break;
            case 'c': o.minCoverage = (float)atof(optarg); break;
            case 'x': o.diffSubfam = 0; break;
            case 'N': norm = uarg(optarg); break;
            case 'U': norm2 = uarg(optarg); break;
            case 'R': o.rmDup = 1; break;
            case 'T': o.treat = 1; break;
            case 'D': o.discardWrongEnd = 1; break;
            case 'w': keep_wig = 1; break;
            case 'B': bed = 1; break;
            case 'V': bedu = 1; break;
            case 'C': o.addChr = 1; break;
            case 'E': o.extension = uarg(optarg); break;
            case 'I': o.iSize = uarg(optarg); break;
            case 'o': prefix = strdup(optarg); break;
            case 'h': case '?': return stat_usage();
            default: return 1;
        }
    }
    if (optind + 4 > argc) return stat_usage();
    const char *chrom_sizes = argv[optind], *rep_sizes = argv[optind + 1], *rmsk = argv[optind + 2], *bams = argv[optind + 3];
    int nfiles = 1; for (const char *p = bams; *p; p++) if (*p == ',') nfiles++;
    fprintf(stderr, "* Provided %i BAM/SAM file(s)\n", nfiles);
    if (!prefix) { char *first = strdup(bams); char *comma = strchr(first, ','); if (comma) *comma = 0; prefix = stem(first); free(first); }
    static const int NIDX[4] = {9, 8, 6, 0}, NIDX2[3] = {10, 7, 0};
    if (norm > 3 || norm2 > 2) die("Wrong normalization method specified");
    o.isSam = sam;
    if (bed) o.outbed = fmt_alloc("%s.iteres.bed", prefix);
    if (bedu) o.outbed_unique = fmt_alloc("%s.iteres.unique.bed", prefix);
    use_device();
    char err[ITX_ERRLEN]; uint64_t cnt[13];
    itx_index *ix;
    const int ngpu = (bed || bedu || sam) ? 1 : n_gpus_wanted();
    if (ngpu != n_gpus_wanted()) fprintf(stderr, "* -B, -V and -S follow the reads in file order: running on one GPU\n");
    fprintf(stderr, "* Parsing the rmsk file\n");
    if (ngpu > 1) {
        ix = run_on_gpus(ngpu, chrom_sizes, rep_sizes, rmsk, 0, "ALL", 0, 0, bams, &o, cnt);
        fprintf(stderr, "* Total %lld repeats found.\n* Parsing the SAM/BAM file\n", (long long)itx_n_repeats_parsed(ix));
    } else {
    ix = itx_index_build(chrom_sizes, rep_sizes, rmsk, 0, "ALL", err);
    if (!ix) die("%s", err);
    fprintf(stderr, "* Total %lld repeats found.\n", (long long)itx_n_repeats_parsed(ix));
    LAP("index built");
    fprintf(stderr, "* Parsing the SAM/BAM file\n");
    if (itx_scan_alignments(ix, bams, &o, cnt, err) != ITX_OK) die("%s", err);
    }
    LAP("alignments scanned");
    fprintf(stderr, "\r* Processed read ends: %llu\n", (unsigned long long)(cnt[0] + cnt[1]));
    if (itx_sync_counts(ix, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "* Writing stats and Wig file\n");
    char *wig = fmt_alloc("%s.iteres.wig", prefix), *wigu = fmt_alloc("%s.iteres.unique.wig", prefix);
    char *f_sub = fmt_alloc("%s.iteres.subfamily.stat", prefix), *f_fam = fmt_alloc("%s.iteres.family.stat", prefix), *f_cla = fmt_alloc("%s.iteres.class.stat", prefix);
    LAP("counters on the host");
    if (itx_write_stat(ix, f_sub, wig, f_fam, f_cla, wigu, cnt[NIDX[norm]], cnt[NIDX2[norm2]]) != ITX_OK) die("Can't write the stat files for prefix %s", prefix);
    LAP("tables and wiggles written");
    fprintf(stderr, "* Generating bigWig files\n");
    {   /* the two conversions are independent: side by side */
        bw_job ja = {wig, rep_sizes, fmt_alloc("%s.iteres.bigWig", prefix), 0, {0}}, jb = {wigu, rep_sizes, fmt_alloc("%s.iteres.unique.bigWig", prefix), 0, {0}};
        pthread_t tb; const int threaded = pthread_create(&tb, NULL, bw_run, &jb) == 0;
        bw_run(&ja);
        if (threaded) pthread_join(tb, NULL); else bw_run(&jb);
        if (ja.rc != ITX_OK) die("%s", ja.err);
        if (jb.rc != ITX_OK) die("%s", jb.err);
    }
    LAP("bigWig files written");
    fprintf(stderr, "* Preparing report file\n");
    char *rep = fmt_alloc("%s.iteres.report", prefix);
    if (itx_write_report(rep, cnt, o.mapQ, "ALL") != ITX_OK) die("Can't open %s to write", rep);
    if (!keep_wig) { unlink(wig); unlink(wigu); }
    LAP("done");                          /* the process ends here: the index is not torn down piece by piece */
    done_in(t0);
    return 0;
}

static int main_filter(int argc, char **argv) {
    itx_scan_opts o; itx_scan_opts_default(&o); o.filter = 1; o.diffSubfam = 0;
    int c, sam = 0, readlist = 0, threshold = 1; unsigned int norm = 0; char *prefix = NULL, *name = NULL, *cls = NULL, *fam = NULL, *subfam;
    time_t t0 = time(NULL);
    while ((c = getopt(argc, argv, "SQ:g:N:n:c:t:f:rRTDCE:I:o:h?")) >= 0) {
        switch (c) {
            case 'S': sam = 1; break;
            case 'Q': o.mapQ = uarg(optarg); break;
            case 'g': o.minCoverage = (float)atof(optarg); break;
            case 'N': norm = uarg(optarg); break;
            case 't': threshold = (int)uarg(optarg); break;
            case 'r': readlist = 1; break;
            case 'R': o.rmDup = 1; break;
            case 'T': o.treat = 1; break;
            case 'D': o.discardWrongEnd = 1; break;
            case 'C': o.addChr = 1; break;
            case 'n': name = strdup(optarg); break;
            case 'c': cls = strdup(optarg); break;
            case 'f': fam = strdup(optarg); break;
            case 'E': o.extension = uarg(optarg); break;
            case 'I': o.iSize = uarg(optarg); break;
            case 'o': prefix = strdup(optarg); break;
            case 'h': case '?': return filter_usage();
            default: return 1;
        }
    }
    if (optind + 4 > argc) return filter_usage();
    const char *chrom_sizes = argv[optind], *rep_sizes = argv[optind + 1], *rmsk = argv[optind + 2], *bam = argv[optind + 3];
    int field = pick_filter(name, cls, fam, &subfam);
    static const int NIDX[4] = {7, 8, 6, 4};
    if (norm > 3) die("Wrong normalization method specified");
    if (!prefix) prefix = stem(bam);
    o.isSam = sam;
    o.readNames = readlist;
    use_device();
    char err[ITX_ERRLEN]; uint64_t cnt[13];
    itx_index *ix;
    const int ngpu = (readlist || sam || strchr(bam, ',')) ? 1 : n_gpus_wanted();
    if (ngpu != n_gpus_wanted()) fprintf(stderr, "* -r, -S and a file name with a comma in it keep filter on one GPU\n");
    fprintf(stderr, "* Start to parse the rmsk file\n");
    if (ngpu > 1) ix = run_on_gpus(ngpu, chrom_sizes, rep_sizes, rmsk, field, subfam, 0, 0, bam, &o, cnt);
    else {
        ix = itx_index_build(chrom_sizes, rep_sizes, rmsk, field, subfam, err);
        if (!ix) die("%s", err);
    }
    if (field) fprintf(stderr, "* Total %lld repeats for [%s].\n", (long long)itx_n_repeats_parsed(ix), subfam);
    else fprintf(stderr, "* Total %lld repeats found.\n", (long long)itx_n_repeats_parsed(ix));
    fprintf(stderr, "* Start to parse the SAM/BAM file\n");
    if (ngpu == 1 && itx_scan_alignment_file(ix, bam, &o, cnt, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "\r* Processed read ends: %llu\n", (unsigned long long)(cnt[0] + cnt[1]));
    if (itx_sync_counts(ix, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "* Preparing the output file\n");
    char *out = fmt_alloc("%s_%s.iteres.loci", prefix, subfam), *rep = fmt_alloc("%s_%s.iteres.reportloci", prefix, subfam);
    if (itx_write_filter(ix, out, readlist, threshold, cnt[NIDX[norm]]) != ITX_OK) die("Can't open %s to write", out);
    fprintf(stderr, "* Preparing report file\n");
    if (itx_write_report(rep, cnt, o.mapQ, subfam) != ITX_OK) die("Can't open %s to write", rep);
    itx_index_free(ix);
    done_in(t0);
    return 0;
}

static int main_cpgstat(int argc, char **argv) {
    int c, keep_wig = 0; char *prefix = NULL; time_t t0 = time(NULL);
    while ((c = getopt(argc, argv, "wo:h?")) >= 0) {
        switch (c) {
            case 'w': keep_wig = 1; break;
            case 'o': prefix = strdup(optarg); break;
            case 'h': case '?': return cpgstat_usage();
            default: return 1;
        }
    }
    if (optind + 4 > argc) return cpgstat_usage();
    const char *chrom_sizes = argv[optind], *rep_sizes = argv[optind + 1], *rmsk = argv[optind + 2], *bg = argv[optind + 3];
    if (!prefix) prefix = stem(bg);
    use_device();
    char err[ITX_ERRLEN]; uint32_t lines = 0, inrep = 0;
    fprintf(stderr, "* Start to parse the rmsk file\n");
    itx_index *ix;
    const int ngpu = n_gpus_wanted();
    if (ngpu > 1) {
        ix = run_on_gpus(ngpu, chrom_sizes, rep_sizes, rmsk, 0, "ALL", 1, 0, bg, NULL, NULL);
        uint64_t a = 0, b = 0; itx_get_cpg_totals(ix, &a, &b); lines = (uint32_t)a; inrep = (uint32_t)b;
    } else {
        ix = itx_index_build(chrom_sizes, rep_sizes, rmsk, 0, "ALL", err);
        if (!ix) die("%s", err);
    }
    fprintf(stderr, "* Total %lld repeats found.\n", (long long)itx_n_repeats_parsed(ix));
    fprintf(stderr, "* Start to parse the bedGraph file\n");
    if (ngpu == 1 && itx_scan_cpg(ix, bg, 0, &lines, &inrep, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "* Processed CpG sites: %u\n* CpG sites in Repeats: %u\n", lines, inrep);
    if (itx_sync_counts(ix, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "* Writing stats and Wig file\n");
    char *wig = fmt_alloc("%s.CpGstat.wig", prefix);
    if (itx_write_cpg_stat(ix, fmt_alloc("%s.CpG.subfamily.stat", prefix), wig, fmt_alloc("%s.CpG.family.stat", prefix), fmt_alloc("%s.CpG.class.stat", prefix)) != ITX_OK)
        die("Can't write the CpG stat files for prefix %s", prefix);
    fprintf(stderr, "* Generating bigWig files\n");
    if (itx_wig_to_bigwig(wig, rep_sizes, fmt_alloc("%s.CpGstat.bigWig", prefix), err) != ITX_OK) die("%s", err);
    if (!keep_wig) unlink(wig);
    itx_index_free(ix);
    done_in(t0);
    return 0;
}

static int main_cpgfilter(int argc, char **argv) {
    int c; double thr = 0; char *prefix = NULL, *name = NULL, *cls = NULL, *fam = NULL, *subfam; time_t t0 = time(NULL);
    while ((c = getopt(argc, argv, "n:c:f:t:o:h?")) >= 0) {
        switch (c) {
            case 'n': name = strdup(optarg); break;
            case 'c': cls = strdup(optarg); break;
            case 'f': fam = strdup(optarg); break;
            case 't': thr = strtod(optarg, NULL); break;
            case 'o': prefix = strdup(optarg); break;
            case 'h': case '?': return cpgfilter_usage();
            default: return 1;
        }
    }
    if (optind + 4 > argc) return cpgfilter_usage();
    const char *chrom_sizes = argv[optind], *rep_sizes = argv[optind + 1], *rmsk = argv[optind + 2], *bg = argv[optind + 3];
    if (!prefix) prefix = stem(bg);
    int field = pick_filter(name, cls, fam, &subfam);
    use_device();
    char err[ITX_ERRLEN]; uint32_t lines = 0, inrep = 0;
    fprintf(stderr, "* Start to parse the rmsk file\n");
    itx_index *ix;
    const int ngpu = n_gpus_wanted();
    if (ngpu > 1) {
        ix = run_on_gpus(ngpu, chrom_sizes, rep_sizes, rmsk, field, subfam, 1, 1, bg, NULL, NULL);
        uint64_t a = 0, b = 0; itx_get_cpg_totals(ix, &a, &b); lines = (uint32_t)a; inrep = (uint32_t)b;
    } else {
        ix = itx_index_build(chrom_sizes, rep_sizes, rmsk, field, subfam, err);
        if (!ix) die("%s", err);
    }
    if (field) fprintf(stderr, "* Total %lld repeats for [%s].\n", (long long)itx_n_repeats_parsed(ix), subfam);
    else fprintf(stderr, "* Total %lld repeats found.\n", (long long)itx_n_repeats_parsed(ix));
    fprintf(stderr, "* Start to parse the bedGraph file\n");
    if (ngpu == 1 && itx_scan_cpg(ix, bg, 1, &lines, &inrep, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "* Processed CpG sites: %u\n* CpG sites in Repeats: %u\n", lines, inrep);
    if (itx_sync_counts(ix, err) != ITX_OK) die("%s", err);
    fprintf(stderr, "* Preparing the output file\n");
    char *out = fmt_alloc("%s_%s.CpG.loci", prefix, subfam);
    if (itx_write_cpg_filter(ix, out, thr) != ITX_OK) die("Can't open %s to write", out);
    itx_index_free(ix);
    done_in(t0);
    return 0;
}

static int usage(void) {
    fprintf(stderr, "\nProgram: iteres (repeat analysis utils from Wang lab; B200 build: %s)\nVersion: %s\n\n", itx_version(), REF_VERSION);
    fprintf(stderr, "Usage:   iteres <command> [options]\n\n");
    fprintf(stderr, "Command: stat        get repeat alignment statistics\n");
    fprintf(stderr, "         filter      filter alignment statistic on repName/repFamily/repClass\n");
    fprintf(stderr, "         cpgstat     generate CpG density from MRE-Seq data for repeats\n");
    fprintf(stderr, "         cpgfilter   filter CpG statistic on repName/repFamily/repClass\n");
    fprintf(stderr, "         subfamStat  alias of stat;  nameStat  alias of filter\n\n");
    return 1;
}

int main(int argc, char **argv) {
    if (argc < 2) return usage();
    const char *cmd = argv[1];
    if (!strcmp(cmd, "stat") || !strcmp(cmd, "subfamStat")) return main_stat(argc - 1, argv + 1);
    if (!strcmp(cmd, "filter") || !strcmp(cmd, "nameStat")) return main_filter(argc - 1, argv + 1);
    if (!strcmp(cmd, "cpgstat")) return main_cpgstat(argc - 1, argv + 1);
    if (!strcmp(cmd, "cpgfilter")) return main_cpgfilter(argc - 1, argv + 1);
    fprintf(stderr, "[iteres] unrecognized command '%s'\n", cmd);
    return 1;
}
