/* iteres_gpu.h -- C-ABI of libiteres_gpu.so: the B200 (sm_100a) replacement for the iteres hot path.
 *
 * The reference (lidaof/iteres v0.3.3-r123) has no plugin / FFI layer; its drivers (stat.c, filter.c,
 * cpgstat.c, cpgfilter.c) call a handful of C functions in generic.c directly.  Those calls are the
 * drop-in boundary.  Every entry point below names the reference function it replaces (file:line in
 * the reference tree).  Plain pointers and sizes only; no C++ or torch types; errors are returned as
 * a status plus a message (the thin CLI turns status != 0 into the reference's "message on stderr,
 * exit(-1)" behaviour, cuskent/errabort.c:166-181).
 *
 * There is NO CPU fallback: every scan runs on the CUDA device and fails with ITX_ENODEV when none is
 * usable.  The host side only parses text tables, inflates BGZF blocks into pinned buffers and prints
 * the output tables.
 */
#ifndef ITERES_GPU_H
#define ITERES_GPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ITX_ERRLEN 256
#define ITX_OK 0
#define ITX_EIO (-1)       /* file could not be opened / read */
#define ITX_EFORMAT (-2)   /* malformed input (the reference would errAbort) */
#define ITX_ENODEV (-3)    /* no usable CUDA device / CUDA runtime error */
#define ITX_EARG (-4)
#define ITX_ENOMEM (-5)
#define ITX_ENOTSUP (-6)   /* option of the reference that this build does not run on the device yet */

typedef struct itx_index itx_index;

/* The scalar arguments of samFiles2nodupRepbedFileNew / samFile2nodupRepbedFileNew
 * (generic.h:72-73; generic.c:700 and 343), same meaning, same defaults as stat.c:32-44 / filter.c:32-44. */
typedef struct itx_scan_opts {
    uint32_t mapQ;             /* -Q  (10)   unique <=> MAPQ >= mapQ                     generic.c:817 */
    int32_t  filter;           /* 0: stat (subfamily/family/class counters)  1: filter (per-locus counters) */
    int32_t  rmDup;            /* -R  (0)    first read of a chr:start:end:strand key wins, in file order   generic.c:907-919 */
    int32_t  addChr;           /* -C  (0)    GL* skipped, MT->chrM, chr prefix           generic.c:781-791 */
    int32_t  discardWrongEnd;  /* -D  (0)                                                generic.c:862 */
    uint32_t iSize;            /* -I  (500)                                              generic.c:839 */
    uint32_t extension;        /* -E  (150)                                              generic.c:825-833 */
    float    minCoverage;      /* -c  (1e-4f)                                            generic.c:961 */
    int32_t  treat;            /* -T  (0)                                                generic.c:815 */
    int32_t  diffSubfam;       /* !-x (1 for stat, 0 for filter)                         generic.c:972 */
    /* order-dependent side outputs, written by a host pass over the device's per-record verdicts in file order */
    int32_t  readNames;        /* filter -r: keep the read names of every counted read per locus   generic.c:662-666 */
    int32_t  isSam;            /* -S: the files are SAM text (plain or gzip), converted on the host    sam.c:39-65, bam_import.c:237-456 */
    const char *outbed;        /* -B: bed line per fragment that survives -R (NULL: none)           generic.c:925-931 */
    const char *outbed_unique; /* -V: the same for unique reads only                                generic.c:932-936 */
} itx_scan_opts;
void itx_scan_opts_default(itx_scan_opts *o);

/* ---- device selection / library info ---- */
int  itx_device_count(void);
int  itx_set_device(int device);            /* CUDA device used by indexes built afterwards (default 0) */
const char *itx_version(void);

/* ---- index: replaces hashNameIntFile x2 (stat.c:137-138 -> cuskent/obscure.c:139-150) and
 *      rmsk2binKeeperHash (generic.h:76; generic.c:1578-1707).  filter_field 0 / 10 / 11 / 12 and
 *      filter_name as filter.c:93-113.  Returns NULL and fills err on failure. ---- */
itx_index *itx_index_build(const char *chrom_sizes, const char *rep_sizes, const char *rmsk,
                           int filter_field, const char *filter_name, char err[ITX_ERRLEN]);
void itx_index_free(itx_index *ix);
void itx_index_reset_counts(itx_index *ix);  /* zero every counter on the device (a new run on the same index) */

/* ---- alignment scan: replaces samFiles2nodupRepbedFileNew (generic.c:700-1062) and the single-file
 *      twin samFile2nodupRepbedFileNew (generic.c:343-697).  bam_list is the reference's comma
 *      separated list of BGZF .bam paths.  Counters persist across files and calls until
 *      itx_index_reset_counts.  cnt[13] as generic.c:1048-1060. ---- */
int itx_scan_alignments(itx_index *ix, const char *bam_list, const itx_scan_opts *o,
                        uint64_t cnt[13], char err[ITX_ERRLEN]);
/* the single-file twin samFile2nodupRepbedFileNew (generic.h:73; generic.c:343-697), what `iteres filter` calls: `path` is ONE
 * file name and is not split at commas */
int itx_scan_alignment_file(itx_index *ix, const char *path, const itx_scan_opts *o,
                            uint64_t cnt[13], char err[ITX_ERRLEN]);
/* same path, the BGZF file image already in host memory */
int itx_scan_bgzf_memory(itx_index *ix, const uint8_t *bgzf, uint64_t len, const itx_scan_opts *o,
                         uint64_t cnt[13], char err[ITX_ERRLEN]);
/* same path after inflate: an UNCOMPRESSED BAM byte stream (magic, header, records) in HOST memory;
 * staged to the device through pinned buffers inside the call */
int itx_scan_bam_host(itx_index *ix, const uint8_t *bam, uint64_t len, const itx_scan_opts *o,
                      uint64_t cnt[13], char err[ITX_ERRLEN]);
/* device-resident variant used to time the kernels alone: d_bam is a CUDA device pointer to the
 * uncompressed stream (at least len + 64 bytes allocated), hdr_len/n_ref/tid tables come from
 * itx_bam_header_parse on the host copy of the first bytes. */
typedef struct itx_bam_header itx_bam_header;
itx_bam_header *itx_bam_header_parse(itx_index *ix, const uint8_t *bam, uint64_t len, int addChr, char err[ITX_ERRLEN]);
uint64_t itx_bam_header_len(const itx_bam_header *h);
void itx_bam_header_free(itx_bam_header *h);
int itx_scan_bam_device(itx_index *ix, const itx_bam_header *h, const void *d_bam, uint64_t len,
                        const itx_scan_opts *o, uint64_t cnt[13], char err[ITX_ERRLEN]);

/* ---- CpG scan: replaces cpgBedGraphOverlapRepeat (generic.h:81; generic.c:1064-1139) ---- */
int itx_scan_cpg(itx_index *ix, const char *bedgraph, int filter, uint32_t *n_lines, uint32_t *n_in_repeat,
                 char err[ITX_ERRLEN]);

/* ---- results back on the host (after a scan; copies the device counters once) ---- */
int itx_sync_counts(itx_index *ix, char err[ITX_ERRLEN]);

/* ---- writers: byte-identical tables.
 *      itx_write_stat       = writeWigandStat      (generic.h:67; generic.c:72-113)
 *      itx_write_report     = writeReport          (generic.h:65; generic.c:53-70)
 *      itx_write_filter     = writeFilterOut       (generic.h:77; generic.c:1709-1746)
 *      itx_write_cpg_stat   = MREwriteWigandStat   (generic.h:68; generic.c:115-152)
 *      itx_write_cpg_filter = writeFilterOutMRE    (generic.h:82; generic.c:1748-1771) ---- */
int itx_write_stat(itx_index *ix, const char *subfam_stat, const char *wig, const char *fam_stat,
                   const char *class_stat, const char *wig_unique, uint64_t reads_num, uint64_t reads_num_unique);
int itx_write_report(const char *path, const uint64_t cnt[13], uint32_t mapQ, const char *subfam);
int itx_write_filter(itx_index *ix, const char *path, int readlist, int threshold, uint64_t reads_num);
int itx_write_cpg_stat(itx_index *ix, const char *subfam_stat, const char *wig, const char *fam_stat, const char *class_stat);
int itx_write_cpg_filter(itx_index *ix, const char *path, double score_threshold);
/* wiggle -> bigWig = bigWigFileCreate(wig, rep_size_file, 256, 1024, 0, 1, bigWig) (stat.c:157-158, cpgstat.c:75;
 * cuskent/bwgCreate.c:1088-1112): byte-identical files for the fixedStep wiggles itx_write_stat / itx_write_cpg_stat
 * make.  Host only.  An empty wiggle is an error ("... is empty of data"), as in the reference. */
int itx_wig_to_bigwig(const char *wig, const char *chrom_sizes, const char *bigwig, char err[ITX_ERRLEN]);
/* the SAM text front end on its own (what a scan with isSam does first): SAM (plain or gzip) -> the uncompressed BAM
 * stream samtools 0.1.18 would have built record by record (bam_import.c:237-456).  *bam is released with itx_free. */
int itx_sam_to_bam(const char *sam, uint8_t **bam, uint64_t *len, char err[ITX_ERRLEN]);
void itx_free(void *p);

/* ---- plain accessors (tests, bindings).  which: 0 subfamily, 1 family, 2 class; i in output-row
 *      order (the reference's hash iteration order, cuskent/hash.c:511-551). ---- */
int32_t itx_n_subfam(const itx_index *ix);
int32_t itx_n_fam(const itx_index *ix);
int32_t itx_n_class(const itx_index *ix);
int64_t itx_n_elem(const itx_index *ix);
/* repeat_num of rmsk2binKeeperHash (generic.c:1593, 1697-1701): rows that passed the -n/-c/-f filter, counted BEFORE the rows on
 * chromosomes missing from the size file are dropped -- the number the reference prints in "* Total N repeats found." */
int64_t itx_n_repeats_parsed(const itx_index *ix);
int32_t itx_n_chrom(const itx_index *ix);
const char *itx_name(const itx_index *ix, int which, int32_t i);
void itx_counts(const itx_index *ix, int which, int32_t i, uint64_t out[4] /* read_count, unique, total_length, genome_count */);
uint32_t itx_subfam_length(const itx_index *ix, int32_t i);
const uint32_t *itx_subfam_bp(const itx_index *ix, int32_t i, int unique);
/* per-locus counters of filter mode, indexed by rmsk row (0-based among parsed rows); n = itx_n_rows */
int64_t itx_n_rows(const itx_index *ix);
const uint32_t *itx_elem_counts_by_row(itx_index *ix, int unique);

/* ---- per-record trace of the last scan (tests: checks decode and overlap separately).  Enabled with
 *      itx_trace_enable(ix, cap) before the scan; entries in file order. ---- */
#define ITX_T_FRAGMENT 1u
#define ITX_T_UNIQ     2u
#define ITX_T_MINUS    4u
#define ITX_T_HAS_XA   8u
#define ITX_T_DIFFSUB  16u
#define ITX_T_COUNTED  32u
#define ITX_T_DUP      64u   /* -R: dropped as a duplicate (generic.c:907-919) */
typedef struct itx_trace { uint32_t start, end; int32_t tid; int32_t sel_row; uint32_t flags; } itx_trace;
int itx_trace_enable(itx_index *ix, uint64_t cap);
uint64_t itx_trace_fetch(itx_index *ix, itx_trace *out, uint64_t cap);

/* single query against the device index: the overlap + "last ascent" selection of generic.c:945-970.
 * chrom by name; returns selected rmsk row or -1 per query.  (property tests of the overlap kernel) */
int itx_query_select(itx_index *ix, const char *chrom, const uint32_t *start, const uint32_t *end, int64_t n,
                     float min_cov, int32_t *sel_row, int32_t *n_hits, char err[ITX_ERRLEN]);

/* ---- measurement: device time of the kernels of the last scan (CUDA events on the scan stream) ---- */
typedef struct itx_profile {
    double decode_ms;      /* record-boundary + decode kernel (+ chain verification) */
    double overlap_ms;     /* overlap / selection / accumulation kernel */
    double finalize_ms;    /* coverage prefix sums */
    double total_ms;       /* first launch to last launch of the scan, on the device */
    double h2d_ms;         /* host->device copies (streaming paths) */
    double inflate_ms;     /* wall time the host inflate threads were busy (max over threads) */
    uint64_t n_records, n_fragments, stream_bytes, h2d_bytes, d2h_bytes;
    uint64_t n_launches;   /* kernels launched by the scan */
    uint64_t n_bad_chunks; /* speculated chunk entries that the chain check had to repair */
    int32_t inflate_threads;
    int32_t fused;         /* 1: the launch groups ran as one k_scan each (its time is decode_ms; overlap_ms is 0) */
    uint64_t n_replayed_windows;   /* launch groups counted again through the tuple path after a failed chain check */
    double cpg_kernel_ms;          /* itx_scan_cpg: device time of the k_bedgraph launches (sum) */
    /* itx_scan_alignments_shard with -R, summed over the files: wall time of phase 1 (the parts settled, their keys collected), of
     * the exchange (all-gathers, key export, broadcasts) and of phase 2 (admissions and the counting scan); bytes of keys every
     * rank holds after the broadcasts (16 per unique fragment of the files) */
    double rmdup_keys_ms, rmdup_exchange_ms, rmdup_count_ms;
    uint64_t rmdup_bcast_bytes;
} itx_profile;
void itx_last_profile(const itx_index *ix, itx_profile *p);
/* device-side stopwatch on the scan stream: itx_mark records CUDA event `slot` (0..7) after everything
 * enqueued so far; itx_elapsed_ms synchronises on both events and returns the time between them */
int itx_mark(itx_index *ix, int slot);
double itx_elapsed_ms(itx_index *ix, int slot_from, int slot_to);
/* knobs (0 keeps the default): chunk bytes per decode thread, window bytes per launch group, host inflate threads */
int itx_tune(itx_index *ix, uint32_t chunk_bytes, uint64_t window_bytes, int32_t inflate_threads);

/* ---- multi-GPU: one rank per GPU; every rank scans its own shard, then ONE allreduce(sum) of the
 *      packed integer counter block (u64 counts, u32 wrapping coverage difference arrays).  The NCCL
 *      unique id is created by rank 0 and handed to the other ranks by the caller. ---- */
#define ITX_NCCL_ID_BYTES 128
int itx_comm_unique_id(uint8_t id[ITX_NCCL_ID_BYTES], char err[ITX_ERRLEN]);
int itx_comm_init(itx_index *ix, const uint8_t id[ITX_NCCL_ID_BYTES], int rank, int nranks, char err[ITX_ERRLEN]);
int itx_comm_allreduce_counts(itx_index *ix, char err[ITX_ERRLEN]);   /* afterwards itx_get_counters returns the global sums */
void itx_get_counters(const itx_index *ix, uint64_t cnt[13]);
void itx_comm_destroy(itx_index *ix);

/* ---- ONE BAM file across the ranks (SURVEY.md 8(e): "split the BAM into G contiguous ranges of BGZF blocks"; the reference reads
 *      its files in one loop, generic.c:700-745, block by block, cussamtools/bgzf.c:471-521).  Rank r owns the BGZF blocks that
 *      START in the r-th share of the file's bytes and the records that start in those blocks; it guesses its first record start
 *      out of the bytes (no .bai needed) and reads past its last block until the straddling record is whole.  The ranks then
 *      compare notes: a rank whose guess is not where the chain of the ranks before it arrives scans its part again from the
 *      right place, so the counts are those of one pass over the file, bit for bit.  -R runs in two phases with an exchange of
 *      duplicate keys between them (below); -B/-V and filter -r (file-order outputs) and SAM text are not sharded (ITX_ENOTSUP). ---- */
#define ITX_SHARD_GUESS 0xfffffffffffffffdULL
#define ITX_SHARD_END   0xfffffffffffffffeULL   /* the record chain ended (a cut record): nothing after it counts */
#define ITX_SHARD_NONE  0xffffffffffffffffULL   /* no record start */
typedef struct itx_shard_report {
    uint64_t entry_rel;        /* first record start the rank settled on, as an offset into its own uncompressed bytes */
    uint64_t exit_rel;         /* where the chain left the part, as an offset into the NEXT rank's bytes */
    uint64_t own_bytes;        /* uncompressed size of the rank's own blocks */
} itx_shard_report;
/* one rank, one file; entry = ITX_SHARD_GUESS or what itx_shard_chain_check handed back */
int itx_scan_shard_file(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                        itx_shard_report *rep, uint64_t cnt[13], char err[ITX_ERRLEN]);
/* the reports of all ranks -> first rank that must scan again (and from where), or -1.  Pure host arithmetic. */
int itx_shard_chain_check(int nranks, const itx_shard_report *rep, uint64_t *forced_entry);
/* -R across ranks, step by step (what itx_scan_alignments_shard does with NCCL, for callers that move the keys themselves).
 * File order is (file, rank, place in the rank's part).  Per file, every rank:
 *   1. itx_shard_dedup_keys: the scan of itx_scan_shard_file (same entry guess, margin retry; repeated from the entry
 *      itx_shard_chain_check forces), counting nothing: it collects the keys of the part's unique fragments.  flags bit 0: the part
 *      has a unique fragment, bit 1: some other fragment.  A part with no record start or a cut chain has neither.
 *   2. itx_shard_dedup_fetch: the keys (16 bytes each, in no particular order) into dst, at most cap of them; returns how many.
 *   3. itx_dedup_admit with the keys and OR-ed flags of the parts of ranks < rank, itx_scan_shard_file_rmdup from the settled entry
 *      (the part phase 1 left on the device, counted with -R), itx_dedup_admit with those of ranks > rank.
 * Keys and flags persist across the files of a run, as in a single scan. */
int itx_shard_dedup_keys(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                         itx_shard_report *rep, uint64_t *n_keys, uint32_t *flags, char err[ITX_ERRLEN]);
uint64_t itx_shard_dedup_fetch(itx_index *ix, void *dst, uint64_t cap);
int itx_dedup_admit(itx_index *ix, const void *keys, uint64_t n, uint32_t flags, char err[ITX_ERRLEN]);
int itx_scan_shard_file_rmdup(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                              itx_shard_report *rep, uint64_t cnt[13], char err[ITX_ERRLEN]);
/* the whole protocol for a comma separated list of files, rank and size taken from itx_comm_init: scan, all-gather the
 * reports (NCCL), scan again where the check says so; with -R the keys are exchanged (ncclBroadcast) and each part is counted
 * as in 3. above.  Afterwards every rank holds the counts of ITS parts; itx_comm_allreduce_counts makes them the job's. */
int itx_scan_alignments_shard(itx_index *ix, const char *bam_list, const itx_scan_opts *o, uint64_t cnt[13], char err[ITX_ERRLEN]);
/* cpgBedGraphOverlapRepeat over the rank-th of nranks parts of the bedGraph (cut at line ends); the u32 counts and f64 score
 * sums are merged by itx_comm_allreduce_counts (1e-9 relative on the sums), the line totals by itx_get_cpg_totals after it */
int itx_scan_cpg_shard(itx_index *ix, const char *bedgraph, int filter, int rank, int nranks, uint32_t *n_lines, uint32_t *n_in_repeat,
                       char err[ITX_ERRLEN]);
void itx_get_cpg_totals(const itx_index *ix, uint64_t *n_lines, uint64_t *n_in_repeat);
int itx_comm_rank(const itx_index *ix, int *rank, int *nranks);
/* like itx_set_device + itx_index_build in one call (several indexes, one per device, can be built from threads of one process) */
itx_index *itx_index_build_on(int device, const char *chrom_sizes, const char *rep_sizes, const char *rmsk,
                              int filter_field, const char *filter_name, char err[ITX_ERRLEN]);

/* ---- raw device helpers for benchmarks (so a harness needs no other CUDA binding) ---- */
void *itx_dev_alloc(uint64_t bytes);
void itx_dev_free(void *p);
int itx_dev_upload(void *dst, const void *src, uint64_t bytes);
void *itx_host_alloc_pinned(uint64_t bytes);
void itx_host_free_pinned(void *p);
int itx_dev_flush_l2(itx_index *ix);           /* writes a 256 MiB scratch buffer */
/* test hook: the uncompressed BAM stream the last host/BGZF scan left on the device (what the device inflate produced); returns the bytes copied */
uint64_t itx_stream_fetch(itx_index *ix, uint8_t *out, uint64_t cap);
int itx_dev_sync(void);

#ifdef __cplusplus
}
#endif
#endif
