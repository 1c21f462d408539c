/* itx_internal.h -- structures shared by the host C code (itx_host.c, itx_bgzf.c) and the CUDA
 * translation unit (itx_gpu.cu).  Not part of the public ABI. */
#ifndef ITX_INTERNAL_H
#define ITX_INTERNAL_H
#include <stdint.h>
#include <stddef.h>
#include "../../include/iteres_gpu.h"
#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ name tables (host) */
typedef struct {
    char **names; int32_t n, cap;
    int32_t *slot; uint32_t nslot;       /* open addressing on an FNV hash: index+1, 0 = empty */
} itx_strtab;
void itx_strtab_init(itx_strtab *t);
void itx_strtab_free(itx_strtab *t);
int32_t itx_strtab_findn(const itx_strtab *t, const char *name, size_t len);
int32_t itx_strtab_find(const itx_strtab *t, const char *name);
int32_t itx_strtab_add(itx_strtab *t, const char *name);           /* appends; the newest shadows older ones on find */
int32_t itx_strtab_intern(itx_strtab *t, const char *name);        /* find or add */
/* output-row order of a Kent hash holding these names (cuskent/hash.c:41-53, 136-140, 374-410, 511-551) */
int32_t *itx_kent_order(const itx_strtab *t, int pow2_initial);
uint32_t itx_fnv1a(const char *s, size_t n);
/* n names as eight zero-padded little-endian words each (a name of 32 bytes and more: all ones, which no padded name equals); malloc'ed */
uint32_t *itx_names32(char *const *names, int32_t n);

/* ------------------------------------------------------------------ per-group counters (host copy) */
typedef struct {
    uint64_t genome_count, total_length;
    uint64_t read_count, read_count_unique;
    uint32_t cpg_count; double cpg_score;
    int32_t first_fam, first_cla;        /* name ids of the family / class strings of the FIRST rmsk row of this group */
} itx_group;

/* ------------------------------------------------------------------ interval table */
/* Per chromosome the elements are ordered by (start, row); pmax = running maximum of `end` inside the
 * chromosome; one 16-byte load per candidate.  `bucket` maps (chromosome, position >> ITX_BSH) to the
 * first element whose start is >= the bucket's first base, so a lower_bound only searches one bucket. */
typedef struct { int32_t start, end, pmax; uint32_t row; } itx_iv;
#define ITX_BSH 10
typedef struct { uint32_t cons_start, cons_end, row, sub; } itx_meta;     /* 16 B, one load */
typedef struct { int32_t fam, cla; } itx_meta2;
/* per chromosome: first element, first bucket, size -- one 16-byte load per query */
typedef struct { uint32_t off, bucket; int32_t size; uint32_t n; } itx_chrominfo;
/* per subfamily: consensus length (0 = no coverage vector), offset of its difference array, case-folded name id */
typedef struct { uint32_t len; int32_t fold; unsigned long long bp_off; } itx_subinfo;

typedef struct {
    const itx_iv *iv; const itx_meta *meta; const itx_meta2 *meta2;
    const itx_iv *ivf;                   /* iv with the element's case-folded subfamily id in place of its row: all the walk of an XA:Z alternate needs, in one load */
    const itx_chrominfo *cinfo; const itx_subinfo *sinfo;
    const uint32_t *bucket; const long long *chrom_bucket;   /* bucket[chrom_bucket[c] + (pos >> ITX_BSH)], (size >> ITX_BSH) + 2 entries per chromosome */
    const long long *chrom_off;          /* n_chrom + 1 */
    const int32_t *chrom_size;           /* binKeeper maxPos (from the chrom size file) */
    int32_t n_chrom; long long n_elem;
    /* chromosome names for XA lookups: open addressing (FNV-1a) -> chrom id + 1; names NUL-terminated in a pool */
    const uint32_t *cname_slot; uint32_t cname_nslot; const uint32_t *cname_off; const char *cname_pool;
    const uint32_t *cname32;             /* the same names, eight zero-padded words each (all ones: a name of 32 bytes and more); NULL: not built */
    int32_t n_sub, n_fam, n_cla;
    int32_t stat_mode;                   /* 1 when the group tables exist (filter_field == 0) */
    const uint32_t *sub_len;             /* consensus length or 0 */
    const unsigned long long *sub_bp_off;/* offset of the subfamily's (len + 1)-entry difference array */
    const int32_t *sub_fold;             /* id of the case-folded name (sameWord equivalence classes) */
    /* counters: one packed block so that a single allreduce covers everything */
    unsigned long long *cnt;             /* [16] (13 used) */
    unsigned long long *grp;             /* [(n_sub + n_fam + n_cla) * 2]  (all, unique) interleaved */
    uint32_t *bp_diff, *bp_diff_u;       /* bp_len entries each */
    uint32_t *el_cnt, *el_cnt_u;         /* per element, sorted order (filter mode) */
    uint32_t *grp_cpg; double *grp_cpg_score; double *bp_cpg; uint32_t *el_cpg; double *el_cpg_score;
    uint32_t *tid_unknown_seen;          /* bitmap-ish: one word per BAM tid (first ITX_MAX_TID_SEEN tids) */
    uint32_t *status;                    /* [0] corrupt stream, [1] repaired chunk entries, [2] malformed XA, [3] hit-list overflow */
} itx_dev_index;
#define ITX_MAX_TID_SEEN 65536

typedef struct {
    uint32_t cend;                       /* chromSize - 1 */
    int32_t  chrom;                      /* index into the rmsk chromosome table or -1 */
    uint32_t flags;
    int32_t  csid;                       /* index of the (renamed) chromosome in the chrom-size table: the identity -R keys on, stable across files */
} itx_tidinfo;
#define ITX_TID_UNKNOWN 1u               /* not in the chrom size file: warn once, discard (generic.c:796-801) */
#define ITX_TID_GLSKIP  2u               /* -C and the name starts with GL (generic.c:783) */

struct itx_bam_header {
    uint64_t hdr_len; int32_t n_ref;
    char **names; uint32_t *lens;
    itx_tidinfo *tid;                    /* host */
    itx_tidinfo *d_tid;                  /* device copy */
    int addChr;
};

/* decode tuple: 16 bytes per BAM record, file order inside a chunk */
typedef struct { uint32_t start, end, info, rec_off; } itx_tuple;
#define ITX_F_DUP     (1u << 23)         /* -R: an earlier read has the same chr:start:end:strand key (set by k_dedup) */
#define ITX_F_FRAG    (1u << 24)
#define ITX_F_UNIQ    (1u << 25)
#define ITX_F_MINUS   (1u << 26)
#define ITX_F_HASXA   (1u << 27)
#define ITX_F_SLOT2   (1u << 28)
#define ITX_F_MAPPED  (1u << 29)
#define ITX_F_USED    (1u << 30)
#define ITX_F_UNKNOWN (1u << 31)
#define ITX_CHROM_MASK 0x007fffffu
#define ITX_CHROM_NONE 0x007fffffu

#define ITX_OFF_GUESS 0xfffffffffffffffdULL  /* carry of a scan that starts in the middle of a stream: the first record start is guessed like any span's */
#define ITX_OFF_END  0xfffffffffffffffeULL   /* the record chain ended here (truncated / corrupt record) */
#define ITX_OFF_NONE 0xffffffffffffffffULL   /* speculation found no plausible record start */

typedef struct {
    uint32_t mapQ, iSize, extension; float minCoverage;
    int32_t filter, discardWrongEnd, treat, diffSubfam;
} itx_dev_opts;

/* ------------------------------------------------------------------ the index */
typedef struct itx_cuda itx_cuda;        /* device buffers, stream, events (itx_gpu.cu) */

struct itx_index {
    int device, filter_field, stat_mode;
    itx_strtab chromsize; int *chromsize_val;
    itx_strtab repsize; int *repsize_val;
    itx_strtab chroms; int32_t *chrom_size; long long *chrom_off;       /* rmsk chromosomes, first-seen order */
    itx_strtab subs, fams, clas;                                         /* names (always interned, for printing) */
    itx_group *sub, *fam, *cla;                                          /* counters (stat_mode only) */
    uint32_t *sub_len; unsigned long long *sub_bp_off; int32_t *sub_fold; uint64_t bp_len;
    long long n_elem, n_rows;
    long long n_kept;                    /* rows that passed the -n/-c/-f filter, before rows on chromosomes missing from the size file were dropped (repeat_num, generic.c:1593) */
    itx_iv *iv; itx_meta *meta; itx_meta2 *meta2; int32_t *el_chrom;   /* sorted order */
    itx_iv *ivf;                         /* iv with sub_fold[meta.sub] in place of the row (mapped2diffSubfam's walks) */
    uint32_t *bucket; long long *chrom_bucket; long long n_bucket;
    itx_chrominfo *cinfo; itx_subinfo *sinfo;
    long long *row2el;                   /* rmsk row -> sorted element index or -1 */
    /* host mirrors of the device results (filled by itx_sync_counts) */
    uint64_t cnt[13];
    uint64_t cpg_lines, cpg_in_repeat;   /* totals of the CpG scans since the last reset (summed over the ranks by itx_comm_allreduce_counts) */
    uint32_t *bp, *bp_u;                 /* prefix-summed coverage, bp_len entries (entry len of each group unused) */
    double *bp_cpg;
    uint32_t *el_cnt, *el_cnt_u, *el_cpg; double *el_cpg_score;
    uint32_t *row_cnt, *row_cnt_u;       /* by rmsk row (filled on demand) */
    int32_t *sub_order, *fam_order, *cla_order;
    /* read names per element for filter -r (host, file order) */
    char ***el_names; uint32_t *el_names_n, *el_names_cap;
    itx_cuda *cu;
    itx_profile prof;
    uint32_t tune_chunk; uint64_t tune_window; int32_t tune_threads;
    uint64_t trace_cap;
    /* tids already warned about (the reference's nochr hash persists across files) */
    itx_strtab warned;
};

/* host side (itx_host.c) */
int itx_host_index_load(struct itx_index *ix, const char *chrom_sizes, const char *rep_sizes, const char *rmsk,
                        int filter_field, const char *filter_name, char err[ITX_ERRLEN]);
void itx_host_index_free(struct itx_index *ix);
int itx_host_parse_bam_header(struct itx_index *ix, const uint8_t *bam, uint64_t len, int addChr,
                              struct itx_bam_header *h, char err[ITX_ERRLEN]);

/* SAM text -> uncompressed BAM stream (itx_sam.c); the caller frees *out_bam */
int itx_sam_to_bam_stream(const char *path, uint8_t **out_bam, uint64_t *out_len, char err[ITX_ERRLEN]);

/* bigWig (itx_bigwig.c) */
int itx_bigwig_from_wig(const char *wig_path, long (*chrom_size)(void *ctx, const char *name), void *ctx, const char *out_path, char err[ITX_ERRLEN]);

/* BGZF (itx_bgzf.c) */
typedef struct { uint64_t coff; uint32_t csize, isize; uint64_t uoff; } itx_bgzf_block;
int itx_bgzf_scan(const uint8_t *file, uint64_t len, itx_bgzf_block **blocks, uint64_t *n_blocks, uint64_t *total_u,
                  char err[ITX_ERRLEN]);
/* inflate blocks [b0,b1) into dst + (uoff - uoff[b0]) with nth threads; returns 0 or ITX_EFORMAT */
int itx_parallel_copy(const uint8_t *file, uint64_t o0, uint64_t o1, uint8_t *dst, int nth);
int itx_parallel_pread(int fd, uint64_t o0, uint64_t o1, uint8_t *dst, int nth);
int itx_bgzf_header_ok(const uint8_t *h18);
int64_t itx_bgzf_find_block(const uint8_t *buf, uint64_t n, int at_eof);
int itx_bgzf_inflate_range(const uint8_t *file, const itx_bgzf_block *blocks, uint64_t b0, uint64_t b1,
                           uint8_t *dst, int nth, double *busy_ms);

#ifdef __cplusplus
}
#endif
#endif
