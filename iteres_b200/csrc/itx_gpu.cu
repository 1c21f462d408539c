/* itx_gpu.cu -- device side of libiteres_gpu.so: index upload, the scan pipelines (device-resident
 * stream, host stream through pinned staging, BGZF file through host inflate threads), result
 * download, NCCL allreduce of the counter block.  Built for sm_100a only. */
#include "itx_kernels.cuh"
#include "itx_ordered.h"
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <errno.h>
#include <time.h>
#include <unistd.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <vector>

#define ITX_SLACK 64
#define ITX_MAX_EVENTS 4096
#define ITX_SEEN_FAST 1024                 /* unknown-tid marks fetched with the end-of-scan report (BAM headers with more references take one more copy) */
#define ITX_SCRATCH_BYTES (256 + ITX_SEEN_FAST * 4)
#define ITX_MAX_WINDOWS 65536              /* launch groups of one scan that k_scan can log (more: the tuple path takes over) */
#define ITX_INF_LANES_DEFAULT 16           /* blocks per k_inflate warp (ITX_INF_LANES), and for the last groups of a file (ITX_INF_TAIL_LANES) */
#define ITX_INF_TAIL_LANES_DEFAULT 8
#define ITX_INF_STREAMS 8                  /* inflate groups in flight: copy, Huffman pass, match pass and scan of different groups overlap */

/* a -R key table (k_dedup): keys, smallest ordinal per key, mins[3] (itx_dedup_args) */
struct dup_table { itx_k128 *keys; unsigned long long *ords, *mins; uint64_t cap; };
struct itx_cuda {
    int device; cudaStream_t stream, copy_stream;
    int sm_count; size_t smem_optin;
    /* index */
    itx_dev_index D;
    void *d_iv, *d_ivf, *d_bucket, *d_chrom_bucket, *d_cinfo, *d_sinfo, *d_meta, *d_meta2, *d_chrom_off, *d_chrom_size, *d_cname_slot, *d_cname_off, *d_cname_pool, *d_cname32;
    void *d_sub_len, *d_sub_bp_off, *d_sub_fold;
    /* counter block */
    void *d_u64; size_t n_u64;           /* cnt[16] + grp */
    void *d_u32; size_t n_u32;           /* bp_diff, bp_diff_u, el_cnt, el_cnt_u */
    void *d_cpg_u32; size_t n_cpg_u32;   /* grp_cpg, el_cpg */
    void *d_cpg_f64; size_t n_cpg_f64;   /* grp_cpg_score, bp_cpg, el_cpg_score */
    void *d_misc;                        /* tid_unknown_seen[ITX_MAX_TID_SEEN] + status[8] */
    void *d_D;                           /* D itself in global memory, for the out-of-line device functions (the kernels read their by-value copy) */
    uint32_t *d_bp, *d_bp_u;             /* prefix-summed coverage (finalize output) */
    /* scan workspace */
    uint32_t C, S; uint64_t cap_chunks;                      /* spans the tuple buffers hold (one launch group of the tuple path) */
    uint64_t cap_log;                                         /* spans the entry / exit logs hold (one launch group of k_scan, >= cap_chunks) */
    itx_tuple *d_tuples; unsigned long long *d_entry, *d_exit, *d_carry, *d_rec_base, *d_running; uint32_t *d_nrec, *d_winbad;
    long long *d_sel; int want_sel;
    unsigned long long *h_scratch;                            /* pinned: [0] the carry a scan uploads (no wait for the copy); from byte 64 the end-of-scan report:
                                                               * cnt[16] u64, status[8] u32, first bad launch group u32, then (byte 256) the first ITX_SEEN_FAST unknown-tid marks */
    unsigned long long *d_xa_q; uint64_t xa_cap; uint32_t *d_xa_n; int xa_attr;      /* k_scan -> k_xa: record offsets of the reads whose XA:Z alternates have to be looked at */
    unsigned long long *d_carry_log; uint32_t *d_fused;      /* k_scan: carry per window; [0] first bad window, [1] CTA ticket */
    int scan_ctas[4];                                         /* resident CTAs per SM of the k_scan instances */
    uint32_t *d_work; int decode_variant;   /* 0: k_decode_span (TMA staged stages, chain carried inside a span), 1: k_decode (thread per chunk) */
    int decode_ctas;                        /* resident CTAs per SM of k_decode_span */
    itx_trace *d_trace; uint64_t trace_cap;
    /* staging for host streams */
    uint8_t *d_stream; uint64_t d_stream_cap;
    uint8_t *d_comp; uint64_t d_comp_cap; itx_bgzf_block *d_blk; uint64_t d_blk_cap;   /* compressed file image + block table (device inflate) */
    uint16_t *d_tabs; uint64_t d_tabs_threads;   /* symbol arrays of k_inflate's long codes */
    uint32_t *d_mpl; uint16_t *d_md; uint32_t *d_mn; uint64_t d_m_slots;   /* match lists: ITX_INF_STREAMS groups in flight */
    dup_table dup; uint64_t dup_ord_base;            /* -R: key table, state persists across the files of a run */
    /* -R across ranks: the key table of this rank's part of the file (phase 1, itx_shard_dedup_keys), the dense key array exported
     * from it and exchanged between ranks, and what the counting scan (itx_scan_shard_file_rmdup) needs of the stream phase 1 left
     * on the device */
    dup_table part; itx_k128 *d_xkeys; uint64_t xkeys_cap; unsigned long long *d_xn;
    struct { itx_bam_header *h; char *path; int rank, nranks; uint64_t len, own, n_keys; uint32_t flags; itx_shard_report rep; } p1;
    /* order-dependent side outputs (-B / -V bed files, filter -r read names): host pass per launch group */
    FILE *bed_f, *bed_uf; int bed_owner;             /* opened by the outermost entry point of the run */
    uint64_t ord_cap;                                /* trace entries one launch group may need (0: not in ordered mode) */
    itx_trace *h_ord_trace; uint64_t h_ord_trace_cap; uint8_t *h_ord_buf; uint64_t h_ord_buf_cap;
    int l2_persist_on;
    int used_bp;                                     /* a stat-mode scan has run since the last reset (the coverage difference arrays may be non-zero) */
    void *d_snap; size_t snap_cap;                   /* counter snapshot of a sharded scan (counters_snapshot) */
    unsigned long long *d_shard;                     /* sharded scan: this rank's report + everybody's (NCCL all-gather) */
    int used_el, used_cpg, used_cpg_el, host_el, host_cpg, host_cpg_el;   /* per-locus / CpG counters touched on the device since the last reset; host copies not all zero */
    cudaStream_t inf_stream[ITX_INF_STREAMS]; cudaEvent_t inf_done[ITX_INF_STREAMS]; int inf_made;
    uint8_t *h_stage[2]; uint64_t h_stage_cap;
    uint8_t *h_ring[4]; uint64_t h_ring_cap;          /* pinned slots of the compressed-window reader (ITX_RD_SLOTS) */
    void *d_flush;
    cudaEvent_t ev[ITX_MAX_EVENTS]; int n_ev_made;
    cudaEvent_t marks[8]; int marks_made;
    cudaEvent_t grp_ev[64];                          /* one per inflate group in flight (the compressed ring's overwrite protection) */
    cudaEvent_t *inf_ev; int inf_ev_made;            /* ITX_TIMING / profile: launch and end of every inflate group (events of THIS device) */
    /* NCCL (dlopen) */
    void *nccl_lib; void *nccl_comm; int nranks, rank;
};

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(err, ITX_ERRLEN, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); return ITX_ENODEV; } } while (0)
#define CKN(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(err, ITX_ERRLEN, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); goto fail; } } while (0)

static int g_device = 0;
static int env_int_early(const char *name, int dflt) { const char *v = getenv(name); return v && *v ? atoi(v) : dflt; }
static double now_ms(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }

extern "C" int itx_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }
/* only noted here: the device is first touched by itx_index_build, where the driver start-up overlaps the table parse */
extern "C" int itx_set_device(int device) { if (device < 0) return ITX_EARG; g_device = device; return ITX_OK; }
static void *cuda_warm_up(void *arg) { if (cudaSetDevice((int)(intptr_t)arg) == cudaSuccess) cudaFree(0); return NULL; }
extern "C" void *itx_dev_alloc(uint64_t bytes) { void *p = NULL; cudaSetDevice(g_device); if (cudaMalloc(&p, bytes) != cudaSuccess) return NULL; return p; }
extern "C" void itx_dev_free(void *p) { cudaFree(p); }
extern "C" int itx_dev_upload(void *dst, const void *src, uint64_t bytes) { return cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess ? ITX_OK : ITX_ENODEV; }
extern "C" void *itx_host_alloc_pinned(uint64_t bytes) { void *p = NULL; cudaSetDevice(g_device); if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return NULL; return p; }
extern "C" void itx_host_free_pinned(void *p) { cudaFreeHost(p); }
extern "C" int itx_dev_sync(void) { return cudaDeviceSynchronize() == cudaSuccess ? ITX_OK : ITX_ENODEV; }

template <typename T> static int upload(void **dst, const T *src, size_t n, char *err) {
    size_t bytes = sizeof(T) * (n ? n : 1);
    CK(cudaMalloc(dst, bytes));
    if (n) CK(cudaMemcpy(*dst, src, sizeof(T) * n, cudaMemcpyHostToDevice));
    return ITX_OK;
}

static void cuda_free_all(itx_cuda *cu) {
    if (!cu) return;
    cudaSetDevice(cu->device);
    void *ptrs[] = {cu->d_iv, cu->d_ivf, cu->d_bucket, cu->d_chrom_bucket, cu->d_cinfo, cu->d_sinfo, cu->d_work, cu->d_meta, cu->d_meta2, cu->d_chrom_off, cu->d_chrom_size, cu->d_cname_slot, cu->d_cname_off,
                    cu->d_cname_pool, cu->d_cname32, cu->d_sub_len, cu->d_sub_bp_off, cu->d_sub_fold, cu->d_u64, cu->d_u32, cu->d_cpg_u32, cu->d_cpg_f64,
                    cu->d_misc, cu->d_D, cu->d_bp, cu->d_bp_u, cu->d_tuples, cu->d_entry, cu->d_exit, cu->d_carry, cu->d_rec_base, cu->d_running,
                    cu->d_nrec, cu->d_winbad, cu->d_sel, cu->d_trace, cu->d_stream, cu->d_flush, cu->d_comp, cu->d_blk, cu->d_tabs, cu->d_mpl, cu->d_md, cu->d_mn, cu->dup.keys, cu->dup.ords, cu->dup.mins,
                    cu->part.keys, cu->part.ords, cu->part.mins, cu->d_xkeys, cu->d_xn, cu->d_carry_log, cu->d_fused, cu->d_snap, cu->d_shard, cu->d_xa_q, cu->d_xa_n};
    for (size_t i = 0; i < sizeof(ptrs) / sizeof(ptrs[0]); i++) if (ptrs[i]) cudaFree(ptrs[i]);
    itx_bam_header_free(cu->p1.h); free(cu->p1.path);
    for (int i = 0; i < 2; i++) if (cu->h_stage[i]) cudaFreeHost(cu->h_stage[i]);
    for (int i = 0; i < 4; i++) if (cu->h_ring[i]) cudaFreeHost(cu->h_ring[i]);
    if (cu->h_scratch) cudaFreeHost(cu->h_scratch);
    for (int i = 0; i < cu->n_ev_made; i++) cudaEventDestroy(cu->ev[i]);
    if (cu->marks_made) for (int i = 0; i < 8; i++) cudaEventDestroy(cu->marks[i]);
    for (int i = 0; i < cu->inf_ev_made; i++) cudaEventDestroy(cu->inf_ev[i]);
    for (int i = 0; i < 64; i++) if (cu->grp_ev[i]) cudaEventDestroy(cu->grp_ev[i]);
    free(cu->inf_ev);
    if (cu->inf_made) for (int i = 0; i < ITX_INF_STREAMS; i++) { cudaStreamDestroy(cu->inf_stream[i]); cudaEventDestroy(cu->inf_done[i]); }
    if (cu->stream) cudaStreamDestroy(cu->stream);
    if (cu->copy_stream) cudaStreamDestroy(cu->copy_stream);
    free(cu);
}

extern "C" void itx_index_free(itx_index *ix) {
    if (!ix) return;
    itx_comm_destroy(ix);
    cuda_free_all(ix->cu);
    itx_host_index_free(ix);
    free(ix);
}

/* all = 0: only the blocks a scan has touched since they were last zeroed (the per-locus and CpG blocks are large and
 * most runs never write them) */
static int zero_counters(itx_index *ix, char *err, int all) {
    itx_cuda *cu = ix->cu;
    const size_t bp2 = 2 * (size_t)ix->bp_len;
    CK(cudaMemsetAsync(cu->d_u64, 0, cu->n_u64 * 8, cu->stream));
    CK(cudaMemsetAsync(cu->d_u32, 0, ((all || cu->used_el) ? cu->n_u32 : bp2) * 4, cu->stream));
    if (all || cu->used_cpg || cu->used_cpg_el) {
        CK(cudaMemsetAsync(cu->d_cpg_u32, 0, cu->n_cpg_u32 * 4, cu->stream));
        CK(cudaMemsetAsync(cu->d_cpg_f64, 0, cu->n_cpg_f64 * 8, cu->stream));
    }
    CK(cudaMemsetAsync(cu->d_misc, 0, (2 * ITX_MAX_TID_SEEN + 8) * 4, cu->stream));
    CK(cudaStreamSynchronize(cu->stream));
    return ITX_OK;
}

extern "C" void itx_index_reset_counts(itx_index *ix) {
    char err[ITX_ERRLEN];
    cudaSetDevice(ix->cu->device);
    zero_counters(ix, err, 0);
    ix->cu->used_el = ix->cu->used_cpg = ix->cu->used_cpg_el = ix->cu->used_bp = 0;
    ix->cpg_lines = ix->cpg_in_repeat = 0;
    if (ix->cu->dup.keys) {          /* forget the reads of the previous run */
        cudaMemset(ix->cu->dup.keys, 0xff, ix->cu->dup.cap * sizeof(itx_k128)); cudaMemset(ix->cu->dup.ords, 0xff, ix->cu->dup.cap * 8);
        cudaMemset(ix->cu->dup.mins, 0xff, 16); cudaMemset(ix->cu->dup.mins + 2, 0, 8);
    }
    ix->cu->dup_ord_base = 0;
    memset(ix->cnt, 0, sizeof ix->cnt);
    for (int32_t i = 0; i < ix->subs.n; i++) { ix->sub[i].read_count = ix->sub[i].read_count_unique = 0; ix->sub[i].cpg_count = 0; ix->sub[i].cpg_score = 0; }
    for (int32_t i = 0; i < ix->fams.n; i++) { ix->fam[i].read_count = ix->fam[i].read_count_unique = 0; ix->fam[i].cpg_count = 0; ix->fam[i].cpg_score = 0; }
    for (int32_t i = 0; i < ix->clas.n; i++) { ix->cla[i].read_count = ix->cla[i].read_count_unique = 0; ix->cla[i].cpg_count = 0; ix->cla[i].cpg_score = 0; }
    if (ix->el_names) for (long long i = 0; i < ix->n_elem; i++) { for (uint32_t k = 0; k < ix->el_names_n[i]; k++) free(ix->el_names[i][k]); ix->el_names_n[i] = 0; }
    itx_strtab_free(&ix->warned); itx_strtab_init(&ix->warned);
}

extern "C" itx_index *itx_index_build(const char *chrom_sizes, const char *rep_sizes, const char *rmsk,
                                      int filter_field, const char *filter_name, char err[ITX_ERRLEN]) {
    return itx_index_build_on(g_device, chrom_sizes, rep_sizes, rmsk, filter_field, filter_name, err);
}
extern "C" itx_index *itx_index_build_on(int device, const char *chrom_sizes, const char *rep_sizes, const char *rmsk,
                                         int filter_field, const char *filter_name, char err[ITX_ERRLEN]) {
    const int g_device = device;               /* shadows the process-wide default: this index lives on `device` */
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    itx_index *ix = (itx_index *)calloc(1, sizeof(itx_index));
    /* the CUDA driver and context come up on a second thread while this one parses rmsk.txt */
    pthread_t warm; const bool warming = pthread_create(&warm, NULL, cuda_warm_up, (void *)(intptr_t)g_device) == 0;
    const int host_rc = itx_host_index_load(ix, chrom_sizes, rep_sizes, rmsk, filter_field, filter_name, err);
    if (warming) pthread_join(warm, NULL);
    cudaGetLastError();
    if (host_rc != ITX_OK) { itx_host_index_free(ix); free(ix); return NULL; }
    itx_cuda *cu = (itx_cuda *)calloc(1, sizeof(itx_cuda));
    ix->cu = cu; ix->device = cu->device = g_device;
    {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= g_device) {
            snprintf(err, ITX_ERRLEN, "no usable CUDA device %d (libiteres_gpu has no CPU path)", g_device);
            goto fail;
        }
        CKN(cudaSetDevice(g_device));
        cudaDeviceProp prop; CKN(cudaGetDeviceProperties(&prop, g_device));
        cu->sm_count = prop.multiProcessorCount; cu->smem_optin = prop.sharedMemPerBlockOptin;
        CKN(cudaStreamCreateWithFlags(&cu->stream, cudaStreamNonBlocking));
        CKN(cudaStreamCreateWithFlags(&cu->copy_stream, cudaStreamNonBlocking));
        const size_t ne = (size_t)ix->n_elem; const int32_t nc = ix->chroms.n, ns = ix->subs.n, nf = ix->fams.n, ncl = ix->clas.n;
        if (upload(&cu->d_iv, ix->iv, ne, err) || upload(&cu->d_ivf, ix->ivf, ne, err) || upload(&cu->d_bucket, ix->bucket, (size_t)ix->n_bucket, err) ||
            upload(&cu->d_chrom_bucket, ix->chrom_bucket, (size_t)nc + 1, err) || upload(&cu->d_cinfo, ix->cinfo, (size_t)nc, err) ||
            upload(&cu->d_sinfo, ix->sinfo, (size_t)ns, err) || upload(&cu->d_meta, ix->meta, ne, err) ||
            upload(&cu->d_meta2, ix->meta2, ne, err) || upload(&cu->d_chrom_off, ix->chrom_off, (size_t)nc + 1, err) ||
            upload(&cu->d_chrom_size, ix->chrom_size, (size_t)nc, err) || upload(&cu->d_sub_len, ix->sub_len, (size_t)ns, err) ||
            upload(&cu->d_sub_bp_off, ix->sub_bp_off, (size_t)ns + 1, err) || upload(&cu->d_sub_fold, ix->sub_fold, (size_t)ns, err)) goto fail;
        /* chromosome-name table for XA lookups */
        uint32_t nslot = 16; while (nslot < (uint32_t)nc * 2u + 2u) nslot <<= 1;
        uint32_t *slot = (uint32_t *)calloc(nslot, 4), *noff = (uint32_t *)calloc((size_t)nc + 1, 4);
        size_t pool = 0; for (int32_t c = 0; c < nc; c++) pool += strlen(ix->chroms.names[c]) + 1;
        char *poolb = (char *)calloc(pool + 1, 1); size_t w = 0;
        for (int32_t c = 0; c < nc; c++) {
            const char *nm = ix->chroms.names[c]; size_t l = strlen(nm);
            noff[c] = (uint32_t)w; memcpy(poolb + w, nm, l + 1); w += l + 1;
            uint32_t i = itx_fnv1a(nm, l) & (nslot - 1);
            while (slot[i]) i = (i + 1) & (nslot - 1);
            slot[i] = (uint32_t)c + 1;
        }
        int r = upload(&cu->d_cname_slot, slot, nslot, err) || upload(&cu->d_cname_off, noff, (size_t)nc + 1, err) || upload(&cu->d_cname_pool, poolb, pool + 1, err);
        free(slot); free(noff); free(poolb);
        if (r) goto fail;
        {
            uint32_t *n32 = itx_names32(ix->chroms.names, nc);
            r = upload(&cu->d_cname32, n32, (size_t)(nc > 0 ? nc : 1) * 8, err);
            free(n32);
            if (r) goto fail;
        }
        /* counter block */
        const size_t ng = (size_t)(ns + nf + ncl);
        cu->n_u64 = 16 + 2 * ng; cu->n_u32 = 2 * (size_t)ix->bp_len + 2 * ne;
        cu->n_cpg_u32 = ng + ne; cu->n_cpg_f64 = ng + (size_t)ix->bp_len + ne;
        CKN(cudaMalloc(&cu->d_u64, (cu->n_u64 ? cu->n_u64 : 1) * 8)); CKN(cudaMalloc(&cu->d_u32, (cu->n_u32 ? cu->n_u32 : 1) * 4));
        CKN(cudaMalloc(&cu->d_cpg_u32, (cu->n_cpg_u32 ? cu->n_cpg_u32 : 1) * 4)); CKN(cudaMalloc(&cu->d_cpg_f64, (cu->n_cpg_f64 ? cu->n_cpg_f64 : 1) * 8));
        CKN(cudaMalloc(&cu->d_misc, (2 * ITX_MAX_TID_SEEN + 8) * 4));      /* unknown-tid marks of the scan, of the running k_scan launch, status words */
        CKN(cudaMalloc((void **)&cu->d_bp, ((size_t)ix->bp_len + 1) * 4)); CKN(cudaMalloc((void **)&cu->d_bp_u, ((size_t)ix->bp_len + 1) * 4));
        CKN(cudaMalloc((void **)&cu->d_carry, 8)); CKN(cudaMalloc((void **)&cu->d_running, 8)); CKN(cudaMalloc((void **)&cu->d_winbad, 4));
        CKN(cudaMalloc((void **)&cu->d_work, 16)); CKN(cudaMemset(cu->d_work, 0, 16));
        CKN(cudaMalloc((void **)&cu->d_carry_log, ITX_MAX_WINDOWS * 8)); CKN(cudaMalloc((void **)&cu->d_fused, 32)); CKN(cudaMemset(cu->d_fused, 0, 32));
        CKN(cudaHostAlloc((void **)&cu->h_scratch, ITX_SCRATCH_BYTES, cudaHostAllocDefault));
        CKN(cudaFuncSetAttribute(k_decode_span, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CKN(cudaFuncSetAttribute(k_lz_resolve, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        itx_dev_index &D = cu->D;
        D.iv = (const itx_iv *)cu->d_iv; D.ivf = (const itx_iv *)cu->d_ivf; D.bucket = (const uint32_t *)cu->d_bucket; D.chrom_bucket = (const long long *)cu->d_chrom_bucket;
        D.cinfo = (const itx_chrominfo *)cu->d_cinfo; D.sinfo = (const itx_subinfo *)cu->d_sinfo; D.meta = (const itx_meta *)cu->d_meta; D.meta2 = (const itx_meta2 *)cu->d_meta2;
        D.chrom_off = (const long long *)cu->d_chrom_off; D.chrom_size = (const int32_t *)cu->d_chrom_size; D.n_chrom = nc; D.n_elem = ix->n_elem;
        D.cname_slot = (const uint32_t *)cu->d_cname_slot; D.cname_nslot = nslot; D.cname_off = (const uint32_t *)cu->d_cname_off; D.cname_pool = (const char *)cu->d_cname_pool; D.cname32 = (const uint32_t *)cu->d_cname32;
        D.n_sub = ns; D.n_fam = nf; D.n_cla = ncl; D.stat_mode = ix->stat_mode;
        D.sub_len = (const uint32_t *)cu->d_sub_len; D.sub_bp_off = (const unsigned long long *)cu->d_sub_bp_off; D.sub_fold = (const int32_t *)cu->d_sub_fold;
        D.cnt = (unsigned long long *)cu->d_u64; D.grp = D.cnt + 16;
        D.bp_diff = (uint32_t *)cu->d_u32; D.bp_diff_u = D.bp_diff + ix->bp_len; D.el_cnt = D.bp_diff_u + ix->bp_len; D.el_cnt_u = D.el_cnt + ne;
        D.grp_cpg = (uint32_t *)cu->d_cpg_u32; D.el_cpg = D.grp_cpg + ng;
        D.grp_cpg_score = (double *)cu->d_cpg_f64; D.bp_cpg = D.grp_cpg_score + ng; D.el_cpg_score = D.bp_cpg + ix->bp_len;
        D.tid_unknown_seen = (uint32_t *)cu->d_misc; D.status = D.tid_unknown_seen + 2 * ITX_MAX_TID_SEEN;
        CKN(cudaMalloc(&cu->d_D, sizeof D)); CKN(cudaMemcpy(cu->d_D, &D, sizeof D, cudaMemcpyHostToDevice));
        if (zero_counters(ix, err, 1)) goto fail;
    }
    ix->tune_chunk = 65536; ix->tune_window = 1ull << 30; ix->tune_threads = 0;
    return ix;
fail:
    cuda_free_all(cu); ix->cu = NULL;
    itx_host_index_free(ix); free(ix);
    return NULL;
}

extern "C" int itx_tune(itx_index *ix, uint32_t chunk_bytes, uint64_t window_bytes, int32_t inflate_threads) {
    if (chunk_bytes) { if (chunk_bytes < 256 || chunk_bytes > (1u << 20) || (chunk_bytes & 63)) return ITX_EARG; ix->tune_chunk = chunk_bytes; }
    if (window_bytes) { if (window_bytes < (1u << 16)) return ITX_EARG; ix->tune_window = window_bytes; }
    if (inflate_threads) ix->tune_threads = inflate_threads;
    return ITX_OK;
}
extern "C" int itx_mark(itx_index *ix, int slot) {
    itx_cuda *cu = ix->cu;
    if (slot < 0 || slot >= 8) return ITX_EARG;
    cudaSetDevice(cu->device);
    if (!cu->marks_made) { for (int i = 0; i < 8; i++) cudaEventCreate(&cu->marks[i]); cu->marks_made = 1; }
    return cudaEventRecord(cu->marks[slot], cu->stream) == cudaSuccess ? ITX_OK : ITX_ENODEV;
}
extern "C" double itx_elapsed_ms(itx_index *ix, int a, int b) {
    itx_cuda *cu = ix->cu;
    if (a < 0 || a >= 8 || b < 0 || b >= 8 || !cu->marks_made) return -1.0;
    cudaSetDevice(cu->device);
    if (cudaEventSynchronize(cu->marks[a]) != cudaSuccess || cudaEventSynchronize(cu->marks[b]) != cudaSuccess) return -1.0;
    float ms = -1.0f;
    if (cudaEventElapsedTime(&ms, cu->marks[a], cu->marks[b]) != cudaSuccess) return -1.0;
    return (double)ms;
}
extern "C" int itx_trace_enable(itx_index *ix, uint64_t cap) { ix->trace_cap = cap; return ITX_OK; }
extern "C" void itx_last_profile(const itx_index *ix, itx_profile *p) { *p = ix->prof; }

/* ------------------------------------------------------------------ BAM header */
extern "C" itx_bam_header *itx_bam_header_parse(itx_index *ix, const uint8_t *bam, uint64_t len, int addChr, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    itx_bam_header *h = (itx_bam_header *)calloc(1, sizeof *h);
    if (itx_host_parse_bam_header(ix, bam, len, addChr, h, err) != ITX_OK) { itx_bam_header_free(h); return NULL; }
    cudaSetDevice(ix->cu->device);
    size_t n = (size_t)(h->n_ref ? h->n_ref : 1);
    if (cudaMalloc((void **)&h->d_tid, n * sizeof(itx_tidinfo)) != cudaSuccess ||
        cudaMemcpy(h->d_tid, h->tid, n * sizeof(itx_tidinfo), cudaMemcpyHostToDevice) != cudaSuccess) {
        snprintf(err, ITX_ERRLEN, "CUDA error uploading the reference table"); itx_bam_header_free(h); return NULL;
    }
    return h;
}
extern "C" uint64_t itx_bam_header_len(const itx_bam_header *h) { return h->hdr_len; }
extern "C" void itx_bam_header_free(itx_bam_header *h) {
    if (!h) return;
    if (h->names) for (int32_t i = 0; i < h->n_ref; i++) free(h->names[i]);
    free(h->names); free(h->lens); free(h->tid);
    if (h->d_tid) cudaFree(h->d_tid);
    free(h);
}

/* ------------------------------------------------------------------ scan machinery */
/* window_bytes: the largest launch group of the tuple path (16 bytes of tuple per 36 bytes of stream); log_bytes: the
 * largest launch group of k_scan, which only needs the spans' entry / exit logs and so can cover a whole resident stream */
/* the queue k_scan hands its XA:Z reads to k_xa in: one entry per 42 bytes of a launch group (no record that carries an XA list is
 * shorter), so it cannot overflow.  0: no room on the device -- the caller takes the tuple path, which looks at XA in line. */
static int ensure_xa_queue(itx_cuda *cu, uint64_t group_bytes) {
    const uint64_t need = group_bytes / 42 + 1024 + 8192ull * ITX_XA_BLK;      /* + a block (reserved, perhaps never filled) per warp of the largest grid */
    if (!cu->d_xa_n) { if (cudaMalloc((void **)&cu->d_xa_n, 8) != cudaSuccess || cudaMemset(cu->d_xa_n, 0, 8) != cudaSuccess) { cudaGetLastError(); return 0; } }
    if (cu->d_xa_q && cu->xa_cap >= need) return 1;
    cudaStreamSynchronize(cu->stream);
    cudaFree(cu->d_xa_q); cu->d_xa_q = NULL; cu->xa_cap = 0;
    if (cudaMalloc((void **)&cu->d_xa_q, need * 8) != cudaSuccess) { cudaGetLastError(); return 0; }
    cu->xa_cap = need;
    return 1;
}
static int ensure_work(itx_index *ix, uint64_t window_bytes, uint64_t log_bytes, char *err) {
    itx_cuda *cu = ix->cu;
    uint32_t C = ix->tune_chunk, S = C / 36 + 1;
    uint64_t need = window_bytes / C + 2;
    uint64_t need_log = (log_bytes > window_bytes ? log_bytes : window_bytes) / C + 2;
    bool want_trace = ix->trace_cap != 0 || cu->ord_cap != 0;
    const uint64_t trace_need = ix->trace_cap > cu->ord_cap ? ix->trace_cap : cu->ord_cap;
    if (cu->d_tuples && cu->C == C && cu->cap_chunks >= need && cu->cap_log >= need_log && (!want_trace || cu->d_rec_base) && (!cu->want_sel || cu->d_sel)) goto trace;
    cudaFree(cu->d_tuples); cudaFree(cu->d_entry); cudaFree(cu->d_exit); cudaFree(cu->d_nrec); cudaFree(cu->d_rec_base); cudaFree(cu->d_sel);
    cu->d_tuples = NULL; cu->d_entry = cu->d_exit = cu->d_rec_base = NULL; cu->d_nrec = NULL; cu->d_sel = NULL;
    cu->C = C; cu->S = S; cu->cap_chunks = need; cu->cap_log = need_log;
    CK(cudaMalloc((void **)&cu->d_tuples, need * S * sizeof(itx_tuple)));
    need = need_log;                                          /* the per-span arrays below are sized for the logs */
    CK(cudaMalloc((void **)&cu->d_entry, need * 8)); CK(cudaMalloc((void **)&cu->d_exit, need * 8)); CK(cudaMalloc((void **)&cu->d_nrec, need * 4));
    {
        CK(cudaFuncSetAttribute(k_decode_span, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ITX_DECODE_SMEM));
        int nb = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_decode_span, ITX_DW * 32, ITX_DECODE_SMEM));
        cu->decode_ctas = nb > 0 ? nb : 1;
    }
    if (want_trace) CK(cudaMalloc((void **)&cu->d_rec_base, need * 8));
    if (cu->want_sel) CK(cudaMalloc((void **)&cu->d_sel, cu->cap_chunks * S * sizeof(long long)));
trace:
    if (want_trace && (!cu->d_trace || cu->trace_cap < trace_need)) {
        cudaFree(cu->d_trace); cu->d_trace = NULL;
        CK(cudaMalloc((void **)&cu->d_trace, trace_need * sizeof(itx_trace)));
        cu->trace_cap = trace_need;
    }
    return ITX_OK;
}
static cudaEvent_t get_event(itx_cuda *cu, int i) {
    while (cu->n_ev_made <= i && cu->n_ev_made < ITX_MAX_EVENTS) cudaEventCreate(&cu->ev[cu->n_ev_made++]);
    return cu->ev[i < ITX_MAX_EVENTS ? i : ITX_MAX_EVENTS - 1];
}
static itx_dev_opts dev_opts(const itx_scan_opts *o) {
    itx_dev_opts d; d.mapQ = o->mapQ; d.iSize = o->iSize; d.extension = o->extension; d.minCoverage = o->minCoverage;
    d.filter = o->filter; d.discardWrongEnd = o->discardWrongEnd; d.treat = o->treat; d.diffSubfam = o->diffSubfam;
    return d;
}
static int check_opts(const itx_scan_opts *o, char *err) { (void)o; (void)err; return ITX_OK; }

/* -R: room for `extra` more keys in the table (load kept below 0.7); a full table moves into one twice the size */
static int ensure_dup_table(itx_cuda *cu, dup_table *T, uint64_t extra, char *err) {
    unsigned long long have = 0;
    if (T->mins) { CK(cudaStreamSynchronize(cu->stream)); CK(cudaMemcpy(&have, T->mins + 2, 8, cudaMemcpyDeviceToHost)); }
    else {
        CK(cudaMalloc((void **)&T->mins, 24));
        CK(cudaMemset(T->mins, 0xff, 16)); CK(cudaMemset(T->mins + 2, 0, 8));
    }
    if (T->keys && (have + extra) * 10 <= T->cap * 7) return ITX_OK;
    uint64_t cap = 1ull << 20; while (cap * 7 < (have + extra) * 10 * 2) cap <<= 1;
    itx_k128 *nk = NULL; unsigned long long *no = NULL;
    if (cudaMalloc((void **)&nk, cap * sizeof(itx_k128)) != cudaSuccess || cudaMalloc((void **)&no, cap * 8) != cudaSuccess) {
        cudaGetLastError(); cudaFree(nk); snprintf(err, ITX_ERRLEN, "cannot allocate the -R key table (%llu entries)", (unsigned long long)cap); return ITX_ENOMEM;
    }
    CK(cudaMemsetAsync(nk, 0xff, cap * sizeof(itx_k128), cu->stream)); CK(cudaMemsetAsync(no, 0xff, cap * 8, cu->stream));
    if (T->keys) {
        CK(cudaMemsetAsync(T->mins + 2, 0, 8, cu->stream));
        itx_dedup_args A; memset(&A, 0, sizeof A); A.keys = nk; A.ords = no; A.mask = cap - 1; A.mins = T->mins; A.status = cu->D.status;
        k_dedup_rehash<<<cu->sm_count * 8, 256, 0, cu->stream>>>(T->keys, T->ords, T->cap, A);
        CK(cudaStreamSynchronize(cu->stream));
        cudaFree(T->keys); cudaFree(T->ords);
    }
    T->keys = nk; T->ords = no; T->cap = cap;
    return ITX_OK;
}
/* an empty table (the part table before each phase-1 scan: a wrong first-record guess may have entered keys of decoy records) */
static int dup_table_clear(itx_cuda *cu, dup_table *T, char *err) {
    int rc = ensure_dup_table(cu, T, 0, err); if (rc) return rc;
    CK(cudaMemsetAsync(T->keys, 0xff, T->cap * sizeof(itx_k128), cu->stream)); CK(cudaMemsetAsync(T->ords, 0xff, T->cap * 8, cu->stream));
    CK(cudaMemsetAsync(T->mins, 0xff, 16, cu->stream)); CK(cudaMemsetAsync(T->mins + 2, 0, 8, cu->stream));
    return ITX_OK;
}

/* Scan context: the stream lives in one device buffer `b` of `len` bytes (plus slack); the window
 * loop processes chunks [k_next, k_hi) once `avail` bytes are on the device. */
typedef struct scan_ctx_s {
    itx_index *ix; const itx_bam_header *h; const uint8_t *b; uint64_t len; itx_dev_opts o;
    uint64_t k_first, k_end, k_next; int ev_n; int windows;
    int n_launch;
    int rmdup;
    int collect;            /* phase 1 of -R across ranks: the tuple path enters the unique fragments' keys into the part table and counts nothing */
    uint64_t first_entry;   /* collect mode, guessed first record: the first record start the repaired chain met (what k_scan logs in the fused path) */
    /* fused mode: k_scan instead of the tuple path; the windows are logged so that a failed chain check can be replayed */
    int fused; uint32_t n_win, wins_cap; struct scan_win { uint64_t k0; uint32_t n; uint64_t avail, len, own; } *wins;
    /* a scan that is one rank's shard of a stream: record starts at or past `own` are the next rank's; the first record start is
     * guessed (carry0 == ITX_OFF_GUESS) or handed in; what the chain did at both ends comes back in entry_out / carry_out */
    uint64_t own, carry0, entry_out, carry_out;
    /* ordered mode */
    int ordered, names; uint32_t mapQ; uint64_t p_cur; char **tname;
} scan_ctx;

/* ------------------------------------------------------------------ ordered mode: -B / -V bed lines, filter -r read names */
/* These outputs follow the reads in file order and need their names and aux strings, so they are produced on the
 * host -- but from the device's verdicts: every launch group leaves one trace entry per record (fragment, flags,
 * selected rmsk row); the host pulls the entries and the group's bytes of the stream, walks the records once and
 * prints.  Nothing about a read is decided on the host. */
static int ordered_open_files(itx_cuda *cu, const itx_scan_opts *o, char *err) {
    if (cu->bed_owner) return ITX_OK;                  /* an outer entry point of the same run holds them */
    if (cu->bed_f) { fclose(cu->bed_f); cu->bed_f = NULL; }             /* left behind by a scan that failed */
    if (cu->bed_uf) { fclose(cu->bed_uf); cu->bed_uf = NULL; }
    if (o->outbed && !cu->bed_f && !(cu->bed_f = fopen(o->outbed, "w"))) { snprintf(err, ITX_ERRLEN, "Can't open %s to write: %s", o->outbed, strerror(errno)); return ITX_EIO; }
    if (o->outbed_unique && !cu->bed_uf && !(cu->bed_uf = fopen(o->outbed_unique, "w"))) { snprintf(err, ITX_ERRLEN, "Can't open %s to write: %s", o->outbed_unique, strerror(errno)); return ITX_EIO; }
    return ITX_OK;
}
static void ordered_close_files(itx_cuda *cu) {
    if (cu->bed_f) { fclose(cu->bed_f); cu->bed_f = NULL; }
    if (cu->bed_uf) { fclose(cu->bed_uf); cu->bed_uf = NULL; }
    cu->bed_owner = 0;
}
static int ordered_begin(scan_ctx *sc, const itx_scan_opts *o, char *err) {
    itx_index *ix = sc->ix; itx_cuda *cu = ix->cu; const itx_bam_header *h = sc->h;
    int rc = ordered_open_files(cu, o, err); if (rc) return rc;
    sc->p_cur = h->hdr_len;
    sc->tname = itx_ordered_tnames(h);
    if (sc->names) itx_ordered_names_init(ix);
    return ITX_OK;
}
static void ordered_end(scan_ctx *sc) {
    if (!sc->ordered) return;
    if (sc->tname) { for (int32_t t = 0; t < sc->h->n_ref; t++) free(sc->tname[t]); free(sc->tname); sc->tname = NULL; }
    itx_cuda *cu = sc->ix->cu;
    if (!cu->bed_owner) ordered_close_files(cu);
    if (cu->bed_f) fflush(cu->bed_f);
    if (cu->bed_uf) fflush(cu->bed_uf);
}
/* the launch group just enqueued: wait for it, fetch its trace entries and its bytes, walk its records */
static int ordered_drain(scan_ctx *sc, uint64_t avail, char *err) {
    itx_index *ix = sc->ix; itx_cuda *cu = ix->cu;
    unsigned long long n_w = 0, carry = 0;
    CK(cudaStreamSynchronize(cu->stream));
    CK(cudaMemcpy(&n_w, cu->d_running, 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&carry, cu->d_carry, 8, cudaMemcpyDeviceToHost));
    if (n_w == 0) return ITX_OK;
    if (n_w > cu->trace_cap) { snprintf(err, ITX_ERRLEN, "internal: %llu records in a launch group, room for %llu trace entries", n_w, (unsigned long long)cu->trace_cap); return ITX_ENOMEM; }
    uint64_t p_end = carry;                                            /* the next group's first record, or past the end of a cut stream */
    const uint64_t lim = avail < sc->len ? avail : sc->len;
    if (p_end > lim) p_end = lim;
    if (p_end < sc->p_cur) p_end = sc->p_cur;
    if (cu->h_ord_trace_cap < n_w) { free(cu->h_ord_trace); cu->h_ord_trace = (itx_trace *)malloc(n_w * sizeof(itx_trace)); cu->h_ord_trace_cap = n_w; }
    const uint64_t nbytes = p_end - sc->p_cur;
    if (cu->h_ord_buf_cap < nbytes + ITX_SLACK) { free(cu->h_ord_buf); cu->h_ord_buf = (uint8_t *)malloc(nbytes + ITX_SLACK); cu->h_ord_buf_cap = nbytes + ITX_SLACK; }
    if (!cu->h_ord_trace || !cu->h_ord_buf) { snprintf(err, ITX_ERRLEN, "out of host memory in the ordered pass"); return ITX_ENOMEM; }
    CK(cudaMemcpy(cu->h_ord_trace, cu->d_trace, n_w * sizeof(itx_trace), cudaMemcpyDeviceToHost));
    if (nbytes) CK(cudaMemcpy(cu->h_ord_buf, sc->b + sc->p_cur, nbytes, cudaMemcpyDeviceToHost));
    memset(cu->h_ord_buf + nbytes, 0, ITX_SLACK);
    itx_ordered_sink K; K.bed = cu->bed_f; K.bed_u = cu->bed_uf; K.names = sc->names; K.mapQ = sc->mapQ; K.tname = sc->tname; K.n_ref = sc->h->n_ref; K.ix = ix;
    const uint64_t p = itx_ordered_walk(K, cu->h_ord_buf, nbytes, cu->h_ord_trace, n_w);
    sc->p_cur += p;
    return ITX_OK;
}

/* window: bytes per launch group; resident != 0: the whole stream is already on the device, so k_scan (which writes no
 * tuples) takes it in ONE launch group unless itx_tune set a window -- one tail instead of one per GiB */
#define ITX_DEFAULT_WINDOW (1ull << 30)
static void l2_persist_window(itx_index *ix);
#define ITX_CARRY_HEADER (~0ull)          /* scan_begin: the chain starts right after the BAM header (a scan from the start of a stream) */
static int scan_begin(scan_ctx *sc, itx_index *ix, const itx_bam_header *h, const uint8_t *d_bam, uint64_t len, const itx_scan_opts *o, uint64_t window, char *err, int resident = 0,
                      uint64_t carry0 = ITX_CARRY_HEADER) {
    itx_cuda *cu = ix->cu;
    memset(sc, 0, sizeof *sc);
    sc->ix = ix; sc->h = h; sc->b = d_bam; sc->len = len; sc->o = dev_opts(o);
    sc->own = ~0ull; sc->carry0 = carry0 == ITX_CARRY_HEADER ? h->hdr_len : carry0; sc->entry_out = sc->carry_out = ITX_OFF_NONE; sc->first_entry = ITX_OFF_NONE;
    if (o->filter) cu->used_el = 1; else if (ix->stat_mode) cu->used_bp = 1;
    sc->rmdup = o->rmDup != 0;
    cu->want_sel = 0;
    sc->ordered = (o->outbed || o->outbed_unique || o->readNames) ? 1 : 0; sc->names = o->readNames != 0; sc->mapQ = o->mapQ;
    if (sc->ordered) {
        if (window > (256ull << 20)) window = 256ull << 20;         /* the host pass buffers one launch group */
        cu->ord_cap = window / 37 + (uint64_t)ix->tune_chunk / 37 * 4 + 4096;    /* a record is at least 37 bytes long */
    } else cu->ord_cap = 0;
    uint64_t log_window = window;
    if (resident && !sc->ordered && ix->tune_window == ITX_DEFAULT_WINDOW && len > window) log_window = len < (1ull << 40) ? len : (1ull << 40);
    int rc = ensure_work(ix, window, log_window, err); if (rc) return rc;
    if (sc->ordered && (rc = ordered_begin(sc, o, err))) return rc;
    {
        const uint64_t first = sc->carry0 >= ITX_OFF_GUESS ? 0 : sc->carry0;
        sc->k_first = first / cu->C; sc->k_end = len > first ? (len + cu->C - 1) / cu->C : sc->k_first;
    }
    sc->k_next = sc->k_first;
    cu->h_scratch[0] = sc->carry0;              /* the previous scan ended with a synchronize: its copy out of the scratch is long done */
    CK(cudaMemcpyAsync(cu->d_carry, cu->h_scratch, 8, cudaMemcpyHostToDevice, cu->stream));
    CK(cudaMemsetAsync(cu->d_work, 0, 16, cu->stream));
    CK(cudaMemsetAsync(cu->D.status, 0, 8 * sizeof(uint32_t), cu->stream));      /* per-scan flags and failure counts */
    {   /* ITX_DECODE_KERNEL=thread selects the one-thread-per-chunk kernel (A/B measurement); chunks that are not whole tiles use it too */
        const char *v = getenv("ITX_DECODE_KERNEL");
        cu->decode_variant = ((v && strcmp(v, "thread") == 0) || (cu->C % ITX_STAGE) != 0 || cu->C > (1u << 20)) ? 1 : 0;
        if (((uintptr_t)d_bam & 15) != 0) cu->decode_variant = 1;
    }
    if (ix->trace_cap || sc->ordered) CK(cudaMemsetAsync(cu->d_running, 0, 8, cu->stream));
    {   /* one fused kernel per launch group unless something needs the tuples (-R, the ordered outputs, traces, ITX_FUSED=0) */
        const char *v = getenv("ITX_FUSED");
        sc->fused = !(v && strcmp(v, "0") == 0) && cu->decode_variant == 0 && !sc->rmdup && !sc->ordered && !ix->trace_cap && !cu->want_sel;
        if (sc->fused && sc->o.diffSubfam) {
            /* a k_scan launch group covers at most cap_log spans */
            const uint64_t group = (cu->cap_log) * (uint64_t)cu->C;
            if (!ensure_xa_queue(cu, group < len + cu->C ? group : len + cu->C)) sc->fused = 0;
        }
        if (sc->carry0 == ITX_OFF_GUESS && (sc->rmdup || sc->ordered)) { snprintf(err, ITX_ERRLEN, "-R, -B / -V and filter -r follow the reads in file order: they are not available in a sharded scan"); return ITX_ENOTSUP; }
        if (sc->fused) { CK(cudaMemsetAsync(cu->d_fused, 0xff, 4, cu->stream)); CK(cudaMemsetAsync(cu->d_fused + 1, 0, 12, cu->stream)); CK(cudaMemsetAsync(cu->d_fused + 4, 0xff, 8, cu->stream)); }
    }
    l2_persist_window(ix);
    if (!resident) CK(cudaStreamSynchronize(cu->stream));      /* the streaming paths go on to use other streams (copies, inflate) that read the flags just reset */
    return ITX_OK;
}
/* ITX_L2_PERSIST (default 1; 0 switches it off): the coverage difference arrays (the target of k_scan's scattered reductions) are asked to stay in L2
 * (persisting access-policy window on the scan stream) while the stream bytes pass through */
static void l2_persist_window(itx_index *ix) {
    itx_cuda *cu = ix->cu;
    const int want = env_int_early("ITX_L2_PERSIST", 1) ? 1 : 0;      /* default on: DRAM writes of a 50 M read k_scan 0.31 GB -> 0.01 GB, reads -0.3 GB (profiles/r02_k_scan_traffic_attribution.txt) */
    if (want == cu->l2_persist_on) return;
    cudaStreamAttrValue v; memset(&v, 0, sizeof v);
    if (want) {
        cudaDeviceProp prop; cudaGetDeviceProperties(&prop, cu->device);
        size_t bytes = 2 * (size_t)ix->bp_len * 4;
        if (bytes > (size_t)prop.accessPolicyMaxWindowSize) bytes = (size_t)prop.accessPolicyMaxWindowSize;
        size_t lim = bytes < (size_t)prop.persistingL2CacheMaxSize ? bytes : (size_t)prop.persistingL2CacheMaxSize;
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, lim);
        v.accessPolicyWindow.base_ptr = cu->d_u32; v.accessPolicyWindow.num_bytes = bytes; v.accessPolicyWindow.hitRatio = 1.0f;
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting; v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    cudaStreamSetAttribute(cu->stream, cudaStreamAttributeAccessPolicyWindow, &v);
    if (!want) cudaCtxResetPersistingL2Cache();
    cudaGetLastError();
    cu->l2_persist_on = want;
}
static itx_decode_args decode_args(const scan_ctx *sc, uint64_t k0, uint32_t n, uint64_t avail, uint64_t len, uint64_t own) {
    itx_cuda *cu = sc->ix->cu;
    itx_decode_args A;
    A.b = sc->b; A.len = len; A.avail = avail; A.k0 = k0; A.nchunks = n; A.C = cu->C; A.S = cu->S;
    A.own = own < len ? own : len;
    A.tid = sc->h->d_tid; A.n_ref = sc->h->n_ref; A.o = sc->o;
    A.tuples = cu->d_tuples; A.entry = cu->d_entry; A.exit_ = cu->d_exit; A.nrec = cu->d_nrec;
    A.carry = cu->d_carry; A.winbad = cu->d_winbad; A.status = cu->D.status; A.work = cu->d_work;
    return A;
}
static size_t hist_bytes(const itx_cuda *cu) { return 2ull * (size_t)(cu->D.n_sub + cu->D.n_fam + cu->D.n_cla) * 4; }
/* the tuple path for chunks [k0, k0 + n): k_decode_span (or k_decode) -> k_verify -> k_fixup -> [k_dedup x2] -> k_overlap */
static int launch_tuple_path(scan_ctx *sc, uint64_t k0, uint32_t n, uint64_t avail, uint64_t len, uint64_t own, char *err) {
    itx_index *ix = sc->ix; itx_cuda *cu = ix->cu;
    const itx_decode_args A = decode_args(sc, k0, n, avail, len, own);
    bool timed = sc->ev_n + 3 <= ITX_MAX_EVENTS;
    if (timed) cudaEventRecord(get_event(cu, sc->ev_n), cu->stream);
    if (cu->decode_variant == 0) {
        uint32_t db = (n + ITX_DW - 1) / ITX_DW, dmax = (uint32_t)(cu->sm_count * cu->decode_ctas);
        k_decode_span<<<db < dmax ? db : dmax, ITX_DW * 32, ITX_DECODE_SMEM, cu->stream>>>(A);
    } else k_decode<<<(n + 127) / 128, 128, 0, cu->stream>>>(A);
    k_verify<<<(n + 255) / 256, 256, 0, cu->stream>>>(A);
    k_fixup<<<1, 32, 0, cu->stream>>>(A);
    if (sc->collect && sc->carry0 == ITX_OFF_GUESS && sc->first_entry == ITX_OFF_NONE) {
        /* the span entries as k_fixup left them: the first one that is a record start is where the part's chain begins */
        std::vector<unsigned long long> en(n);
        CK(cudaMemcpyAsync(en.data(), cu->d_entry, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, cu->stream));
        CK(cudaStreamSynchronize(cu->stream));
        for (uint32_t i = 0; i < n && sc->first_entry == ITX_OFF_NONE; i++) sc->first_entry = en[i];
    }
    if (sc->rmdup || sc->collect) {
        dup_table *T = sc->collect ? &cu->part : &cu->dup;
        int rcd = ensure_dup_table(cu, T, (uint64_t)n * cu->C / 37 + 64, err); if (rcd) return rcd;
        itx_dedup_args R; R.b = sc->b; R.k0 = k0; R.nchunks = n; R.C = cu->C; R.S = cu->S; R.tuples = cu->d_tuples; R.nrec = cu->d_nrec;
        R.tid = sc->h->d_tid; R.n_ref = sc->h->n_ref; R.ord_base = sc->collect ? 0 : cu->dup_ord_base;
        R.keys = T->keys; R.ords = T->ords; R.mask = T->cap - 1; R.mins = T->mins; R.status = cu->D.status;
        const unsigned gb = (n + 7) / 8 < (unsigned)cu->sm_count * 8u ? (n + 7) / 8 : (unsigned)cu->sm_count * 8u;
        k_dedup<false><<<gb, 256, 0, cu->stream>>>(R);
        if (!sc->collect) k_dedup<true><<<gb, 256, 0, cu->stream>>>(R);
        sc->n_launch += sc->collect ? 1 : 2;
    }
    if (timed) cudaEventRecord(get_event(cu, sc->ev_n + 1), cu->stream);
    sc->n_launch += 3;
    if (sc->collect) {
        if (timed) { cudaEventRecord(get_event(cu, sc->ev_n + 2), cu->stream); sc->ev_n += 3; }
        return ITX_OK;
    }
    itx_overlap_args B;
    B.D = cu->D; B.b = sc->b; B.k0 = k0; B.nchunks = n; B.C = cu->C; B.S = cu->S; B.tuples = cu->d_tuples; B.nrec = cu->d_nrec; B.o = sc->o;
    B.trace = NULL; B.trace_cap = 0; B.rec_base = NULL; B.sel_out = cu->want_sel ? cu->d_sel : NULL; B.work = cu->d_work + 1; B.Dg = (const itx_dev_index *)cu->d_D;
    if (ix->trace_cap || sc->ordered) {
        if (sc->ordered) cudaMemsetAsync(cu->d_running, 0, 8, cu->stream);          /* the group's records are traced from slot 0 */
        k_rec_base<<<1, 1024, 0, cu->stream>>>(cu->d_nrec, n, cu->d_rec_base, cu->d_running);
        B.trace = cu->d_trace; B.trace_cap = cu->trace_cap; B.rec_base = cu->d_rec_base; sc->n_launch++;
    }
    const size_t hist = hist_bytes(cu);
    bool smem = (sc->o.filter == 0 && cu->D.stat_mode) && hist + ITX_OVL_WIN_SMEM + 1024 <= cu->smem_optin && hist <= 160 * 1024;
    int blocks = cu->sm_count * (hist > 48 * 1024 ? 1 : (hist > 24 * 1024 ? 2 : 4));
    uint32_t need_blocks = (n * ((cu->S + ITX_PART - 1) / ITX_PART) + 7) / 8; if ((uint32_t)blocks > need_blocks) blocks = (int)need_blocks; if (blocks < 1) blocks = 1;
    /* dynamic shared memory: the histogram (when it fits), then a table window per warp */
    if (smem) {
        const size_t sm = ((hist + 15) & ~(size_t)15) + ITX_OVL_WIN_SMEM;
        if (sm > 48 * 1024) cudaFuncSetAttribute(k_overlap<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        k_overlap<true><<<blocks, 256, sm, cu->stream>>>(B);
    } else k_overlap<false><<<blocks, 256, ITX_OVL_WIN_SMEM, cu->stream>>>(B);
    sc->n_launch++;
    if (timed) { cudaEventRecord(get_event(cu, sc->ev_n + 2), cu->stream); sc->ev_n += 3; }
    return ITX_OK;
}
/* the fused path: ONE kernel per launch group (k_scan); sign -1 takes a group's counts back */
static bool fused_smem_hist(const scan_ctx *sc) {
    const itx_cuda *cu = sc->ix->cu;
    return (sc->o.filter == 0 && cu->D.stat_mode) && ITX_SCAN_SMEM_BASE(ITX_SCAN_NW) + hist_bytes(cu) + 1024 <= cu->smem_optin;
}
template <bool SH, int NW, bool AB>
static void launch_scan_kernel(itx_cuda *cu, const itx_scan_args &P, uint32_t n, size_t smem, int *ctas) {
    if (!*ctas) {
        /* the device's opt-in maximum, not this index's need: the attribute belongs to the function, and another index of the
         * same process (other table sizes, another histogram) must not find it lowered */
        cudaFuncSetAttribute(k_scan<SH, NW, AB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cu->smem_optin - 1024);       /* (the kernel has a little static shared memory too) */
        cudaFuncSetAttribute(k_scan<SH, NW, AB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        int nb = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_scan<SH, NW, AB>, NW * 32, smem);
        *ctas = nb > 0 ? nb : 1;
    }
    const uint32_t want = (n + NW - 1) / NW, most = (uint32_t)(cu->sm_count * *ctas);
    k_scan<SH, NW, AB><<<want < most ? want : most, NW * 32, smem, cu->stream>>>(P);
}
static int launch_fused(scan_ctx *sc, uint32_t window, uint64_t k0, uint32_t n, uint64_t avail, uint64_t len, uint64_t own, int sign) {
    itx_cuda *cu = sc->ix->cu;
    itx_scan_args P; P.A = decode_args(sc, k0, n, avail, len, own); P.D = cu->D; P.Dg = (const itx_dev_index *)cu->d_D; P.sign = sign; P.window = window;
    P.carry_log = cu->d_carry_log; P.first_bad = cu->d_fused;
    P.xa_q = cu->d_xa_q; P.xa_n = cu->d_xa_n; P.xa_cap = sc->o.diffSubfam ? cu->xa_cap : 0;
    const bool sh = fused_smem_hist(sc);
    const size_t smem = ITX_SCAN_SMEM_BASE(ITX_SCAN_NW) + (sh ? hist_bytes(cu) : 0);
    /* the product kernel has its switches compiled in; ITX_SCAN_FLAGS selects the kernel that reads them at run time
     * (tests, A/B measurements: the counts do not depend on them) */
    P.flags = ITX_SCAN_PRODUCT;
    const char *fv = getenv("ITX_SCAN_FLAGS");
    const bool ab = fv != NULL;
    if (fv) P.flags = (uint32_t)strtoul(fv, NULL, 0);
    int *ctas = &cu->scan_ctas[(ab ? 2 : 0) + (sh ? 1 : 0)];
    if (!ab) { if (sh) launch_scan_kernel<true, ITX_SCAN_NW, false>(cu, P, n, smem, ctas); else launch_scan_kernel<false, ITX_SCAN_NW, false>(cu, P, n, smem, ctas); }
    else { if (sh) launch_scan_kernel<true, ITX_SCAN_NW, true>(cu, P, n, smem, ctas); else launch_scan_kernel<false, ITX_SCAN_NW, true>(cu, P, n, smem, ctas); }
    sc->n_launch++;
    if (sc->o.diffSubfam) {
        /* the reads k_scan queued (XA:Z alternates): mapped2diffSubfam and their accumulation, with the launch's sign */
        itx_xa_args X; X.D = cu->D; X.Dg = (const itx_dev_index *)cu->d_D; X.b = sc->b; X.tid = sc->h->d_tid; X.n_ref = sc->h->n_ref; X.o = sc->o;
        X.q = cu->d_xa_q; X.q_n = cu->d_xa_n; X.q_cap = cu->xa_cap; X.sign = sign; X.flags = P.flags;
        uint64_t blocks = ((uint64_t)n * cu->C / 42 + 255) / 256, most = (uint64_t)cu->sm_count * 8;
        if (blocks > most) blocks = most;
        if (blocks < 1) blocks = 1;
        const size_t fc_bytes = 2 * (size_t)(cu->D.n_fam + cu->D.n_cla) * 4;
        X.hist_fc = (sc->o.filter == 0 && cu->D.stat_mode && fc_bytes <= 4096) ? 1u : 0u;
        if (!cu->xa_attr) { cudaFuncSetAttribute(k_xa, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ITX_XA_SMEM + 4096); cu->xa_attr = 1; }
        k_xa<<<(unsigned)blocks, 256, ITX_XA_SMEM + (X.hist_fc ? fc_bytes : 0), cu->stream>>>(X);
        sc->n_launch++;
    }
    return ITX_OK;
}
/* launch the kernels for chunks [k_next, k_hi) (k_hi <= k_end); avail = bytes valid on the device */
static int scan_window(scan_ctx *sc, uint64_t k_hi, uint64_t avail, char *err) {
    itx_index *ix = sc->ix; itx_cuda *cu = ix->cu;
    while (sc->k_next < k_hi) {
        const uint64_t cap = (sc->fused ? cu->cap_log : cu->cap_chunks) - 1;
        uint64_t n64 = k_hi - sc->k_next; if (n64 > cap) n64 = cap;
        uint32_t n = (uint32_t)n64;
        if (sc->fused && sc->n_win >= ITX_MAX_WINDOWS) { snprintf(err, ITX_ERRLEN, "more than %d launch groups in one scan: raise the window with itx_tune", ITX_MAX_WINDOWS); return ITX_ENOTSUP; }
        if (sc->fused) {
            if (sc->n_win == sc->wins_cap) { sc->wins_cap = sc->wins_cap ? sc->wins_cap * 2 : 64; sc->wins = (scan_ctx::scan_win *)realloc(sc->wins, sc->wins_cap * sizeof(*sc->wins)); }
            sc->wins[sc->n_win].k0 = sc->k_next; sc->wins[sc->n_win].n = n; sc->wins[sc->n_win].avail = avail; sc->wins[sc->n_win].len = sc->len; sc->wins[sc->n_win].own = sc->own;
            bool timed = sc->ev_n + 3 <= ITX_MAX_EVENTS;
            if (timed) cudaEventRecord(get_event(cu, sc->ev_n), cu->stream);
            launch_fused(sc, sc->n_win, sc->k_next, n, avail, sc->len, sc->own, +1);
            if (timed) { cudaEventRecord(get_event(cu, sc->ev_n + 1), cu->stream); cudaEventRecord(get_event(cu, sc->ev_n + 2), cu->stream); sc->ev_n += 3; }
            sc->n_win++;
        } else {
            int rc = launch_tuple_path(sc, sc->k_next, n, avail, sc->len, sc->own, err); if (rc) return rc;
        }
        sc->windows++;
        sc->k_next += n;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { snprintf(err, ITX_ERRLEN, "kernel launch failed: %s", cudaGetErrorString(e)); return ITX_ENODEV; }
        if (sc->ordered) { int rco = ordered_drain(sc, avail, err); if (rco) return rco; }
    }
    return ITX_OK;
}
/* a chain check failed in window `first` (a span's guessed first record was not where the previous span ended): take back
 * what k_scan counted from that window on and count those windows again through the tuple path, which repairs guesses */
static int fused_replay(scan_ctx *sc, uint32_t first, char *err) {
    itx_cuda *cu = sc->ix->cu;
    for (uint32_t w = first; w < sc->n_win; w++) launch_fused(sc, w, sc->wins[w].k0, sc->wins[w].n, sc->wins[w].avail, sc->wins[w].len, sc->wins[w].own, -1);
    CK(cudaMemcpyAsync(cu->d_carry, cu->d_carry_log + first, 8, cudaMemcpyDeviceToDevice, cu->stream));
    for (uint32_t w = first; w < sc->n_win; w++)              /* a k_scan launch group may be larger than the tuple buffers: in pieces */
        for (uint64_t d = 0; d < sc->wins[w].n; d += cu->cap_chunks - 1) {
            const uint64_t n = sc->wins[w].n - d < cu->cap_chunks - 1 ? sc->wins[w].n - d : cu->cap_chunks - 1;
            int rc = launch_tuple_path(sc, sc->wins[w].k0 + d, (uint32_t)n, sc->wins[w].avail, sc->wins[w].len, sc->wins[w].own, err); if (rc) return rc;
        }
    return ITX_OK;
}
static int scan_end(scan_ctx *sc, uint64_t cnt[13], char *err) {
    itx_index *ix = sc->ix; itx_cuda *cu = ix->cu;
    ordered_end(sc);
    /* one round trip for everything the host reads at the end of a scan -- the chain verdict of k_scan, the 13 counters, the
     * flags, the unknown-tid marks -- into pinned memory, so the four copies queue up behind the kernels without a wait each */
    unsigned long long *hc = cu->h_scratch + 8; uint32_t *st = (uint32_t *)(cu->h_scratch + 24); uint32_t *first_bad_p = st + 8;
    uint32_t *seen_fast = (uint32_t *)((uint8_t *)cu->h_scratch + 256);
    const int32_t nt = sc->h->n_ref < ITX_MAX_TID_SEEN ? sc->h->n_ref : ITX_MAX_TID_SEEN, nt_fast = nt < ITX_SEEN_FAST ? nt : ITX_SEEN_FAST;
    *first_bad_p = 0xffffffffu;
    unsigned long long *carry_p = cu->h_scratch + 29, *entry_p = cu->h_scratch + 30;      /* bytes 232 and 240 of the report */
    *entry_p = ITX_OFF_NONE;
    if (sc->fused) CK(cudaMemcpyAsync(first_bad_p, cu->d_fused, 4, cudaMemcpyDeviceToHost, cu->stream));
    if (sc->fused && sc->carry0 == ITX_OFF_GUESS) CK(cudaMemcpyAsync(entry_p, cu->d_fused + 4, 8, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaMemcpyAsync(carry_p, cu->d_carry, 8, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaMemcpyAsync(hc, cu->D.cnt, 16 * 8, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaMemcpyAsync(st, cu->D.status, 8 * 4, cudaMemcpyDeviceToHost, cu->stream));
    if (nt_fast > 0) CK(cudaMemcpyAsync(seen_fast, cu->D.tid_unknown_seen, sizeof(uint32_t) * (size_t)nt_fast, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaStreamSynchronize(cu->stream));
    uint32_t first_bad = *first_bad_p;
    if (sc->fused) {
        if (first_bad == 0xffffffffu && sc->n_win && getenv("ITX_FUSED_TEST_REPLAY")) first_bad = 0;      /* test hook: replay everything */
        if (first_bad != 0xffffffffu) {
            int rc = fused_replay(sc, first_bad, err);
            if (rc) { free(sc->wins); sc->wins = NULL; return rc; }
            ix->prof.n_replayed_windows = sc->n_win - first_bad;
            CK(cudaMemcpyAsync(hc, cu->D.cnt, 16 * 8, cudaMemcpyDeviceToHost, cu->stream));
            CK(cudaMemcpyAsync(st, cu->D.status, 8 * 4, cudaMemcpyDeviceToHost, cu->stream));
            CK(cudaMemcpyAsync(carry_p, cu->d_carry, 8, cudaMemcpyDeviceToHost, cu->stream));
            if (nt_fast > 0) CK(cudaMemcpyAsync(seen_fast, cu->D.tid_unknown_seen, sizeof(uint32_t) * (size_t)nt_fast, cudaMemcpyDeviceToHost, cu->stream));
            CK(cudaStreamSynchronize(cu->stream));
        }
        free(sc->wins); sc->wins = NULL;
    }
    for (int k = 0; k < 13; k++) ix->cnt[k] = hc[k];
    if (cnt) memcpy(cnt, ix->cnt, sizeof ix->cnt);
    sc->carry_out = *carry_p; sc->entry_out = sc->carry0 == ITX_OFF_GUESS ? (sc->fused ? *entry_p : sc->first_entry) : sc->carry0;
    itx_profile *P = &ix->prof;
    P->decode_ms = P->overlap_ms = 0; P->total_ms = 0;
    for (int i = 0; i + 2 < sc->ev_n + 1 && i + 2 < ITX_MAX_EVENTS; i += 3) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, cu->ev[i], cu->ev[i + 1]); cudaEventElapsedTime(&b, cu->ev[i + 1], cu->ev[i + 2]);
        P->decode_ms += a; P->overlap_ms += b;
    }
    if (sc->ev_n >= 3) { float t = 0; cudaEventElapsedTime(&t, cu->ev[0], cu->ev[sc->ev_n - 1]); P->total_ms = t; }
    P->n_records = ix->cnt[0] + ix->cnt[1]; P->n_fragments = ix->cnt[6]; P->stream_bytes = sc->len;
    P->n_launches = (uint64_t)sc->n_launch; P->n_bad_chunks = st[1]; P->fused = sc->fused;
    P->d2h_bytes = 16 * 8 + 8 * 4 + sizeof(uint32_t) * (size_t)nt;
    if (sc->rmdup) cu->dup_ord_base += (sc->k_end + 1) * (uint64_t)cu->S;           /* the next file's reads come after this file's */
    if (st[4]) { snprintf(err, ITX_ERRLEN, "the -R key table overflowed"); return ITX_ENOMEM; }
    if (st[0] & 8u) { snprintf(err, ITX_ERRLEN, "internal: the XA queue overflowed"); return ITX_ENOMEM; }
    if (st[0] & 4u) { snprintf(err, ITX_ERRLEN, "a TMA bulk copy never completed (device-side time-out in k_decode_span)"); return ITX_ENODEV; }
    if (st[0] & 2u) { snprintf(err, ITX_ERRLEN, "a BAM record is longer than the staged window (%llu bytes); raise the window with itx_tune", (unsigned long long)ix->tune_window); return ITX_ENOTSUP; }
    /* chromosomes absent from the size file: the reference warns once per name (generic.c:796-801) */
    if (nt > 0) {
        uint32_t *seen = seen_fast, *big = NULL;
        if (nt > nt_fast) {
            big = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)nt);
            if (!big || cudaMemcpy(big, cu->D.tid_unknown_seen, sizeof(uint32_t) * (size_t)nt, cudaMemcpyDeviceToHost) != cudaSuccess) { free(big); big = NULL; }
            seen = big;
        }
        bool any = false;
        if (seen) for (int32_t t = 0; t < nt; t++) if (seen[t]) {
            any = true;
            char nm[600]; const char *raw = sc->h->names[t];
            if (sc->h->addChr && strcasecmp(raw, "MT") == 0) snprintf(nm, sizeof nm, "chrM");
            else if (sc->h->addChr && strncmp(raw, "chr", 3) != 0) snprintf(nm, sizeof nm, "chr%s", raw);
            else snprintf(nm, sizeof nm, "%s", raw);
            if (itx_strtab_find(&ix->warned, nm) < 0) {
                itx_strtab_add(&ix->warned, nm);
                fprintf(stderr, "* Warning: read ends mapped to chromosome %s will be discarded as %s not existed in the chromosome size file\n", nm, nm);
            }
        }
        if (any) cudaMemsetAsync(cu->D.tid_unknown_seen, 0, sizeof(uint32_t) * (size_t)nt, cu->stream);
        free(big);
    }
    return ITX_OK;
}

extern "C" int itx_scan_bam_device(itx_index *ix, const itx_bam_header *h, const void *d_bam, uint64_t len,
                                   const itx_scan_opts *o, uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    int rc = check_opts(o, err); if (rc) return rc;
    CK(cudaSetDevice(ix->cu->device));
    memset(&ix->prof, 0, sizeof ix->prof);
    scan_ctx sc;
    if ((rc = scan_begin(&sc, ix, h, (const uint8_t *)d_bam, len, o, ix->tune_window < len ? ix->tune_window : len, err, 1))) return rc;
    if ((rc = scan_window(&sc, sc.k_end, len, err))) return rc;
    return scan_end(&sc, cnt, err);
}

/* host stream -> device: the whole uncompressed stream is kept in one device buffer (sized to the
 * stream), filled window by window; window w is scanned once window w+1 (or the end) has landed. */
static int ensure_stream_buffer(itx_cuda *cu, uint64_t len, char *err) {
    if (cu->d_stream && cu->d_stream_cap >= len + ITX_SLACK) return ITX_OK;
    cudaFree(cu->d_stream); cu->d_stream = NULL;
    size_t fr = 0, tot = 0; cudaMemGetInfo(&fr, &tot);
    if (len + ITX_SLACK + (1ull << 30) > fr) { snprintf(err, ITX_ERRLEN, "stream of %llu bytes does not fit the device (%llu free)", (unsigned long long)len, (unsigned long long)fr); return ITX_ENOMEM; }
    CK(cudaMalloc((void **)&cu->d_stream, len + ITX_SLACK));
    cu->d_stream_cap = len + ITX_SLACK;
    return ITX_OK;
}
static int ensure_stage(itx_cuda *cu, uint64_t bytes, char *err) {
    if (cu->h_stage[0] && cu->h_stage_cap >= bytes) return ITX_OK;
    for (int i = 0; i < 2; i++) { if (cu->h_stage[i]) cudaFreeHost(cu->h_stage[i]); cu->h_stage[i] = NULL; }
    for (int i = 0; i < 2; i++) CK(cudaHostAlloc((void **)&cu->h_stage[i], bytes, cudaHostAllocDefault));
    cu->h_stage_cap = bytes;
    return ITX_OK;
}

extern "C" int itx_scan_bam_host(itx_index *ix, const uint8_t *bam, uint64_t len, const itx_scan_opts *o,
                                 uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    int rc = check_opts(o, err); if (rc) return rc;
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    memset(&ix->prof, 0, sizeof ix->prof);
    itx_bam_header *h = itx_bam_header_parse(ix, bam, len, o->addChr, err);
    if (!h) return ITX_EFORMAT;
    uint64_t W = ix->tune_window < (256ull << 20) ? ix->tune_window : (256ull << 20);
    if (W > len) W = len;
    W = ((W + ix->tune_chunk - 1) / ix->tune_chunk) * (uint64_t)ix->tune_chunk;         /* whole chunks per copy */
    scan_ctx sc;
    if ((rc = ensure_stream_buffer(cu, len, err))) { itx_bam_header_free(h); return rc; }
    if ((rc = scan_begin(&sc, ix, h, cu->d_stream, len, o, W, err))) { itx_bam_header_free(h); return rc; }
    cudaPointerAttributes at; bool pinned = cudaPointerGetAttributes(&at, bam) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (!pinned && (rc = ensure_stage(cu, W, err))) { itx_bam_header_free(h); return rc; }
    cudaEvent_t done[2]; cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming); cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming);
    double t0 = now_ms();
    uint64_t copied = 0; int slot = 0;
    rc = ITX_OK;
    while (copied < len && rc == ITX_OK) {
        uint64_t n = len - copied < W ? len - copied : W;
        if (pinned) {
            if (cudaMemcpyAsync(cu->d_stream + copied, bam + copied, n, cudaMemcpyHostToDevice, cu->stream) != cudaSuccess) rc = ITX_ENODEV;
        } else {
            cudaEventSynchronize(done[slot]);
            memcpy(cu->h_stage[slot], bam + copied, n);
            if (cudaMemcpyAsync(cu->d_stream + copied, cu->h_stage[slot], n, cudaMemcpyHostToDevice, cu->stream) != cudaSuccess) rc = ITX_ENODEV;
            cudaEventRecord(done[slot], cu->stream); slot ^= 1;
        }
        copied += n;
        /* everything strictly before the window just copied can be scanned now */
        uint64_t k_hi = copied >= len ? sc.k_end : (copied - n) / cu->C;
        if (rc == ITX_OK && k_hi > sc.k_next) rc = scan_window(&sc, k_hi, copied, err);
    }
    if (rc == ITX_OK && sc.k_next < sc.k_end) rc = scan_window(&sc, sc.k_end, len, err);
    if (rc == ITX_OK) rc = scan_end(&sc, cnt, err);
    else if (!err[0]) snprintf(err, ITX_ERRLEN, "CUDA error while streaming: %s", cudaGetErrorString(cudaGetLastError()));
    ix->prof.h2d_bytes = len; ix->prof.h2d_ms = now_ms() - t0;
    cudaEventDestroy(done[0]); cudaEventDestroy(done[1]);
    itx_bam_header_free(h);
    return rc;
}

/* ------------------------------------------------------------------ BGZF file / memory image */
/* where the compressed bytes come from: a file descriptor (pread, no mapping and so no page faults) or memory */
typedef struct { int fd; const uint8_t *mem; uint64_t len; } itx_bgzf_src;
static int src_read(const itx_bgzf_src *S, uint64_t o0, uint64_t o1, uint8_t *dst, int nth) {
    return S->fd >= 0 ? itx_parallel_pread(S->fd, o0, o1, dst, nth) : itx_parallel_copy(S->mem, o0, o1, dst, nth);
}
/* grow a device buffer, keeping its first `keep` bytes; both streams are drained first (kernels in flight hold the old pointer) */
static int grow_device(itx_cuda *cu, void **p, uint64_t *cap, uint64_t need, uint64_t keep, const char *what, char *err) {
    if (*p && *cap >= need) return ITX_OK;
    cudaStreamSynchronize(cu->stream); cudaStreamSynchronize(cu->copy_stream);
    void *q = NULL;
    if (!keep && *p) { cudaFree(*p); *p = NULL; *cap = 0; }
    if (cudaMalloc(&q, need) != cudaSuccess) { cudaGetLastError(); snprintf(err, ITX_ERRLEN, "cannot allocate %llu bytes on the device for %s", (unsigned long long)need, what); return ITX_ENOMEM; }
    if (*p && keep && cudaMemcpy(q, *p, keep, cudaMemcpyDeviceToDevice) != cudaSuccess) { cudaFree(q); snprintf(err, ITX_ERRLEN, "device copy failed while growing %s", what); return ITX_ENODEV; }
    cudaFree(*p); *p = q; *cap = need;
    return ITX_OK;
}

/* ------------------------------------------------------------------ compressed windows: from the source towards the device */
/* The compressed bytes cross PCIe window by window (Wc bytes).  A source that is pinned host memory is handed to the copy
 * engine where it lies (no host copy at all); anything else -- a file descriptor, pageable memory -- goes through a ring of
 * pinned slots that a reader thread keeps filled ahead of the consumer (pread / memcpy by the pool's threads), so that reading
 * window w + 2 overlaps walking the block headers of window w + 1 and the DMA of window w.  A window ends in the middle of
 * a block; the cut block's bytes are moved in front of the next slot (every slot has ITX_RD_HEAD bytes of room there), so the
 * consumer always sees whole blocks without anything being read twice. */
#define ITX_RD_SLOTS 4
#define ITX_RD_HEAD 65536u
typedef struct comp_reader {
    const itx_bgzf_src *S; uint64_t begin, end, Wc; int nth, direct, device;
    uint8_t *slot[ITX_RD_SLOTS]; cudaEvent_t freed[ITX_RD_SLOTS];
    pthread_t th; int th_started; pthread_mutex_t mu; pthread_cond_t cv;
    uint64_t produced, released; int failed, stop;
} comp_reader;
static void *comp_reader_main(void *arg) {
    comp_reader *R = (comp_reader *)arg;
    cudaSetDevice(R->device);
    for (uint64_t w = 0;; w++) {
        const uint64_t o0 = R->begin + w * R->Wc;
        if (o0 >= R->end) break;
        pthread_mutex_lock(&R->mu);
        while (!R->stop && w >= R->released + ITX_RD_SLOTS) pthread_cond_wait(&R->cv, &R->mu);
        const int stop = R->stop;
        pthread_mutex_unlock(&R->mu);
        if (stop) break;
        const int sl = (int)(w % ITX_RD_SLOTS);
        cudaEventSynchronize(R->freed[sl]);                         /* the copy out of this slot's previous window is done */
        const uint64_t o1 = o0 + R->Wc < R->end ? o0 + R->Wc : R->end;
        const int rc = src_read(R->S, o0, o1, R->slot[sl] + ITX_RD_HEAD, R->nth);
        pthread_mutex_lock(&R->mu);
        if (rc != ITX_OK) R->failed = 1;
        R->produced = w + 1;
        pthread_cond_broadcast(&R->cv);
        pthread_mutex_unlock(&R->mu);
        if (rc != ITX_OK) break;
    }
    return NULL;
}
static int comp_reader_open(comp_reader *R, itx_cuda *cu, const itx_bgzf_src *S, uint64_t begin, uint64_t end, uint64_t Wc, int nth, char *err) {
    memset(R, 0, sizeof *R);
    R->S = S; R->begin = begin; R->end = end; R->Wc = Wc; R->nth = nth; R->device = cu->device;
    if (S->fd < 0) {
        cudaPointerAttributes at;
        R->direct = cudaPointerGetAttributes(&at, S->mem) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
        { const char *v = getenv("ITX_PINNED_DIRECT"); if (v && atoi(v) == 0) R->direct = 0; }      /* A/B: stage even pinned memory */
    }
    if (R->direct) return ITX_OK;
    if (cu->h_ring_cap < Wc + ITX_RD_HEAD + 64) {
        for (int i = 0; i < ITX_RD_SLOTS; i++) { if (cu->h_ring[i]) cudaFreeHost(cu->h_ring[i]); cu->h_ring[i] = NULL; }
        cu->h_ring_cap = 0;
        for (int i = 0; i < ITX_RD_SLOTS; i++) CK(cudaHostAlloc((void **)&cu->h_ring[i], Wc + ITX_RD_HEAD + 64, cudaHostAllocDefault));
        cu->h_ring_cap = Wc + ITX_RD_HEAD + 64;
    }
    for (int i = 0; i < ITX_RD_SLOTS; i++) { R->slot[i] = cu->h_ring[i]; CK(cudaEventCreateWithFlags(&R->freed[i], cudaEventDisableTiming)); }
    pthread_mutex_init(&R->mu, NULL); pthread_cond_init(&R->cv, NULL);
    if (pthread_create(&R->th, NULL, comp_reader_main, R) != 0) { snprintf(err, ITX_ERRLEN, "cannot start the reader thread"); return ITX_ENOMEM; }
    R->th_started = 1;
    return ITX_OK;
}
/* window w as the consumer sees it: *p points at file offset `cur` (<= the window's own first byte: what the window before
 * left over lies in front), *n bytes are there */
static int comp_reader_get(comp_reader *R, uint64_t w, uint64_t cur, const uint8_t **p, uint64_t *n) {
    if (R->direct) { *p = R->S->mem + cur; *n = R->end - cur < R->Wc ? R->end - cur : R->Wc; return ITX_OK; }
    const uint64_t o0 = R->begin + w * R->Wc;
    if (o0 >= R->end) { *p = R->slot[w % ITX_RD_SLOTS] + ITX_RD_HEAD - (o0 - cur); *n = o0 - cur; return ITX_OK; }      /* only the leftover */
    pthread_mutex_lock(&R->mu);
    while (R->produced <= w && !R->failed) pthread_cond_wait(&R->cv, &R->mu);
    const int failed = R->failed && R->produced <= w;
    pthread_mutex_unlock(&R->mu);
    if (failed) return ITX_EIO;
    const uint64_t o1 = o0 + R->Wc < R->end ? o0 + R->Wc : R->end;
    *p = R->slot[w % ITX_RD_SLOTS] + ITX_RD_HEAD - (o0 - cur); *n = o1 - cur;
    return ITX_OK;
}
/* the consumer is done with window w: its DMA (if any) has been enqueued on `copy`; the bytes from `cur` on were not used and go in front of the next slot */
static void comp_reader_release(comp_reader *R, uint64_t w, const uint8_t *p, uint64_t n, uint64_t used, cudaStream_t copy) {
    if (R->direct) return;
    const uint64_t left = n - used;
    const int nx = (int)((w + 1) % ITX_RD_SLOTS);
    if (left && left <= ITX_RD_HEAD) {
        cudaEventSynchronize(R->freed[nx]);                         /* the DMA that read that slot's front (ITX_RD_SLOTS - 1 windows ago) is done */
        memmove(R->slot[nx] + ITX_RD_HEAD - left, p + used, left);
    }
    cudaEventRecord(R->freed[w % ITX_RD_SLOTS], copy);
    pthread_mutex_lock(&R->mu);
    R->released = w + 1;
    pthread_cond_broadcast(&R->cv);
    pthread_mutex_unlock(&R->mu);
}
static void comp_reader_close(comp_reader *R) {
    if (R->th_started) {
        pthread_mutex_lock(&R->mu); R->stop = 1; pthread_cond_broadcast(&R->cv); pthread_mutex_unlock(&R->mu);
        pthread_join(R->th, NULL);
        pthread_mutex_destroy(&R->mu); pthread_cond_destroy(&R->cv);
    }
    if (!R->direct) for (int i = 0; i < ITX_RD_SLOTS; i++) if (R->freed[i]) { cudaEventSynchronize(R->freed[i]); cudaEventDestroy(R->freed[i]); }
}

/* the BAM header of a BGZF source, parsed on the host out of the file's first blocks (whatever part of the file the caller goes on to scan) */
static itx_bam_header *bam_header_from_src(itx_index *ix, const itx_bgzf_src *S, int addChr, int nth, char *err) {
    itx_bam_header *h = NULL; uint8_t *cbuf = NULL, *hb = NULL; itx_bgzf_block *blk = NULL;
    char e2[ITX_ERRLEN]; e2[0] = 0;
    for (uint64_t want = 1u << 20;; want *= 4) {
        const uint64_t n = want < S->len ? want : S->len;
        const uint8_t *c = S->mem;
        if (S->fd >= 0) {
            cbuf = (uint8_t *)realloc(cbuf, n + 64);
            if (!cbuf || itx_parallel_pread(S->fd, 0, n, cbuf, nth) != ITX_OK) { snprintf(err, ITX_ERRLEN, "read error at the start of the BAM file"); break; }
            c = cbuf;
        }
        uint64_t nblk = 0, total = 0;
        free(blk); blk = NULL;
        if (itx_bgzf_scan(c, n, &blk, &nblk, &total, e2) != ITX_OK) { snprintf(err, ITX_ERRLEN, "%s", e2); break; }
        bool stop = nblk == 0;                                 /* not a BGZF file at all */
        for (uint64_t nb = 1; nb <= nblk && !h && !stop; nb = nb < 4 ? nb + 1 : nb * 2) {
            const uint64_t n1 = nb < nblk ? nb : nblk, ub = blk[n1 - 1].uoff + blk[n1 - 1].isize;
            hb = (uint8_t *)realloc(hb, ub + 64);
            if (!hb || itx_bgzf_inflate_range(c, blk, 0, n1, hb, nth, NULL) != ITX_OK) { snprintf(e2, ITX_ERRLEN, "BGZF inflate failed in the header blocks"); stop = true; break; }
            h = itx_bam_header_parse(ix, hb, ub, addChr, e2);
            if (!h && memcmp(hb, "BAM\1", 4) != 0) stop = true;
            if (n1 == nblk) break;
        }
        if (h || stop || n == S->len) {
            if (!h) snprintf(err, ITX_ERRLEN, "%s", e2[0] ? e2 : (nblk ? "truncated BAM header" : "invalid BAM binary header (this is not a BAM file)"));
            break;
        }
    }
    free(cbuf); free(hb); free(blk);
    return h;
}

/* what one rank of a sharded scan is told and what it reports (itx_scan_shard_file) */
typedef struct {
    int rank, nranks;
    uint64_t entry;            /* in: ITX_OFF_GUESS, or the rank-local offset of the first record (from the rank before) */
    uint64_t margin;           /* in: uncompressed bytes read past the own range for the record that straddles its end */
    uint64_t entry_rel;        /* out: the first record start the scan settled on (rank-local; NONE: it met none) */
    uint64_t exit_rel;         /* out: where the chain left the own range, relative to its end (ITX_OFF_END: the chain ended) */
    uint64_t own_bytes;        /* out: uncompressed bytes of the own blocks */
    int more_after;            /* out: there was more of the file after what was read (a chain that ended may just have run out of margin) */
    int collect;               /* in: phase 1 of -R across ranks (scan_ctx::collect); the header is then kept in cu->p1.h */
    uint64_t len;              /* out: uncompressed bytes on the device (the own range and the margin) */
} shard_io;

/* BGZF -> HBM in ONE pass, the inflate on the device.  The compressed bytes arrive window by window (above); the main
 * thread walks the block headers of each window (BSIZE at byte 16, ISIZE in the footer: bgzf.c:401-411, 471-521),
 * which gives every block its place in the uncompressed stream, and sends window and block table over PCIe on the copy
 * stream -- into a RING on the device when the file is larger than the ring (a window's place is recycled once the groups
 * that read it are done).  Blocks are handed to the device in groups: one k_inflate (Huffman decoding, literals, match
 * lists, then the match copies by the same warp) per group on one of ITX_INF_STREAMS streams, and the scan kernels follow
 * 64 MiB (the largest BAM record) behind the inflated front.  The stream's total size is only known at the end: the
 * stream buffer is sized from the first window's compression ratio and grown if that was too small.
 * sh != NULL: this is rank sh->rank of sh->nranks.  The rank owns the blocks that START in its share of the file's bytes
 * (boundaries found by itx_bgzf_find_block), a record belongs to the rank in whose blocks it starts, and the scan reads
 * on past the own range until the straddling record is whole. */
template <uint32_t LG>
static void launch_inflate(const itx_inflate_args &IA, cudaStream_t st) {
    static bool attr_set[8] = {false, false, false, false, false, false, false, false};
    if (!attr_set[LG]) { cudaFuncSetAttribute(k_inflate<LG>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); attr_set[LG] = true; }
    const uint64_t nb = (IA.nblk + (1u << LG) - 1) >> LG;
    k_inflate<LG><<<(unsigned)nb, ITX_INF_THREADS, ITX_INF_SMEM(LG), st>>>(IA);
}
static int env_int(const char *name, int dflt) { const char *v = getenv(name); return v && *v ? atoi(v) : dflt; }

static int scan_bgzf_device_inflate(itx_index *ix, const itx_bgzf_src *S, const itx_scan_opts *o, uint64_t cnt[13], char *err, int nth, shard_io *sh) {
    itx_cuda *cu = ix->cu;
    const uint64_t flen = S->len;
    int rc = ITX_OK;
    /* every stream / event call of the pipeline is checked where it is made: a failure is reported with its line, not as a later launch error */
#define EV(call) do { const cudaError_t e_ = (call); if (e_ != cudaSuccess && rc == ITX_OK) { snprintf(err, ITX_ERRLEN, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); rc = ITX_ENODEV; } } while (0)
    const bool timing = getenv("ITX_TIMING") != NULL; const double tm0 = now_ms();
    uint64_t Wc = 64ull << 20;                               /* compressed bytes per window */
    { const int mb = env_int("ITX_COMP_WINDOW_MB", 0); if (mb > 0) Wc = (uint64_t)mb << 20; }
    if (Wc > flen) Wc = flen;
    if (Wc < (1u << 20)) Wc = 1u << 20;
    cudaEvent_t copied = NULL, begin_ev = NULL;
    enum { MAXW = 256 }; cudaEvent_t *wev = NULL; int nw = 0;
    itx_bgzf_block *blk = NULL; uint64_t *foff = NULL, *babs = NULL; uint64_t nblk = 0, blk_cap = 0, total = 0;      /* per block: file offset, absolute (ever-growing) ring position */
    itx_bam_header *h = NULL;
    scan_ctx sc; bool begun = false;
    comp_reader R; bool reader_open = false;
    double inflate_ms = 0, wall0 = now_ms();
    /* launched groups, oldest first: where their compressed bytes start in the ring (absolute, ever-growing position) and the event slot that says they are done */
    enum { GQ = 64 }; uint64_t g_abs[GQ]; uint64_t g_waited = 0;
    do {
        /* ---- this rank's share of the file */
        uint64_t r_begin = 0, r_end = flen;
        const bool sharded = sh && sh->nranks > 1;
        if (sh) { sh->entry_rel = ITX_OFF_NONE; sh->exit_rel = ITX_OFF_NONE; sh->own_bytes = 0; sh->more_after = 0; }
        if (sharded) {
            r_begin = flen / (uint64_t)sh->nranks * (uint64_t)sh->rank; r_end = sh->rank + 1 == sh->nranks ? flen : flen / (uint64_t)sh->nranks * (uint64_t)(sh->rank + 1);
            if (sh->rank > 0) {
                /* the first block that starts at or after r_begin (a block is at most 64 KiB long) */
                uint64_t probe = 3u << 16; int64_t at = -1;
                uint8_t *pb = NULL;
                for (; at < 0; probe *= 4) {
                    const uint64_t n = flen - r_begin < probe ? flen - r_begin : probe;
                    const uint8_t *c = S->mem ? S->mem + r_begin : NULL;
                    if (S->fd >= 0) { pb = (uint8_t *)realloc(pb, n + 64); if (!pb || itx_parallel_pread(S->fd, r_begin, r_begin + n, pb, nth) != ITX_OK) { rc = ITX_EIO; break; } c = pb; }
                    at = itx_bgzf_find_block(c, n, r_begin + n == flen);
                    if (at < 0 && (r_begin + n == flen || probe > (64u << 20))) break;
                }
                free(pb);
                if (rc) { snprintf(err, ITX_ERRLEN, "read error in the BAM file at offset %llu", (unsigned long long)r_begin); break; }
                r_begin = at < 0 ? flen : r_begin + (uint64_t)at;          /* no block starts in the rest of the file: nothing to own */
            }
            if (r_end < r_begin) r_end = r_begin;
        }
        if (!(h = bam_header_from_src(ix, S, o->addChr, nth, err))) { rc = ITX_EFORMAT; break; }
        if ((rc = comp_reader_open(&R, cu, S, r_begin, flen, Wc, nth, err))) break;
        if (timing) fprintf(stderr, "[itx timing] header parsed, reader open (pinned slots) at %.1f ms\n", now_ms() - tm0);
        reader_open = true;
        /* the compressed bytes on the device: the whole range when it fits the ring, else a ring */
        uint64_t ring_cap = (uint64_t)env_int("ITX_COMP_RING_MB", 8192) << 20;
        if (ring_cap < 4 * (Wc + ITX_RD_HEAD)) ring_cap = 4 * (Wc + ITX_RD_HEAD);
        { const uint64_t whole = flen - r_begin + ITX_RD_HEAD; if (!sharded && whole < ring_cap) ring_cap = whole; else if (sharded && (r_end - r_begin) + (sh->margin + (4u << 20)) * 2 + ITX_RD_HEAD < ring_cap) ring_cap = (r_end - r_begin) + (sh->margin + (4u << 20)) * 2 + ITX_RD_HEAD; }
        if ((rc = grow_device(cu, (void **)&cu->d_comp, &cu->d_comp_cap, ring_cap + ITX_SLACK, 0, "the compressed bytes", err))) break;
        ring_cap = cu->d_comp_cap - ITX_SLACK;                /* a larger buffer left by an earlier scan is used whole */
        if (timing) fprintf(stderr, "[itx timing] compressed ring on the device (%.2f GB) at %.1f ms\n", (double)cu->d_comp_cap / 1e9, now_ms() - tm0);
        cudaEventCreateWithFlags(&copied, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&begin_ev, cudaEventDisableTiming);
        if (!cu->inf_ev) {
            cu->inf_ev = (cudaEvent_t *)calloc(2 * MAXW, sizeof(cudaEvent_t));
            for (int i = 0; cu->inf_ev && i < 2 * MAXW; i++) { if (cudaEventCreate(&cu->inf_ev[i]) != cudaSuccess) break; cu->inf_ev_made = i + 1; }
            cudaGetLastError();
        }
        wev = cu->inf_ev;
        /* a group = a run of consecutive blocks handed to the device as one k_inflate launch on one of
         * ITX_INF_STREAMS streams.  A thread needs milliseconds for its block whatever the launch size, so groups are kept
         * to a fraction of the resident threads and several are in flight: the file's copy, the inflate passes and the
         * scan of successive groups overlap.  Towards the end of the file nothing is left to hide that latency behind:
         * the last groups are smaller and run fewer blocks per warp (shorter rounds). */
        if (!cu->inf_made) {
            for (int i = 0; i < ITX_INF_STREAMS; i++) { cudaStreamCreateWithFlags(&cu->inf_stream[i], cudaStreamNonBlocking); cudaEventCreateWithFlags(&cu->inf_done[i], cudaEventDisableTiming); }
            cu->inf_made = 1;
        }
        uint64_t GROUP = 16384;                    /* 151 ms per 3.4 GB file against 158 ms at 8192 and 173 ms at 4096 (B200, round 1) */
        { const int v = env_int("ITX_INF_GROUP", 0); if (v >= 32) GROUP = (uint64_t)v / 32 * 32; }
        {   /* small files: no more slots than the file can have blocks (should a file beat the estimate, groups simply close earlier) */
            const uint64_t est = (flen - r_begin) / 2048 + 64;
            if (GROUP > est) GROUP = (est + 31) / 32 * 32;
        }
        /* smaller groups towards the end of the file were measured too (ITX_INF_TAIL_GROUP): 153 ms against 147.5 ms without them -- the
         * throughput of the inflate passes, not the latency of the last group, bounds a large file.  A group that is small anyway (a
         * small file, the last blocks of a large one) runs 8 blocks per warp: shorter rounds, lower latency per block. */
        uint64_t TAIL_GROUP = GROUP;
        { const int v = env_int("ITX_INF_TAIL_GROUP", 0); if (v >= 32) TAIL_GROUP = (uint64_t)v / 32 * 32; if (TAIL_GROUP > GROUP) TAIL_GROUP = GROUP; }
        const int LANES = env_int("ITX_INF_LANES", ITX_INF_LANES_DEFAULT), TAIL_LANES = env_int("ITX_INF_TAIL_LANES", ITX_INF_TAIL_LANES_DEFAULT);
        const uint64_t min_lanes = (uint64_t)(LANES < TAIL_LANES ? LANES : TAIL_LANES) >= 8 ? (uint64_t)(LANES < TAIL_LANES ? LANES : TAIL_LANES) : 8;
        const uint64_t tab_warps = (GROUP + min_lanes - 1) / min_lanes * ITX_INF_STREAMS;       /* warps whose long-code symbol arrays may be live at once */
        if (!cu->d_tabs || cu->d_tabs_threads < tab_warps * 32) {
            cudaStreamSynchronize(cu->stream);
            cudaFree(cu->d_tabs); cu->d_tabs = NULL;
            if (cudaMalloc((void **)&cu->d_tabs, tab_warps * 32 * ITX_T_CELLS * 2) != cudaSuccess) { cudaGetLastError(); snprintf(err, ITX_ERRLEN, "cannot allocate the inflate tables"); rc = ITX_ENOMEM; break; }
            cu->d_tabs_threads = tab_warps * 32;
        }
        const uint64_t tab_stride = cu->d_tabs_threads / ITX_INF_STREAMS * ITX_T_CELLS;           /* cells per stream */
        int lz_ctas = 1;
        /* the second pass (match copies).  ITX_LZ=2, the default: inside k_inflate, by the warp that decoded the blocks (itx_lzw_resolve:
         * windows of the block in the warp's own shared memory, no second kernel).  ITX_LZ=0: k_lz_resolve, a CTA per block with the
         * whole block in 64 KiB of shared memory -- its CTAs displace the decoding warps (20 KiB each), so the two passes ran one after
         * the other in effect (140 ms per 3.4 GB file against 113 ms).  ITX_LZ=1: k_lz_jump (pointer jumping over the whole block,
         * 192 KiB per CTA: it waits for every k_inflate warp of an SM to finish) */
        const int lz_mode = env_int("ITX_LZ", 2);
        const bool lz_jump = lz_mode == 1, lz_fused = lz_mode == 2;
        cudaFuncSetAttribute(k_lz_jump, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ITX_LZ2_SMEM);
        cudaFuncSetAttribute(k_lz_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ITX_LZ_SMEM);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&lz_ctas, k_lz_resolve, ITX_LZ_THREADS, ITX_LZ_SMEM);
        if (lz_ctas < 1) lz_ctas = 1;
        if (!cu->d_mpl || cu->d_m_slots < GROUP * ITX_INF_STREAMS) {
            cudaFree(cu->d_mpl); cudaFree(cu->d_md); cudaFree(cu->d_mn); cu->d_mpl = NULL; cu->d_md = NULL; cu->d_mn = NULL;
            const uint64_t ns = GROUP * ITX_INF_STREAMS;
            cudaStreamSynchronize(cu->stream);
            if (cudaMalloc((void **)&cu->d_mpl, ns * ITX_M_WORST * 4) != cudaSuccess || cudaMalloc((void **)&cu->d_md, ns * ITX_M_WORST * 2) != cudaSuccess ||
                cudaMalloc((void **)&cu->d_mn, ns * 4) != cudaSuccess) { cudaGetLastError(); snprintf(err, ITX_ERRLEN, "cannot allocate the match lists (%llu blocks)", (unsigned long long)ns); rc = ITX_ENOMEM; break; }
            cu->d_m_slots = ns;
        }
        const uint64_t m_stride = cu->d_m_slots / ITX_INF_STREAMS;
        if (timing) fprintf(stderr, "[itx timing] inflate tables and match lists (%.2f GB) at %.1f ms\n", (double)cu->d_m_slots * ITX_M_WORST * 6 / 1e9, now_ms() - tm0);
        const uint64_t MARGIN = (64ull << 20) + 65536;      /* a record is at most 2^26 bytes long: chunks this far behind the inflated front are safe to scan */
        uint64_t cur = r_begin, gb0 = 0, n_groups = 0, cabs = 0, own_total = ~0ull, typical_group_bytes = GROUP * 24576ull;
        bool ended = false, own_closed = false;
        /* hand blocks [gb0, upto) to the device; everything they need has been enqueued on the copy stream before `copied` was recorded */
        auto launch_group = [&](uint64_t upto, bool tail) {
            const int gs = (int)(n_groups % ITX_INF_STREAMS); cudaStream_t st = cu->inf_stream[gs];
            EV(cudaStreamWaitEvent(st, copied, 0));
            if (n_groups == 0) EV(cudaStreamWaitEvent(st, begin_ev, 0));           /* the status words are zeroed on the scan stream */
            itx_inflate_args IA; IA.file = cu->d_comp; IA.blk = cu->d_blk; IA.b0 = gb0; IA.nblk = upto - gb0; IA.out = cu->d_stream; IA.status = cu->D.status;
            IA.tabs = cu->d_tabs + (size_t)gs * tab_stride;
            IA.m_pl = cu->d_mpl + (size_t)gs * m_stride * ITX_M_WORST; IA.m_d = cu->d_md + (size_t)gs * m_stride * ITX_M_WORST; IA.m_n = cu->d_mn + (size_t)gs * m_stride; IA.m_cap = ITX_M_WORST; IA.fuse_lz = lz_fused ? 1u : 0u;
            const bool ev_ok = 2 * nw + 1 < cu->inf_ev_made;
            if (ev_ok) EV(cudaEventRecord(wev[2 * nw], st));
            const int lanes = tail ? TAIL_LANES : LANES;
            if (lanes <= 8) launch_inflate<3>(IA, st); else if (lanes <= 16) launch_inflate<4>(IA, st); else launch_inflate<5>(IA, st);
            EV(cudaGetLastError());
            if (lz_fused) {
            } else if (lz_jump) {
                uint64_t lzb = IA.nblk, lzmax = (uint64_t)cu->sm_count; if (lzb > lzmax) lzb = lzmax;
                k_lz_jump<<<(unsigned)lzb, ITX_LZ2_THREADS, ITX_LZ2_SMEM, st>>>(IA);
            } else {
                uint64_t lzb = IA.nblk, lzmax = (uint64_t)cu->sm_count * (uint64_t)lz_ctas; if (lzb > lzmax) lzb = lzmax;
                k_lz_resolve<<<(unsigned)lzb, ITX_LZ_THREADS, ITX_LZ_SMEM, st>>>(IA);
            }
            EV(cudaGetLastError());
            if (ev_ok) { EV(cudaEventRecord(wev[2 * nw + 1], st)); nw++; }
            EV(cudaEventRecord(cu->inf_done[gs], st));
            EV(cudaStreamWaitEvent(cu->stream, cu->inf_done[gs], 0));          /* the scan stream has now waited for every group so far */
            sc.n_launch += 2;
            {   /* an event of its own per group (GQ of them, reused round robin) for the ring: a window may only land on bytes whose groups are done */
                const int gi = (int)(n_groups % GQ);
                if (!cu->grp_ev[gi]) cudaEventCreateWithFlags(&cu->grp_ev[gi], cudaEventDisableTiming);
                else if (n_groups >= GQ) cudaEventSynchronize(cu->grp_ev[gi]);           /* GQ groups back: long done */
                EV(cudaEventRecord(cu->grp_ev[gi], st));
                g_abs[gi] = babs[gb0];                                      /* where the group's first block lies */
            }
            gb0 = upto; n_groups++;
        };
        for (uint64_t w = 0; !ended && rc == ITX_OK; w++) {
            const uint8_t *hs = NULL; uint64_t n = 0;
            if (comp_reader_get(&R, w, cur, &hs, &n) != ITX_OK) { snprintf(err, ITX_ERRLEN, "read error in the BAM file at offset %llu", (unsigned long long)cur); rc = ITX_EIO; break; }
            const bool more_in_file = cur + n < flen;
            /* the blocks that lie completely inside this window */
            const uint64_t nb_before = nblk; uint64_t off = 0;
            std::vector<uint64_t> closes;                                              /* groups that fill up inside this window end at these block counts */
            uint64_t g_first = gb0;                                                    /* first block of the group being filled */
            for (;;) {
                if (off + 18 > n) { if (!more_in_file) ended = true; break; }
                const uint8_t *hd = hs + off;
                if (!itx_bgzf_header_ok(hd)) { ended = true; break; }                  /* a bad header ends the stream silently (bgzf_read) */
                const uint32_t bsize = ((uint32_t)hd[16] | (uint32_t)hd[17] << 8) + 1;
                if (bsize < 26) { ended = true; break; }
                if (off + bsize > n) { if (!more_in_file) ended = true; break; }      /* continues in the next window, or the file is cut short */
                uint32_t isize; memcpy(&isize, hd + bsize - 4, 4);
                if (isize == 0 || isize > 65536) { ended = true; break; }              /* an empty block ends the data (bgzf.c:539-546) */
                if (sharded && !own_closed && cur + off >= r_end) { own_closed = true; own_total = total; }
                if (own_closed && total - own_total >= sh->margin) { ended = true; sh->more_after = 1; break; }      /* the straddling record has its room */
                if (nblk == blk_cap) { blk_cap = blk_cap ? blk_cap * 2 : 4096; blk = (itx_bgzf_block *)realloc(blk, sizeof(itx_bgzf_block) * blk_cap); foff = (uint64_t *)realloc(foff, 8 * blk_cap); babs = (uint64_t *)realloc(babs, 8 * blk_cap); }
                blk[nblk].coff = off; blk[nblk].csize = bsize; blk[nblk].isize = isize; blk[nblk].uoff = total; foff[nblk] = cur + off;
                nblk++; total += isize; off += bsize;
                /* near the end of the file (or of the own range) groups close early */
                const uint64_t left_c = (sharded && !own_closed ? r_end : flen) - (cur + off < (sharded && !own_closed ? r_end : flen) ? cur + off : (sharded && !own_closed ? r_end : flen));
                const uint64_t G = left_c < typical_group_bytes ? TAIL_GROUP : GROUP;
                if (nblk - g_first >= G) { closes.push_back(nblk); g_first = nblk; }
            }
            if (off == 0 && !ended && n >= Wc) ended = true;                           /* no progress is possible */
            if (!begun) {
                /* first guess of the stream size: this window's ratio over this rank's share of the file, with a margin */
                uint64_t guess = total;
                if (!ended) {
                    const uint64_t share = (sharded ? r_end : flen) - r_begin;
                    guess = (uint64_t)((double)share * ((double)total / (double)(off ? off : 1)) * 1.08) + (64ull << 20) + (sharded ? sh->margin + (1u << 20) : 0);
                    if (!(cu->d_stream && cu->d_stream_cap >= guess + ITX_SLACK)) {
                        size_t fr = 0, tot = 0; cudaMemGetInfo(&fr, &tot);
                        const uint64_t room = (uint64_t)fr + (cu->d_stream ? cu->d_stream_cap : 0);      /* the old buffer is released first */
                        if (guess + ITX_SLACK + (1ull << 30) > room && room > (2ull << 30)) guess = room - (1ull << 30) - ITX_SLACK;
                    }
                }
                if (!(cu->d_stream && cu->d_stream_cap >= guess + ITX_SLACK)) { cudaStreamSynchronize(cu->stream); cudaFree(cu->d_stream); cu->d_stream = NULL; cu->d_stream_cap = 0; }
                if ((rc = grow_device(cu, (void **)&cu->d_stream, &cu->d_stream_cap, guess + ITX_SLACK, 0, "the uncompressed stream", err))) break;
                const uint64_t carry0 = (sharded && sh->rank > 0) ? sh->entry : ITX_CARRY_HEADER;
                if ((rc = scan_begin(&sc, ix, h, cu->d_stream, 1ull << 62, o, guess < ix->tune_window ? guess : ix->tune_window, err, 0, carry0))) break;
                if (sh && sh->collect) { sc.collect = 1; sc.fused = 0; }
                begun = true;
                EV(cudaEventRecord(begin_ev, cu->stream));
                if (off) typical_group_bytes = (uint64_t)((double)GROUP * (double)off / (double)(nblk ? nblk : 1));
                if (timing) fprintf(stderr, "[itx timing] first window read, header parsed, buffers ready at %.1f ms\n", now_ms() - tm0);
            }
            if (total + ITX_SLACK > cu->d_stream_cap) {
                /* the guess was too small: grow, keeping what has been inflated (everything before the open group) */
                const uint64_t want = total + total / 2 + (256ull << 20);
                if ((rc = grow_device(cu, (void **)&cu->d_stream, &cu->d_stream_cap, want + ITX_SLACK, gb0 < nblk ? blk[gb0].uoff : total, "the uncompressed stream", err))) break;
                sc.b = cu->d_stream;
            }
            if (nblk > cu->d_blk_cap) {
                const uint64_t want = nblk * 2 + 65536;
                void *pb = cu->d_blk; uint64_t capb = cu->d_blk_cap * sizeof(itx_bgzf_block);
                rc = grow_device(cu, &pb, &capb, want * sizeof(itx_bgzf_block), nb_before * sizeof(itx_bgzf_block), "the block table", err);
                cu->d_blk = (itx_bgzf_block *)pb; cu->d_blk_cap = capb / sizeof(itx_bgzf_block);
                if (rc) break;
            }
            if (off) {
                /* the window's place in the ring; whatever lies there belongs to groups that must be done first */
                if (cabs % ring_cap + off > ring_cap) cabs += ring_cap - cabs % ring_cap;          /* not across the ring's end */
                for (uint64_t k = nb_before; k < nblk; k++) babs[k] = cabs + blk[k].coff;           /* (coff is still relative to the window) */
                if (cabs + off > ring_cap) {
                    const uint64_t low = cabs + off - ring_cap;                                      /* absolute positions below this one are overwritten */
                    if (gb0 < nb_before && babs[gb0] < low) launch_group(nb_before, false);          /* the open group itself is in the way: out it goes */
                    if (g_waited + GQ < n_groups) g_waited = n_groups - GQ;                         /* older ones were waited for on the host */
                    while (g_waited < n_groups && g_abs[g_waited % GQ] < low) { EV(cudaStreamWaitEvent(cu->copy_stream, cu->grp_ev[g_waited % GQ], 0)); g_waited++; }
                }
                const uint64_t cpos = cabs % ring_cap;
                for (uint64_t k = nb_before; k < nblk; k++) blk[k].coff += cpos;
                if (cudaMemcpyAsync(cu->d_comp + cpos, hs, off, cudaMemcpyHostToDevice, cu->copy_stream) != cudaSuccess ||
                    cudaMemcpyAsync(cu->d_blk + nb_before, blk + nb_before, (nblk - nb_before) * sizeof(itx_bgzf_block), cudaMemcpyHostToDevice, cu->copy_stream) != cudaSuccess) { rc = ITX_ENODEV; break; }
                cabs += off;
            }
            EV(cudaEventRecord(copied, cu->copy_stream));
            comp_reader_release(&R, w, hs, n, off, cu->copy_stream);
            cur += off;
            if (own_closed) sc.own = own_total;
            for (size_t k = 0; k < closes.size(); k++) if (closes[k] > gb0) launch_group(closes[k], closes[k] - gb0 <= 4096);
            if (ended && nblk > gb0) launch_group(nblk, nblk - gb0 <= 4096);
            if (!closes.empty() && !ended) {
                const uint64_t front = gb0 ? blk[gb0 - 1].uoff + blk[gb0 - 1].isize : 0;          /* what the groups launched so far inflate */
                uint64_t k_hi = front > MARGIN ? (front - MARGIN) / cu->C : 0;
                if (own_closed) { const uint64_t k_own = (own_total + cu->C - 1) / cu->C; if (k_hi > k_own) k_hi = k_own; }
                if (k_hi > sc.k_next) rc = scan_window(&sc, k_hi, front, err);
            }
        }
        if (rc != ITX_OK) break;
        if (!begun) { snprintf(err, ITX_ERRLEN, "invalid BAM binary header (this is not a BAM file)"); rc = ITX_EFORMAT; break; }
        if (!own_closed) own_total = total;
        sc.len = total; sc.own = own_total;
        {
            const uint64_t first = sc.carry0 >= ITX_OFF_GUESS ? 0 : sc.carry0;
            sc.k_end = own_total > first ? (own_total + cu->C - 1) / cu->C : sc.k_first;
        }
        if (sc.k_next < sc.k_end) rc = scan_window(&sc, sc.k_end, total, err);
        if (timing) fprintf(stderr, "[itx timing] file read, copies and kernels enqueued at %.1f ms (%llu blocks, %llu bytes)\n", now_ms() - tm0, (unsigned long long)nblk, (unsigned long long)total);
        if (rc == ITX_OK) rc = scan_end(&sc, cnt, err);
        if (timing) fprintf(stderr, "[itx timing] device done at %.1f ms\n", now_ms() - tm0);
        if (rc == ITX_OK) {
            uint32_t st[8];
            if (cudaMemcpy(st, cu->D.status, sizeof st, cudaMemcpyDeviceToHost) == cudaSuccess && st[5]) {
                snprintf(err, ITX_ERRLEN, "BGZF inflate failed on %u block(s), e.g. block %u at compressed offset %llu", st[5], st[6], (unsigned long long)(st[6] < nblk ? foff[st[6]] : 0));
                rc = ITX_EFORMAT;
            }
        }
        if (rc == ITX_OK && sh) {
            sh->own_bytes = own_total; sh->len = total;
            sh->entry_rel = sc.k_first == sc.k_end && sc.carry0 == ITX_OFF_GUESS ? ITX_OFF_NONE : sc.entry_out;
            sh->exit_rel = sc.carry_out >= ITX_OFF_GUESS ? (sc.carry_out == ITX_OFF_GUESS ? ITX_OFF_NONE : sc.carry_out) : (sc.carry_out >= own_total ? sc.carry_out - own_total : 0);
        }
        if (timing) for (int i = 0; i < nw; i++) { float a = 0, b = 0; cudaEventElapsedTime(&a, wev[0], wev[2 * i]); cudaEventElapsedTime(&b, wev[0], wev[2 * i + 1]); fprintf(stderr, "[itx timing] inflate group %d: %.1f .. %.1f ms after the first launch\n", i, a, b); }
        /* groups overlap: report the span from the first group's launch to the last group's end */
        for (int i = 0; i < nw; i++) { float ms = 0; if (cudaEventElapsedTime(&ms, wev[0], wev[2 * i + 1]) == cudaSuccess && ms > inflate_ms) inflate_ms = ms; }
    } while (0);
    if (rc != ITX_OK) { cudaStreamSynchronize(cu->stream); cudaStreamSynchronize(cu->copy_stream); if (!err[0]) snprintf(err, ITX_ERRLEN, "CUDA error while streaming: %s", cudaGetErrorString(cudaGetLastError())); }
    ix->prof.h2d_bytes = reader_open ? (nblk ? foff[nblk - 1] + blk[nblk - 1].csize - foff[0] : 0) : 0; ix->prof.h2d_ms = now_ms() - wall0; ix->prof.inflate_ms = inflate_ms; ix->prof.inflate_threads = 0;   /* 0 threads: inflate_ms is device time, first k_inflate launch to last k_lz_resolve end */
    if (rc != ITX_OK && cu->inf_made) for (int i = 0; i < ITX_INF_STREAMS; i++) cudaStreamSynchronize(cu->inf_stream[i]);
    if (reader_open) { cudaStreamSynchronize(cu->copy_stream); comp_reader_close(&R); }
    if (copied) cudaEventDestroy(copied);
    if (begin_ev) cudaEventDestroy(begin_ev);
    free(blk); free(foff); free(babs);
    if (rc == ITX_OK && sh && sh->collect) { itx_bam_header_free(cu->p1.h); cu->p1.h = h; }
    else itx_bam_header_free(h);
    return rc;
}
#undef EV

static bool inflate_on_host(void) { const char *m = getenv("ITX_INFLATE"); return m && strcmp(m, "host") == 0; }   /* A/B switch: zlib on the host threads */
static int scan_bgzf_host_inflate(itx_index *ix, const uint8_t *bgzf, uint64_t flen, const itx_scan_opts *o, uint64_t cnt[13], char *err, int nth);
static int inflate_thread_count(const itx_index *ix) {
    int nth = ix->tune_threads > 0 ? ix->tune_threads : (int)sysconf(_SC_NPROCESSORS_ONLN);
    if (nth < 1) nth = 1;
    if (nth > 256) nth = 256;
    return nth;
}

extern "C" int itx_scan_bgzf_memory(itx_index *ix, const uint8_t *bgzf, uint64_t flen, const itx_scan_opts *o,
                                    uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    int rc = check_opts(o, err); if (rc) return rc;
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    memset(&ix->prof, 0, sizeof ix->prof);
    const int nth = inflate_thread_count(ix);
    if (inflate_on_host()) return scan_bgzf_host_inflate(ix, bgzf, flen, o, cnt, err, nth);
    itx_bgzf_src S; S.fd = -1; S.mem = bgzf; S.len = flen;
    return scan_bgzf_device_inflate(ix, &S, o, cnt, err, nth, NULL);
}

/* the A/B path: block table from a walk over the whole image, zlib on the host threads, uncompressed windows over PCIe */
static int scan_bgzf_host_inflate(itx_index *ix, const uint8_t *bgzf, uint64_t flen, const itx_scan_opts *o, uint64_t cnt[13], char *err, int nth) {
    itx_cuda *cu = ix->cu;
    int rc;
    itx_bgzf_block *blk = NULL; uint64_t nblk = 0, total = 0;
    if ((rc = itx_bgzf_scan(bgzf, flen, &blk, &nblk, &total, err))) return rc;
    if (total < 12) { free(blk); snprintf(err, ITX_ERRLEN, "invalid BAM binary header (this is not a BAM file)"); return ITX_EFORMAT; }
    /* windows of whole BGZF blocks, about W uncompressed bytes each, inflated straight into pinned memory */
    uint64_t W = ix->tune_window < (64ull << 20) ? ix->tune_window : (64ull << 20);
    if (W > total) W = total;
    if (W < 65536) W = 65536;
    if ((rc = ensure_stream_buffer(cu, total, err)) || (rc = ensure_stage(cu, W + 65536, err))) { free(blk); return rc; }
    cudaEvent_t done[2]; cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming); cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming);
    itx_bam_header *h = NULL; scan_ctx sc; bool begun = false;
    uint8_t *hdr_copy = NULL; uint64_t hdr_have = 0;
    double t0 = now_ms(), busy_total = 0;
    uint64_t b = 0, copied = 0; int slot = 0;
    while (b < nblk && rc == ITX_OK) {
        uint64_t b1 = b, ubytes = 0;
        while (b1 < nblk && ubytes + blk[b1].isize <= W) { ubytes += blk[b1].isize; b1++; }
        if (b1 == b) { b1 = b + 1; ubytes = blk[b].isize; }
        cudaEventSynchronize(done[slot]);
        double busy = 0;
        rc = itx_bgzf_inflate_range(bgzf, blk, b, b1, cu->h_stage[slot], nth, &busy);
        busy_total += busy;
        if (rc) { snprintf(err, ITX_ERRLEN, "BGZF inflate failed near compressed offset %llu", (unsigned long long)blk[b].coff); break; }
        if (!begun) {
            /* the BAM header may span several windows: gather until it parses */
            hdr_copy = (uint8_t *)realloc(hdr_copy, hdr_have + ubytes); memcpy(hdr_copy + hdr_have, cu->h_stage[slot], ubytes); hdr_have += ubytes;
            char e2[ITX_ERRLEN];
            h = itx_bam_header_parse(ix, hdr_copy, hdr_have, o->addChr, e2);
            if (h) {
                if ((rc = scan_begin(&sc, ix, h, cu->d_stream, total, o, W + 65536, err))) break;
                begun = true; free(hdr_copy); hdr_copy = NULL;
            } else if (b1 == nblk || memcmp(hdr_copy, "BAM\1", 4) != 0) { memcpy(err, e2, ITX_ERRLEN); rc = ITX_EFORMAT; break; }
        }
        if (cudaMemcpyAsync(cu->d_stream + copied, cu->h_stage[slot], ubytes, cudaMemcpyHostToDevice, cu->stream) != cudaSuccess) { rc = ITX_ENODEV; break; }
        cudaEventRecord(done[slot], cu->stream); slot ^= 1;
        uint64_t before = copied; copied += ubytes; b = b1;
        if (begun) {
            uint64_t k_hi = b >= nblk ? sc.k_end : before / cu->C;
            if (k_hi > sc.k_next) rc = scan_window(&sc, k_hi, copied, err);
        }
    }
    if (rc == ITX_OK && !begun) { snprintf(err, ITX_ERRLEN, "truncated BAM header"); rc = ITX_EFORMAT; }
    if (rc == ITX_OK && sc.k_next < sc.k_end) rc = scan_window(&sc, sc.k_end, total, err);
    if (rc == ITX_OK) rc = scan_end(&sc, cnt, err);
    else { cudaStreamSynchronize(cu->stream); if (!err[0]) snprintf(err, ITX_ERRLEN, "CUDA error while streaming: %s", cudaGetErrorString(cudaGetLastError())); }
    ix->prof.h2d_bytes = total; ix->prof.h2d_ms = now_ms() - t0; ix->prof.inflate_ms = busy_total; ix->prof.inflate_threads = nth;
    cudaEventDestroy(done[0]); cudaEventDestroy(done[1]);
    free(hdr_copy); free(blk); itx_bam_header_free(h);
    return rc;
}

static int scan_one_file(itx_index *ix, const char *path, const itx_scan_opts *o, uint64_t cnt[13], char *err) {
    if (o->isSam) {
        /* -S: the text is turned into the BAM records samtools would have built, then takes the same path */
        uint8_t *bam = NULL; uint64_t len = 0;
        int rcs = itx_sam_to_bam_stream(path, &bam, &len, err);
        if (rcs == ITX_OK) rcs = itx_scan_bam_host(ix, bam, len, o, cnt, err);
        free(bam);
        return rcs;
    }
    int fd = open(path, O_RDONLY);
    if (fd < 0) { snprintf(err, ITX_ERRLEN, "Error\n[bam file %s: %s]", path, strerror(errno)); return ITX_EIO; }
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); snprintf(err, ITX_ERRLEN, "Error\n[bam file %s is empty or unreadable]", path); return ITX_EIO; }
    int rc;
    if (inflate_on_host()) {
        void *m = mmap(NULL, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        close(fd);
        if (m == MAP_FAILED) { snprintf(err, ITX_ERRLEN, "mmap(%s): %s", path, strerror(errno)); return ITX_EIO; }
        madvise(m, (size_t)st.st_size, MADV_SEQUENTIAL);
        rc = itx_scan_bgzf_memory(ix, (const uint8_t *)m, (uint64_t)st.st_size, o, cnt, err);
        munmap(m, (size_t)st.st_size);
        return rc;
    }
    if ((rc = check_opts(o, err))) { close(fd); return rc; }
    if (cudaSetDevice(ix->cu->device) != cudaSuccess) { close(fd); snprintf(err, ITX_ERRLEN, "cudaSetDevice failed"); return ITX_ENODEV; }
    memset(&ix->prof, 0, sizeof ix->prof);
    posix_fadvise(fd, 0, 0, POSIX_FADV_SEQUENTIAL);
    itx_bgzf_src S; S.fd = fd; S.mem = NULL; S.len = (uint64_t)st.st_size;
    rc = scan_bgzf_device_inflate(ix, &S, o, cnt, err, inflate_thread_count(ix), NULL);
    close(fd);
    return rc;
}

/* the single-file twin (samFile2nodupRepbedFileNew, generic.c:343: what `filter` calls): the argument is ONE path, commas and all */
extern "C" int itx_scan_alignment_file(itx_index *ix, const char *path, const itx_scan_opts *o, uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    int rc = ITX_OK;
    if ((o->outbed || o->outbed_unique) && (rc = ordered_open_files(ix->cu, o, err))) return rc;
    ix->cu->bed_owner = (o->outbed || o->outbed_unique) ? 1 : 0;
    rc = scan_one_file(ix, path, o, cnt, err);
    ix->prof.n_records = ix->cnt[0] + ix->cnt[1]; ix->prof.n_fragments = ix->cnt[6];
    ordered_close_files(ix->cu);
    return rc;
}

extern "C" int itx_scan_alignments(itx_index *ix, const char *bam_list, const itx_scan_opts *o, uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    char *list = strdup(bam_list), *save = NULL; int rc = ITX_OK, nfile = 0;
    itx_profile total; memset(&total, 0, sizeof total);
    /* the bed files span the whole list (generic.c:716-727): opened here, appended to by every file's scan */
    if ((o->outbed || o->outbed_unique) && (rc = ordered_open_files(ix->cu, o, err))) { free(list); return rc; }
    ix->cu->bed_owner = (o->outbed || o->outbed_unique) ? 1 : 0;
    for (char *tok = strtok_r(list, ",", &save); tok && rc == ITX_OK; tok = strtok_r(NULL, ",", &save)) {
        if (++nfile > 100) break;                       /* the reference's row[100] */
        rc = scan_one_file(ix, tok, o, cnt, err);
        total.decode_ms += ix->prof.decode_ms; total.overlap_ms += ix->prof.overlap_ms; total.total_ms += ix->prof.total_ms;
        total.h2d_ms += ix->prof.h2d_ms; total.inflate_ms += ix->prof.inflate_ms; total.stream_bytes += ix->prof.stream_bytes;
        total.h2d_bytes += ix->prof.h2d_bytes; total.d2h_bytes += ix->prof.d2h_bytes; total.n_launches += ix->prof.n_launches;
        total.n_bad_chunks += ix->prof.n_bad_chunks; total.inflate_threads = ix->prof.inflate_threads;
        total.fused = ix->prof.fused; total.n_replayed_windows += ix->prof.n_replayed_windows;
    }
    total.n_records = ix->cnt[0] + ix->cnt[1]; total.n_fragments = ix->cnt[6];
    ix->prof = total;
    ordered_close_files(ix->cu);
    free(list);
    return rc;
}

/* ------------------------------------------------------------------ results */
extern "C" int itx_sync_counts(itx_index *ix, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    const size_t ne = (size_t)ix->n_elem, ng = (size_t)(ix->subs.n + ix->fams.n + ix->clas.n), bl = (size_t)ix->bp_len;
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    cudaEventRecord(a, cu->stream);
    if (ix->stat_mode && ix->subs.n) k_finalize<<<cu->sm_count * 2, 256, 0, cu->stream>>>(cu->D, cu->d_bp, cu->d_bp_u);
    cudaEventRecord(b, cu->stream);
    unsigned long long *u64 = (unsigned long long *)malloc((cu->n_u64 ? cu->n_u64 : 1) * 8);
    CK(cudaMemcpyAsync(u64, cu->d_u64, cu->n_u64 * 8, cudaMemcpyDeviceToHost, cu->stream));
    if (!ix->bp) { ix->bp = (uint32_t *)calloc(bl + 1, 4); ix->bp_u = (uint32_t *)calloc(bl + 1, 4); ix->bp_cpg = (double *)calloc(bl + 1, 8); }
    if (!ix->el_cnt) { ix->el_cnt = (uint32_t *)calloc(ne + 1, 4); ix->el_cnt_u = (uint32_t *)calloc(ne + 1, 4); ix->el_cpg = (uint32_t *)calloc(ne + 1, 4); ix->el_cpg_score = (double *)calloc(ne + 1, 8); }
    /* only what a scan has touched since the last reset crosses PCIe: the per-locus counters belong to filter mode, the
     * CpG block to the bedGraph scan; untouched host copies are zero (or are zeroed here if an earlier sync filled them) */
    const bool el = cu->used_el != 0, cpg = cu->used_cpg != 0;
    uint64_t moved = cu->n_u64 * 8;
    if (bl) { CK(cudaMemcpyAsync(ix->bp, cu->d_bp, bl * 4, cudaMemcpyDeviceToHost, cu->stream)); CK(cudaMemcpyAsync(ix->bp_u, cu->d_bp_u, bl * 4, cudaMemcpyDeviceToHost, cu->stream)); moved += bl * 8; }
    if (ne && el) { CK(cudaMemcpyAsync(ix->el_cnt, cu->D.el_cnt, ne * 4, cudaMemcpyDeviceToHost, cu->stream)); CK(cudaMemcpyAsync(ix->el_cnt_u, cu->D.el_cnt_u, ne * 4, cudaMemcpyDeviceToHost, cu->stream)); moved += ne * 8; cu->host_el = 1; }
    else if (ne && cu->host_el) { memset(ix->el_cnt, 0, ne * 4); memset(ix->el_cnt_u, 0, ne * 4); cu->host_el = 0; }
    uint32_t *gc = (uint32_t *)calloc(ng + 1, 4); double *gs = (double *)calloc(ng + 1, 8);
    if (cpg) {
        if (ng) { CK(cudaMemcpyAsync(gc, cu->D.grp_cpg, ng * 4, cudaMemcpyDeviceToHost, cu->stream)); CK(cudaMemcpyAsync(gs, cu->D.grp_cpg_score, ng * 8, cudaMemcpyDeviceToHost, cu->stream)); }
        if (bl) CK(cudaMemcpyAsync(ix->bp_cpg, cu->D.bp_cpg, bl * 8, cudaMemcpyDeviceToHost, cu->stream));
        moved += ng * 12 + bl * 8; cu->host_cpg = 1;
    } else if (cu->host_cpg) {
        if (bl) memset(ix->bp_cpg, 0, bl * 8);
        cu->host_cpg = 0;
    }
    if (ne && cu->used_cpg_el) {       /* the per-locus CpG counters belong to cpgfilter */
        CK(cudaMemcpyAsync(ix->el_cpg, cu->D.el_cpg, ne * 4, cudaMemcpyDeviceToHost, cu->stream)); CK(cudaMemcpyAsync(ix->el_cpg_score, cu->D.el_cpg_score, ne * 8, cudaMemcpyDeviceToHost, cu->stream));
        moved += ne * 12; cu->host_cpg_el = 1;
    } else if (ne && cu->host_cpg_el) { memset(ix->el_cpg, 0, ne * 4); memset(ix->el_cpg_score, 0, ne * 8); cu->host_cpg_el = 0; }
    CK(cudaStreamSynchronize(cu->stream));
    float fm = 0; cudaEventElapsedTime(&fm, a, b); ix->prof.finalize_ms = fm; cudaEventDestroy(a); cudaEventDestroy(b);
    ix->prof.d2h_bytes += moved;
    for (int k = 0; k < 13; k++) ix->cnt[k] = u64[k];
    const unsigned long long *g = u64 + 16;
    const int32_t ns = ix->subs.n, nf = ix->fams.n, nc = ix->clas.n;
    for (int32_t i = 0; i < ns; i++) { ix->sub[i].read_count = g[2 * i]; ix->sub[i].read_count_unique = g[2 * i + 1]; ix->sub[i].cpg_count = gc[i]; ix->sub[i].cpg_score = gs[i]; }
    for (int32_t i = 0; i < nf; i++) { ix->fam[i].read_count = g[2 * (ns + i)]; ix->fam[i].read_count_unique = g[2 * (ns + i) + 1]; ix->fam[i].cpg_count = gc[ns + i]; ix->fam[i].cpg_score = gs[ns + i]; }
    for (int32_t i = 0; i < nc; i++) { ix->cla[i].read_count = g[2 * (ns + nf + i)]; ix->cla[i].read_count_unique = g[2 * (ns + nf + i) + 1]; ix->cla[i].cpg_count = gc[ns + nf + i]; ix->cla[i].cpg_score = gs[ns + nf + i]; }
    free(u64); free(gc); free(gs);
    return ITX_OK;
}

extern "C" uint64_t itx_trace_fetch(itx_index *ix, itx_trace *out, uint64_t cap) {
    itx_cuda *cu = ix->cu;
    if (!cu->d_trace) return 0;
    cudaSetDevice(cu->device);
    unsigned long long n = 0;
    cudaMemcpy(&n, cu->d_running, 8, cudaMemcpyDeviceToHost);
    if (n > cu->trace_cap) n = cu->trace_cap;
    if (n > cap) n = cap;
    cudaMemcpy(out, cu->d_trace, n * sizeof(itx_trace), cudaMemcpyDeviceToHost);
    return n;
}

extern "C" uint64_t itx_stream_fetch(itx_index *ix, uint8_t *out, uint64_t cap) {
    itx_cuda *cu = ix->cu;
    if (!cu->d_stream) return 0;
    cudaSetDevice(cu->device);
    uint64_t n = ix->prof.stream_bytes < cu->d_stream_cap ? ix->prof.stream_bytes : cu->d_stream_cap;
    if (n > cap) n = cap;
    if (n && cudaMemcpy(out, cu->d_stream, n, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}

extern "C" int itx_query_select(itx_index *ix, const char *chrom, const uint32_t *start, const uint32_t *end, int64_t n,
                                float min_cov, int32_t *sel_row, int32_t *n_hits, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    int32_t c = itx_strtab_find(&ix->chroms, chrom);
    if (c < 0 || n <= 0) { for (int64_t i = 0; i < n; i++) { sel_row[i] = -1; if (n_hits) n_hits[i] = 0; } return ITX_OK; }
    uint32_t *ds, *de; int32_t *dr, *dh;
    CK(cudaMalloc((void **)&ds, n * 4)); CK(cudaMalloc((void **)&de, n * 4)); CK(cudaMalloc((void **)&dr, n * 4)); CK(cudaMalloc((void **)&dh, n * 4));
    CK(cudaMemcpy(ds, start, n * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(de, end, n * 4, cudaMemcpyHostToDevice));
    k_query<<<(unsigned)((n + 127) / 128), 128, 0, cu->stream>>>(cu->D, c, ds, de, n, min_cov, dr, dh);
    CK(cudaStreamSynchronize(cu->stream));
    CK(cudaMemcpy(sel_row, dr, n * 4, cudaMemcpyDeviceToHost));
    if (n_hits) CK(cudaMemcpy(n_hits, dh, n * 4, cudaMemcpyDeviceToHost));
    cudaFree(ds); cudaFree(de); cudaFree(dr); cudaFree(dh);
    return ITX_OK;
}

extern "C" int itx_dev_flush_l2(itx_index *ix) {
    itx_cuda *cu = ix->cu;
    cudaSetDevice(cu->device);
    const unsigned long long n = (256ull << 20) / 4;
    if (!cu->d_flush && cudaMalloc(&cu->d_flush, n * 4) != cudaSuccess) return ITX_ENOMEM;
    k_fill_u32<<<cu->sm_count * 8, 256, 0, cu->stream>>>((uint32_t *)cu->d_flush, n, 0x5a5a5a5au);
    return cudaStreamSynchronize(cu->stream) == cudaSuccess ? ITX_OK : ITX_ENODEV;
}

/* ------------------------------------------------------------------ CpG bedGraph (cpgBedGraphOverlapRepeat) */
/* rows already parsed on the host (the lines the device left over) through k_cpg */
typedef struct { int32_t *hc, *dc; uint32_t *hs, *he, *ds, *de; double *hv, *dv; size_t cap, n; } cpg_rows;
static void cpg_rows_free(cpg_rows *R) { cudaFreeHost(R->hc); cudaFreeHost(R->hs); cudaFreeHost(R->he); cudaFreeHost(R->hv); cudaFree(R->dc); cudaFree(R->ds); cudaFree(R->de); cudaFree(R->dv); memset(R, 0, sizeof *R); }
static int cpg_rows_init(cpg_rows *R, size_t cap) {
    memset(R, 0, sizeof *R); R->cap = cap;
    if (cudaHostAlloc((void **)&R->hc, cap * 4, 0) || cudaHostAlloc((void **)&R->hs, cap * 4, 0) || cudaHostAlloc((void **)&R->he, cap * 4, 0) || cudaHostAlloc((void **)&R->hv, cap * 8, 0) ||
        cudaMalloc((void **)&R->dc, cap * 4) || cudaMalloc((void **)&R->ds, cap * 4) || cudaMalloc((void **)&R->de, cap * 4) || cudaMalloc((void **)&R->dv, cap * 8)) { cpg_rows_free(R); return ITX_ENOMEM; }
    return ITX_OK;
}
static int cpg_rows_flush(itx_index *ix, cpg_rows *R, int filter, unsigned long long *d_in_repeat) {
    itx_cuda *cu = ix->cu;
    if (!R->n) return ITX_OK;
    cudaMemcpyAsync(R->dc, R->hc, R->n * 4, cudaMemcpyHostToDevice, cu->stream); cudaMemcpyAsync(R->ds, R->hs, R->n * 4, cudaMemcpyHostToDevice, cu->stream);
    cudaMemcpyAsync(R->de, R->he, R->n * 4, cudaMemcpyHostToDevice, cu->stream); cudaMemcpyAsync(R->dv, R->hv, R->n * 8, cudaMemcpyHostToDevice, cu->stream);
    itx_cpg_args A; A.D = cu->D; A.chrom = R->dc; A.start = R->ds; A.end = R->de; A.score = R->dv; A.n = (long long)R->n; A.filter = filter; A.in_repeat = d_in_repeat;
    k_cpg<<<(unsigned)((R->n + 255) / 256), 256, 0, cu->stream>>>(A);
    R->n = 0;
    return cudaStreamSynchronize(cu->stream) == cudaSuccess ? ITX_OK : ITX_ENODEV;
}
/* one text line [s, e) the reference's way (lineFileNextReal + chopByWhite + strtol / strtod, generic.c:1069-1076):
 * 0 = blank or comment, -k = only k < 4 fields, 1 = a row was appended */
static int cpg_parse_line_host(itx_index *ix, const char *s, const char *e, cpg_rows *R) {
    while (s < e && (*s == ' ' || (*s >= 9 && *s <= 13))) s++;
    if (s >= e || *s == '#') return 0;
    char tmp[4][64]; const char *ws[20], *we[20]; int nw = 0; const char *q = s;
    while (nw < 20 && q < e) { ws[nw] = q; while (q < e && !(*q == ' ' || (*q >= 9 && *q <= 13))) q++; we[nw] = q; nw++; while (q < e && (*q == ' ' || (*q >= 9 && *q <= 13))) q++; }
    if (nw < 4) return -nw - 100;
    char *name = strndup(ws[0], (size_t)(we[0] - ws[0]));
    for (int k = 1; k < 4; k++) { size_t l = (size_t)(we[k] - ws[k]); if (l > 63) l = 63; memcpy(tmp[k], ws[k], l); tmp[k][l] = 0; }
    R->hc[R->n] = itx_strtab_find(&ix->chroms, name); free(name);
    R->hs[R->n] = (uint32_t)strtol(tmp[1], NULL, 0); R->he[R->n] = (uint32_t)strtol(tmp[2], NULL, 0); R->hv[R->n] = strtod(tmp[3], NULL);
    R->n++;
    return 1;
}

/* The bedGraph text is parsed ON THE DEVICE: host threads pread() the file window by window into pinned memory (whole
 * lines per window; a cut last line moves to the next window), the text crosses PCIe as it is and k_bedgraph finds
 * the lines, parses them and accumulates.  The host only sees what the device hands back: the first line with fewer
 * than four fields (an error, as in the reference) and the rare lines whose score needs the full strtod.
 * ITX_CPG_PARSE=host keeps the whole parse on the host (A/B). */
/* first line start at or after `at` (0 stays 0): the byte after the first line feed at or after at - 1; flen if there is none */
static int cpg_line_start(int fd, uint64_t flen, uint64_t at, uint64_t *out) {
    if (at == 0) { *out = 0; return ITX_OK; }
    char buf[65536];
    for (uint64_t o = at - 1; o < flen;) {
        const ssize_t r = pread(fd, buf, sizeof buf, (off_t)o);
        if (r <= 0) return ITX_EIO;
        const char *nl = (const char *)memchr(buf, '\n', (size_t)r);
        if (nl) { *out = o + (uint64_t)(nl - buf) + 1; return ITX_OK; }
        o += (uint64_t)r;
    }
    *out = flen;
    return ITX_OK;
}
static int scan_cpg_part(itx_index *ix, const char *bedgraph, int filter, int rank, int nranks, uint32_t *n_lines, uint32_t *n_in_repeat, char err[ITX_ERRLEN]);
extern "C" int itx_scan_cpg(itx_index *ix, const char *bedgraph, int filter, uint32_t *n_lines, uint32_t *n_in_repeat, char err[ITX_ERRLEN]) {
    return scan_cpg_part(ix, bedgraph, filter, 0, 1, n_lines, n_in_repeat, err);
}
/* a rank owns the lines that START in its share of the file's bytes */
extern "C" int itx_scan_cpg_shard(itx_index *ix, const char *bedgraph, int filter, int rank, int nranks, uint32_t *n_lines, uint32_t *n_in_repeat, char err[ITX_ERRLEN]) {
    if (rank < 0 || nranks < 1 || rank >= nranks) { if (err) snprintf(err, ITX_ERRLEN, "bad rank %d of %d", rank, nranks); return ITX_EARG; }
    return scan_cpg_part(ix, bedgraph, filter, rank, nranks, n_lines, n_in_repeat, err);
}
static int scan_cpg_part(itx_index *ix, const char *bedgraph, int filter, int rank, int nranks, uint32_t *n_lines, uint32_t *n_in_repeat, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    cu->used_cpg = 1;
    if (filter) cu->used_cpg_el = 1;
    struct stat st;
    int fd = (stat(bedgraph, &st) == 0 && S_ISDIR(st.st_mode)) ? -1 : open(bedgraph, O_RDONLY);
    if (fd < 0) { snprintf(err, ITX_ERRLEN, "Couldn't open %s , %s", bedgraph, strerror(errno)); return ITX_EIO; }
    if (fstat(fd, &st) != 0) { close(fd); snprintf(err, ITX_ERRLEN, "Couldn't open %s , %s", bedgraph, strerror(errno)); return ITX_EIO; }
    uint64_t flen = (uint64_t)st.st_size, f_begin = 0;
    if (nranks > 1) {
        uint64_t a = 0, b = flen;
        if (cpg_line_start(fd, flen, flen / (uint64_t)nranks * (uint64_t)rank, &a) != ITX_OK ||
            (rank + 1 < nranks && cpg_line_start(fd, flen, flen / (uint64_t)nranks * (uint64_t)(rank + 1), &b) != ITX_OK)) { close(fd); snprintf(err, ITX_ERRLEN, "read error in %s", bedgraph); return ITX_EIO; }
        f_begin = a; flen = b < a ? a : b;                     /* from here on `flen` is the end of this rank's part */
    }
    const bool host_parse = getenv("ITX_CPG_PARSE") && strcmp(getenv("ITX_CPG_PARSE"), "host") == 0;
    const int nth = inflate_thread_count(ix);
    const uint64_t W = 64ull << 20, CAPW = 2 * W + 4096;                   /* a window holds a cut line of the previous one in front */
    uint8_t *hbuf[2] = {NULL, NULL}, *dbuf[2] = {NULL, NULL}; uint32_t *dfall[2] = {NULL, NULL}; unsigned long long *dcnt = NULL;
    cudaEvent_t done[2] = {NULL, NULL};
    cpg_rows R; int rc = cpg_rows_init(&R, 1u << 20);
    uint64_t used[2] = {0, 0}; bool inflight[2] = {false, false};
    unsigned long long lines = 0, inrep = 0;
    const uint64_t fall_cap = CAPW / 8 + 16;
    for (int i = 0; i < 2 && rc == ITX_OK; i++) {
        if (cudaHostAlloc((void **)&hbuf[i], CAPW + 64, 0) != cudaSuccess || cudaMalloc((void **)&dbuf[i], CAPW + 64) != cudaSuccess ||
            cudaMalloc((void **)&dfall[i], fall_cap * 4) != cudaSuccess || cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess) rc = ITX_ENOMEM;
    }
    if (rc == ITX_OK && cudaMalloc((void **)&dcnt, 2 * 4 * 8 + 8) != cudaSuccess) rc = ITX_ENOMEM;
    if (rc != ITX_OK) snprintf(err, ITX_ERRLEN, "CUDA allocation failed");
    unsigned long long *d_inrep_rows = dcnt ? dcnt + 8 : NULL;             /* k_cpg's own counter */
    if (rc == ITX_OK) cudaMemsetAsync(d_inrep_rows, 0, 8, cu->stream);
    /* what window `i` left for the host: its counters, the malformed line, the lines with a hard score */
    cudaEvent_t kev[4]; for (int i = 0; i < 4; i++) cudaEventCreate(&kev[i]);
    double kernel_ms = 0;
    auto settle = [&](int i) -> int {
        if (!inflight[i]) return ITX_OK;
        inflight[i] = false;
        unsigned long long c[4];
        { float ms = 0; if (cudaEventSynchronize(kev[2 * i + 1]) == cudaSuccess && cudaEventElapsedTime(&ms, kev[2 * i], kev[2 * i + 1]) == cudaSuccess) kernel_ms += ms; }
        if (cudaEventSynchronize(done[i]) != cudaSuccess || cudaMemcpy(c, dcnt + 4 * i, sizeof c, cudaMemcpyDeviceToHost) != cudaSuccess) { snprintf(err, ITX_ERRLEN, "CUDA error in the bedGraph kernel: %s", cudaGetErrorString(cudaGetLastError())); return ITX_ENODEV; }
        lines += c[0]; inrep += c[1];
        const char *tb = (const char *)hbuf[i];
        if (c[2] != ~0ull) {
            const char *s = tb + c[2], *e = s; while (e < tb + used[i] && *e != '\n') e++;
            int k = cpg_parse_line_host(ix, s, e, &R);
            snprintf(err, ITX_ERRLEN, "file %s doesn't appear to be in bedGraph format. At least 4 fields required, got %d", bedgraph, k < 0 ? -k - 100 : 0);
            return ITX_EFORMAT;
        }
        if (c[3]) {
            uint32_t *off = (uint32_t *)malloc((size_t)c[3] * 4);
            if (cudaMemcpy(off, dfall[i], (size_t)c[3] * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { free(off); return ITX_ENODEV; }
            for (unsigned long long k = 0; k < c[3]; k++) {
                const char *s = tb + off[k], *e = s; while (e < tb + used[i] && *e != '\n') e++;
                if (cpg_parse_line_host(ix, s, e, &R) == 1) lines++;
                if (R.n == R.cap) { int r2 = cpg_rows_flush(ix, &R, filter, d_inrep_rows); if (r2) { free(off); return r2; } }
            }
            free(off);
        }
        return ITX_OK;
    };
    uint64_t fo = f_begin, carry = 0; int slot = 0;
    uint8_t *carrybuf = (uint8_t *)malloc(W + 64);
    const bool timing = getenv("ITX_TIMING") != NULL; double t_read = 0, t_settle = 0; const double t_all0 = now_ms();
    while (rc == ITX_OK && (fo < flen || carry)) {
        { const double t0 = now_ms(); rc = settle(slot); t_settle += now_ms() - t0; }      /* the slot's previous window is done with */
        if (rc) break;
        uint8_t *hb = hbuf[slot];
        if (carry) memcpy(hb, carrybuf, carry);
        const double t_r0 = now_ms();
        const uint64_t n = flen - fo < W ? flen - fo : W;
        if (n && itx_parallel_pread(fd, fo, fo + n, hb + carry, nth) != ITX_OK) { snprintf(err, ITX_ERRLEN, "read error in %s", bedgraph); rc = ITX_EIO; break; }
        fo += n; t_read += now_ms() - t_r0;
        uint64_t have = carry + n, use = have;
        if (fo < flen) {                                                   /* whole lines only; the cut one goes to the next window */
            while (use && hb[use - 1] != '\n') use--;
        }
        carry = have - use;
        if (carry > W) { snprintf(err, ITX_ERRLEN, "a line of %s is longer than %llu bytes", bedgraph, (unsigned long long)W); rc = ITX_EFORMAT; break; }
        if (carry) memcpy(carrybuf, hb + use, carry);
        if (use) {
            if (host_parse) {
                const char *s = (const char *)hb, *end = s + use;
                while (s < end && rc == ITX_OK) {
                    const char *e = (const char *)memchr(s, '\n', (size_t)(end - s)); if (!e) e = end;
                    int k = cpg_parse_line_host(ix, s, e, &R);
                    if (k < 0) { snprintf(err, ITX_ERRLEN, "file %s doesn't appear to be in bedGraph format. At least 4 fields required, got %d", bedgraph, -k - 100); rc = ITX_EFORMAT; break; }
                    if (k == 1) lines++;
                    if (R.n == R.cap) rc = cpg_rows_flush(ix, &R, filter, d_inrep_rows);
                    s = e + 1;
                }
            } else {
                used[slot] = use;
                cudaMemcpyAsync(dbuf[slot], hb, use, cudaMemcpyHostToDevice, cu->stream);
                cudaMemsetAsync(dcnt + 4 * slot, 0, 32, cu->stream); cudaMemsetAsync(dcnt + 4 * slot + 2, 0xff, 8, cu->stream);
                itx_bedgraph_args A; A.D = cu->D; A.text = dbuf[slot]; A.n = use; A.filter = filter; A.counts = dcnt + 4 * slot; A.fallback = dfall[slot]; A.fallback_cap = fall_cap;
                cudaEventRecord(kev[2 * slot], cu->stream);
                k_bedgraph<<<(unsigned)((use + ITX_BG_TILE - 1) / ITX_BG_TILE), 256, 0, cu->stream>>>(A);
                cudaEventRecord(kev[2 * slot + 1], cu->stream);
                cudaEventRecord(done[slot], cu->stream);
                inflight[slot] = true;
            }
        }
        slot ^= 1;
    }
    for (int i = 0; i < 2 && rc == ITX_OK; i++) rc = settle(i);
    if (rc == ITX_OK) rc = cpg_rows_flush(ix, &R, filter, d_inrep_rows);
    if (rc == ITX_OK) { unsigned long long x = 0; cudaMemcpy(&x, d_inrep_rows, 8, cudaMemcpyDeviceToHost); inrep += x; }
    else cudaStreamSynchronize(cu->stream);
    if (timing) fprintf(stderr, "[itx timing] bedGraph: %.1f ms in all, %.1f ms reading, %.1f ms waiting for the device\n", now_ms() - t_all0, t_read, t_settle);
    close(fd); free(carrybuf);
    for (int i = 0; i < 2; i++) { if (hbuf[i]) cudaFreeHost(hbuf[i]); cudaFree(dbuf[i]); cudaFree(dfall[i]); if (done[i]) cudaEventDestroy(done[i]); }
    cudaFree(dcnt); cpg_rows_free(&R);
    if (n_lines) *n_lines = (uint32_t)lines;
    if (n_in_repeat) *n_in_repeat = (uint32_t)inrep;
    if (rc == ITX_OK) { ix->cpg_lines += lines; ix->cpg_in_repeat += inrep; }
    for (int i = 0; i < 4; i++) cudaEventDestroy(kev[i]);
    ix->prof.cpg_kernel_ms = kernel_ms; ix->prof.h2d_bytes = flen - f_begin;
    return rc;
}

/* ------------------------------------------------------------------ NCCL (resolved at run time so the library loads without it) */
typedef struct { char internal[ITX_NCCL_ID_BYTES]; } nccl_uid;
typedef int (*fn_uid)(nccl_uid *);
typedef int (*fn_init)(void **, int, nccl_uid, int);
typedef int (*fn_allreduce)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_void)(void);
typedef int (*fn_destroy)(void *);
typedef const char *(*fn_errstr)(int);
static void *nccl_open(char *err) {
    static void *lib = NULL;
    if (lib) return lib;
    const char *names[] = {"libnccl.so.2", "libnccl.so", NULL};
    for (int i = 0; names[i] && !lib; i++) lib = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (!lib) snprintf(err, ITX_ERRLEN, "NCCL not found: %s", dlerror());
    return lib;
}
extern "C" int itx_comm_unique_id(uint8_t id[ITX_NCCL_ID_BYTES], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    void *lib = nccl_open(err); if (!lib) return ITX_ENOTSUP;
    fn_uid f = (fn_uid)dlsym(lib, "ncclGetUniqueId");
    nccl_uid u; int r = f ? f(&u) : -1;
    if (r != 0) { snprintf(err, ITX_ERRLEN, "ncclGetUniqueId failed (%d)", r); return ITX_ENODEV; }
    memcpy(id, u.internal, ITX_NCCL_ID_BYTES);
    return ITX_OK;
}
extern "C" int itx_comm_init(itx_index *ix, const uint8_t id[ITX_NCCL_ID_BYTES], int rank, int nranks, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    itx_cuda *cu = ix->cu;
    void *lib = nccl_open(err); if (!lib) return ITX_ENOTSUP;
    CK(cudaSetDevice(cu->device));
    fn_init f = (fn_init)dlsym(lib, "ncclCommInitRank");
    nccl_uid u; memcpy(u.internal, id, ITX_NCCL_ID_BYTES);
    int r = f ? f(&cu->nccl_comm, nranks, u, rank) : -1;
    if (r != 0) { snprintf(err, ITX_ERRLEN, "ncclCommInitRank failed (%d)", r); return ITX_ENODEV; }
    cu->nccl_lib = lib; cu->rank = rank; cu->nranks = nranks;
    return ITX_OK;
}
/* ONE grouped allreduce(sum) over the parts of the packed counter block that the scans since the last reset wrote: the u64
 * lanes (13 global counters, CpG line totals, the subfamily/family/class pairs), the u32 lanes of the mode that ran (stat:
 * coverage difference arrays; filter: per-locus counts -- wrapping like the reference's unsigned int) and, after a CpG scan,
 * its u32 counts and f64 score sums (the one floating-point lane: the sum order differs from a single scan's, 1e-9 relative).
 * Every rank must have run the same kinds of scan, so that the lanes match. */
extern "C" int itx_comm_allreduce_counts(itx_index *ix, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    itx_cuda *cu = ix->cu;
    if (!cu->nccl_comm) { snprintf(err, ITX_ERRLEN, "itx_comm_init has not been called"); return ITX_EARG; }
    CK(cudaSetDevice(cu->device));
    fn_allreduce ar = (fn_allreduce)dlsym(cu->nccl_lib, "ncclAllReduce");
    fn_void gs = (fn_void)dlsym(cu->nccl_lib, "ncclGroupStart"), ge = (fn_void)dlsym(cu->nccl_lib, "ncclGroupEnd");
    if (!ar || !gs || !ge) { snprintf(err, ITX_ERRLEN, "NCCL symbols missing"); return ITX_ENOTSUP; }
    const int ncclUint32 = 3, ncclUint64 = 5, ncclFloat64 = 8, ncclSum = 0;
    const size_t ne = (size_t)ix->n_elem, ng = (size_t)(ix->subs.n + ix->fams.n + ix->clas.n), bl = (size_t)ix->bp_len;
    /* the CpG line totals ride in two spare u64 lanes */
    unsigned long long tot[2] = {ix->cpg_lines, ix->cpg_in_repeat};
    CK(cudaMemcpyAsync(cu->D.cnt + 13, tot, sizeof tot, cudaMemcpyHostToDevice, cu->stream));
    int r = gs();
    if (!r) r = ar(cu->d_u64, cu->d_u64, cu->n_u64, ncclUint64, ncclSum, cu->nccl_comm, cu->stream);
    if (!r && cu->used_bp && bl) r = ar(cu->D.bp_diff, cu->D.bp_diff, 2 * bl, ncclUint32, ncclSum, cu->nccl_comm, cu->stream);
    if (!r && cu->used_el && ne) r = ar(cu->D.el_cnt, cu->D.el_cnt, 2 * ne, ncclUint32, ncclSum, cu->nccl_comm, cu->stream);
    if (!r && cu->used_cpg) {
        const size_t nu = ng + (cu->used_cpg_el ? ne : 0), nf = ng + bl + (cu->used_cpg_el ? ne : 0);
        if (nu) r = ar(cu->d_cpg_u32, cu->d_cpg_u32, nu, ncclUint32, ncclSum, cu->nccl_comm, cu->stream);
        if (!r && nf) r = ar(cu->d_cpg_f64, cu->d_cpg_f64, nf, ncclFloat64, ncclSum, cu->nccl_comm, cu->stream);
    }
    int r2 = ge(); if (!r) r = r2;
    if (r != 0) { snprintf(err, ITX_ERRLEN, "ncclAllReduce failed (%d)", r); return ITX_ENODEV; }
    unsigned long long hc[16];
    CK(cudaMemcpyAsync(hc, cu->D.cnt, sizeof hc, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaStreamSynchronize(cu->stream));
    for (int k = 0; k < 13; k++) ix->cnt[k] = hc[k];
    ix->cpg_lines = hc[13]; ix->cpg_in_repeat = hc[14];
    return ITX_OK;
}
extern "C" void itx_get_cpg_totals(const itx_index *ix, uint64_t *n_lines, uint64_t *n_in_repeat) { if (n_lines) *n_lines = ix->cpg_lines; if (n_in_repeat) *n_in_repeat = ix->cpg_in_repeat; }
extern "C" int itx_comm_rank(const itx_index *ix, int *rank, int *nranks) {
    if (!ix->cu->nccl_comm) { if (rank) *rank = 0; if (nranks) *nranks = 1; return ITX_EARG; }
    if (rank) *rank = ix->cu->rank;
    if (nranks) *nranks = ix->cu->nranks;
    return ITX_OK;
}

/* ------------------------------------------------------------------ ONE BAM file across the ranks */
/* the touched counter blocks, saved before a rank scans its part of a file and put back if that part has to be scanned again
 * from another first record (the rank before says where the chain really enters) */
static int counters_snapshot(itx_index *ix, int restore, char *err) {
    itx_cuda *cu = ix->cu;
    const size_t b64 = cu->n_u64 * 8, b32 = ((cu->used_el ? cu->n_u32 : 2 * (size_t)ix->bp_len)) * 4, bm = (2 * ITX_MAX_TID_SEEN + 8) * 4;
    if (!cu->d_snap || cu->snap_cap < b64 + b32 + bm) {
        if (restore) { snprintf(err, ITX_ERRLEN, "internal: no counter snapshot to restore"); return ITX_EARG; }
        cudaFree(cu->d_snap); cu->d_snap = NULL;
        CK(cudaMalloc(&cu->d_snap, b64 + b32 + bm)); cu->snap_cap = b64 + b32 + bm;
    }
    uint8_t *q = (uint8_t *)cu->d_snap;
    if (!restore) {
        CK(cudaMemcpyAsync(q, cu->d_u64, b64, cudaMemcpyDeviceToDevice, cu->stream));
        CK(cudaMemcpyAsync(q + b64, cu->d_u32, b32, cudaMemcpyDeviceToDevice, cu->stream));
        CK(cudaMemcpyAsync(q + b64 + b32, cu->d_misc, bm, cudaMemcpyDeviceToDevice, cu->stream));
    } else {
        CK(cudaMemcpyAsync(cu->d_u64, q, b64, cudaMemcpyDeviceToDevice, cu->stream));
        CK(cudaMemcpyAsync(cu->d_u32, q + b64, b32, cudaMemcpyDeviceToDevice, cu->stream));
        CK(cudaMemcpyAsync(cu->d_misc, q + b64 + b32, bm, cudaMemcpyDeviceToDevice, cu->stream));
    }
    CK(cudaStreamSynchronize(cu->stream));
    return ITX_OK;
}

/* Rank `rank` of `nranks` scans its part of ONE BGZF file: the blocks that start in its share of the file's bytes, the records
 * that start in those blocks.  entry = ITX_SHARD_GUESS: the first record start is guessed out of the bytes like any span's (rank 0
 * starts behind the header whatever `entry` says); otherwise entry is the offset -- in the rank's own uncompressed bytes -- that
 * itx_shard_chain_check handed back.  rep tells how the chain entered and left the part. */
/* the scan of one rank's part, shared by the counting scan and phase 1 of -R (collect: the part table is filled, nothing is counted) */
static int shard_scan(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                      itx_shard_report *rep, uint64_t cnt[13], char *err, int collect, uint64_t *len_out) {
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    int fd = open(path, O_RDONLY);
    if (fd < 0) { snprintf(err, ITX_ERRLEN, "Error\n[bam file %s: %s]", path, strerror(errno)); return ITX_EIO; }
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); snprintf(err, ITX_ERRLEN, "Error\n[bam file %s is empty or unreadable]", path); return ITX_EIO; }
    memset(&ix->prof, 0, sizeof ix->prof);
    posix_fadvise(fd, 0, 0, POSIX_FADV_SEQUENTIAL);
    itx_bgzf_src S; S.fd = fd; S.mem = NULL; S.len = (uint64_t)st.st_size;
    int rc = ITX_OK;
    const bool retry_possible = nranks > 1 && rank + 1 < nranks;
    if (!collect && retry_possible && (rc = counters_snapshot(ix, 0, err))) { close(fd); return rc; }
    /* the record that straddles the end of the part needs bytes of the next rank's blocks: 1 MiB of them, more only if a longer record shows up */
    for (uint64_t margin = 1u << 20;; margin = margin < (16u << 20) ? (16u << 20) : (64ull << 20) + 65536) {
        if (collect && (rc = dup_table_clear(cu, &cu->part, err))) break;
        shard_io sh; memset(&sh, 0, sizeof sh);
        sh.rank = rank; sh.nranks = nranks; sh.entry = entry == ITX_SHARD_GUESS ? ITX_OFF_GUESS : entry; sh.margin = margin; sh.collect = collect;
        rc = scan_bgzf_device_inflate(ix, &S, o, cnt, err, inflate_thread_count(ix), &sh);
        if (rc != ITX_OK) break;
        rep->entry_rel = sh.entry_rel; rep->exit_rel = sh.exit_rel; rep->own_bytes = sh.own_bytes;
        if (len_out) *len_out = sh.len;
        if (!(retry_possible && sh.exit_rel == ITX_OFF_END && sh.more_after && margin < (64ull << 20))) break;
        if (!collect && (rc = counters_snapshot(ix, 1, err))) break;      /* the chain ran out of bytes, not out of records: again with more room */
    }
    close(fd);
    return rc;
}
extern "C" int itx_scan_shard_file(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                                   itx_shard_report *rep, uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    if (rank < 0 || nranks < 1 || rank >= nranks || !rep) { snprintf(err, ITX_ERRLEN, "bad rank %d of %d", rank, nranks); return ITX_EARG; }
    if (o->isSam) { snprintf(err, ITX_ERRLEN, "SAM text cannot be split across ranks"); return ITX_ENOTSUP; }
    if (nranks > 1 && o->rmDup) { snprintf(err, ITX_ERRLEN, "-R across ranks takes itx_shard_dedup_keys, an exchange of the keys and itx_scan_shard_file_rmdup"); return ITX_ENOTSUP; }
    if (nranks > 1 && (o->outbed || o->outbed_unique || o->readNames)) { snprintf(err, ITX_ERRLEN, "-B / -V and filter -r follow the reads in file order: they are not available in a sharded scan"); return ITX_ENOTSUP; }
    return shard_scan(ix, path, o, rank, nranks, entry, rep, cnt, err, 0, NULL);
}

/* ------------------------------------------------------------------ -R across ranks */
/* File order across N ranks is (file, rank, place in the rank's part).  Phase 1 settles every part's first record (the chain
 * protocol above) and collects the keys of its unique fragments, counting nothing; the keys and two flags per part (a unique
 * fragment, some other fragment) go to every rank; phase 2 admits those of the parts before its own with an ordinal below all of
 * its own, counts its part with -R, then admits those of the parts after it, so that the next file of the run finds every key of
 * this one in its table (itx_logic.cuh: itx_dup_nonunique_kept, k_dedup). */
static int shard_opts_check(const itx_scan_opts *o, int rank, int nranks, char *err) {
    if (rank < 0 || nranks < 1 || rank >= nranks) { snprintf(err, ITX_ERRLEN, "bad rank %d of %d", rank, nranks); return ITX_EARG; }
    if (o->isSam) { snprintf(err, ITX_ERRLEN, "SAM text cannot be split across ranks"); return ITX_ENOTSUP; }
    if (o->outbed || o->outbed_unique || o->readNames) { snprintf(err, ITX_ERRLEN, "-B / -V and filter -r follow the reads in file order: they are not available in a sharded scan"); return ITX_ENOTSUP; }
    return ITX_OK;
}
static int shard_dedup_keys(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                            itx_shard_report *rep, uint64_t *n_keys, uint32_t *flags, char *err) {
    int rc = shard_opts_check(o, rank, nranks, err); if (rc) return rc;
    itx_cuda *cu = ix->cu;
    itx_scan_opts o1 = *o; o1.rmDup = 0;              /* nothing is counted, so nothing is judged */
    free(cu->p1.path); cu->p1.path = NULL;
    uint64_t len = 0;
    if ((rc = shard_scan(ix, path, &o1, rank, nranks, entry, rep, NULL, err, 1, &len))) return rc;
    unsigned long long m[3];
    CK(cudaMemcpy(m, cu->part.mins, sizeof m, cudaMemcpyDeviceToHost));
    /* a part whose chain found no record start, or ended in a cut record, counts nothing and so exports nothing */
    const bool none = rank > 0 && rep->entry_rel >= ITX_OFF_GUESS;
    cu->p1.n_keys = none ? 0 : m[2];
    cu->p1.flags = none ? 0u : (m[0] != ITX_DUP_EMPTY ? 1u : 0u) | (m[1] != ITX_DUP_EMPTY ? 2u : 0u);
    cu->p1.path = strdup(path); cu->p1.rank = rank; cu->p1.nranks = nranks; cu->p1.len = len; cu->p1.own = rep->own_bytes; cu->p1.rep = *rep;
    if (n_keys) *n_keys = cu->p1.n_keys;
    if (flags) *flags = cu->p1.flags;
    return ITX_OK;
}
extern "C" int itx_shard_dedup_keys(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                                    itx_shard_report *rep, uint64_t *n_keys, uint32_t *flags, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    if (!rep) { snprintf(err, ITX_ERRLEN, "no shard report to fill"); return ITX_EARG; }
    return shard_dedup_keys(ix, path, o, rank, nranks, entry, rep, n_keys, flags, err);
}
static int ensure_xkeys(itx_cuda *cu, uint64_t n, char *err) {
    if (!cu->d_xn) CK(cudaMalloc((void **)&cu->d_xn, 8));
    void *p = cu->d_xkeys; uint64_t cap = cu->xkeys_cap * sizeof(itx_k128);
    int rc = grow_device(cu, &p, &cap, (n ? n : 1) * sizeof(itx_k128), 0, "the -R keys of the other ranks", err);
    cu->d_xkeys = (itx_k128 *)p; cu->xkeys_cap = cap / sizeof(itx_k128);
    return rc;
}
/* the part table's keys, dense, at `dst` on the device (room for cu->p1.n_keys of them) */
static int dedup_export(itx_cuda *cu, itx_k128 *dst, char *err) {
    if (!cu->p1.n_keys) return ITX_OK;
    unsigned long long got = 0;
    CK(cudaMemsetAsync(cu->d_xn, 0, 8, cu->stream));
    uint64_t blocks = (cu->part.cap + 255) / 256, most = (uint64_t)cu->sm_count * 8; if (blocks > most) blocks = most;
    k_dedup_export<<<(unsigned)blocks, 256, 0, cu->stream>>>(cu->part.keys, cu->part.cap, dst, cu->d_xn);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&got, cu->d_xn, 8, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaStreamSynchronize(cu->stream));
    if (got != cu->p1.n_keys) { snprintf(err, ITX_ERRLEN, "internal: %llu keys exported, the part table holds %llu", got, (unsigned long long)cu->p1.n_keys); return ITX_EFORMAT; }
    return ITX_OK;
}
extern "C" uint64_t itx_shard_dedup_fetch(itx_index *ix, void *dst, uint64_t cap) {
    itx_cuda *cu = ix->cu;
    char err[ITX_ERRLEN];
    if (!cu->p1.path || cudaSetDevice(cu->device) != cudaSuccess || ensure_xkeys(cu, cu->p1.n_keys, err) || dedup_export(cu, cu->d_xkeys, err)) return 0;
    const uint64_t n = cu->p1.n_keys < cap ? cu->p1.n_keys : cap;
    if (n && cudaMemcpy(dst, cu->d_xkeys, n * sizeof(itx_k128), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}
/* n keys at d_keys (device) and the flags of the parts they come from, entered into the run's table with a freshly reserved ordinal:
 * above everything this rank has scanned or admitted so far, below everything it scans afterwards */
static int dedup_admit(itx_cuda *cu, const itx_k128 *d_keys, uint64_t n, uint32_t flags, char *err) {
    int rc = ensure_dup_table(cu, &cu->dup, n, err); if (rc) return rc;
    const unsigned long long ord = cu->dup_ord_base++;
    itx_dedup_args A; memset(&A, 0, sizeof A);
    A.keys = cu->dup.keys; A.ords = cu->dup.ords; A.mask = cu->dup.cap - 1; A.mins = cu->dup.mins; A.status = cu->D.status;
    CK(cudaMemsetAsync(cu->D.status + 4, 0, 4, cu->stream));
    uint64_t blocks = (n + 255) / 256, most = (uint64_t)cu->sm_count * 8; if (blocks > most) blocks = most; if (blocks < 1) blocks = 1;
    k_dedup_admit<<<(unsigned)blocks, 256, 0, cu->stream>>>(d_keys, n, ord, flags, A);
    CK(cudaGetLastError());
    uint32_t full = 0;
    CK(cudaMemcpyAsync(&full, cu->D.status + 4, 4, cudaMemcpyDeviceToHost, cu->stream));
    CK(cudaStreamSynchronize(cu->stream));
    if (full) { snprintf(err, ITX_ERRLEN, "the -R key table overflowed"); return ITX_ENOMEM; }
    return ITX_OK;
}
extern "C" int itx_dedup_admit(itx_index *ix, const void *keys, uint64_t n, uint32_t flags, char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    itx_cuda *cu = ix->cu;
    CK(cudaSetDevice(cu->device));
    int rc = ensure_xkeys(cu, n, err); if (rc) return rc;
    if (n) CK(cudaMemcpy(cu->d_xkeys, keys, n * sizeof(itx_k128), cudaMemcpyHostToDevice));
    return dedup_admit(cu, cu->d_xkeys, n, flags, err);
}
/* phase 2: the -R scan of the part phase 1 settled, over the stream phase 1 left on the device (no second read or inflate) */
static int shard_count_rmdup(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                             itx_shard_report *rep, uint64_t cnt[13], char *err) {
    int rc = shard_opts_check(o, rank, nranks, err); if (rc) return rc;
    itx_cuda *cu = ix->cu;
    if (!cu->p1.path || !cu->p1.h || strcmp(cu->p1.path, path) != 0 || cu->p1.rank != rank || cu->p1.nranks != nranks || (rank > 0 && entry != cu->p1.rep.entry_rel)) {
        snprintf(err, ITX_ERRLEN, "itx_shard_dedup_keys has not settled this part (%s, rank %d of %d, entry %llu)", path, rank, nranks, (unsigned long long)entry);
        return ITX_EARG;
    }
    CK(cudaSetDevice(cu->device));
    if (rep) *rep = cu->p1.rep;
    if (rank > 0 && entry >= ITX_OFF_GUESS) { if (cnt) memcpy(cnt, ix->cnt, sizeof ix->cnt); return ITX_OK; }     /* nothing to count */
    itx_scan_opts o2 = *o; o2.rmDup = 1;
    const uint64_t len = cu->p1.len;
    memset(&ix->prof, 0, sizeof ix->prof);
    scan_ctx sc;
    if ((rc = scan_begin(&sc, ix, cu->p1.h, cu->d_stream, len, &o2, ix->tune_window < len ? ix->tune_window : len, err, 1, rank > 0 ? entry : ITX_CARRY_HEADER))) return rc;
    sc.own = cu->p1.own;
    {
        const uint64_t first = sc.carry0 >= ITX_OFF_GUESS ? 0 : sc.carry0;
        sc.k_end = sc.own > first ? (sc.own + cu->C - 1) / cu->C : sc.k_first;
    }
    if ((rc = scan_window(&sc, sc.k_end, len, err))) return rc;
    if ((rc = scan_end(&sc, cnt, err))) return rc;
    const uint64_t x = sc.carry_out, own = sc.own;
    const uint64_t exit_rel = x >= ITX_OFF_GUESS ? (x == ITX_OFF_GUESS ? ITX_OFF_NONE : x) : (x >= own ? x - own : 0);
    if (exit_rel != cu->p1.rep.exit_rel) {
        snprintf(err, ITX_ERRLEN, "internal: the -R scan of %s left rank %d's part at %llu, phase 1 at %llu", path, rank, (unsigned long long)exit_rel, (unsigned long long)cu->p1.rep.exit_rel);
        return ITX_EFORMAT;
    }
    ix->prof.stream_bytes = own;
    return ITX_OK;
}
extern "C" int itx_scan_shard_file_rmdup(itx_index *ix, const char *path, const itx_scan_opts *o, int rank, int nranks, uint64_t entry,
                                         itx_shard_report *rep, uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    return shard_count_rmdup(ix, path, o, rank, nranks, entry, rep, cnt, err);
}
typedef int (*fn_allgather)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef int (*fn_bcast)(const void *, void *, size_t, int, int, void *, cudaStream_t);
/* four u64 of every rank, in rank order, on the host (cu->d_shard holds this rank's four, then everybody's) */
static int gather4(itx_cuda *cu, fn_allgather ag, const unsigned long long mine[4], unsigned long long *all, char *err) {
    if (cudaMemcpyAsync(cu->d_shard, mine, 4 * 8, cudaMemcpyHostToDevice, cu->stream) != cudaSuccess ||
        ag(cu->d_shard, cu->d_shard + 4, 4, 5 /* ncclUint64 */, cu->nccl_comm, cu->stream) != 0 ||
        cudaMemcpyAsync(all, cu->d_shard + 4, 4 * 8 * (size_t)cu->nranks, cudaMemcpyDeviceToHost, cu->stream) != cudaSuccess ||
        cudaStreamSynchronize(cu->stream) != cudaSuccess) { snprintf(err, ITX_ERRLEN, "ncclAllGather failed"); return ITX_ENODEV; }
    return ITX_OK;
}
/* every rank's local status through one all-gather: the first failure, named, on every rank (so that none waits for a collective
 * that another rank will not join) */
static int agree(itx_cuda *cu, fn_allgather ag, int rc_local, const char *e_local, const char *what, unsigned long long *all, char *err) {
    const unsigned long long mine[4] = {(unsigned long long)(unsigned)(-rc_local), 0, 0, 0};
    int rc = gather4(cu, ag, mine, all, err); if (rc) return rc;
    for (int k = 0; k < cu->nranks; k++) if (all[4 * k]) {
        rc = -(int)(unsigned)all[4 * k];
        if (k == cu->rank) snprintf(err, ITX_ERRLEN, "%s", e_local); else snprintf(err, ITX_ERRLEN, "rank %d failed in %s (status %d)", k, what, rc);
        return rc;
    }
    return ITX_OK;
}
/* -R, once the chain of `path` has settled: all-gather (keys, flags) per part, every part's keys to every rank (one grouped
 * ncclBroadcast per root, device to device, into one buffer in rank order), then phase 2 between the admissions of the parts
 * before and after this rank's */
static int shard_rmdup_exchange_count(itx_index *ix, const char *path, const itx_scan_opts *o, uint64_t cnt[13], itx_profile *total, char *err) {
    itx_cuda *cu = ix->cu;
    const int nr = cu->nranks, me = cu->rank;
    fn_allgather ag = (fn_allgather)dlsym(cu->nccl_lib, "ncclAllGather");
    fn_bcast bc = (fn_bcast)dlsym(cu->nccl_lib, "ncclBroadcast");
    fn_void gs = (fn_void)dlsym(cu->nccl_lib, "ncclGroupStart"), ge = (fn_void)dlsym(cu->nccl_lib, "ncclGroupEnd");
    if (!ag || !bc || !gs || !ge) { snprintf(err, ITX_ERRLEN, "NCCL symbols missing"); return ITX_ENOTSUP; }
    const double t0 = now_ms();
    std::vector<unsigned long long> all(4 * (size_t)nr);
    const unsigned long long mine[4] = {cu->p1.n_keys, cu->p1.flags, 0, 0};
    int rc = gather4(cu, ag, mine, all.data(), err); if (rc) return rc;
    std::vector<uint64_t> off((size_t)nr + 1, 0), n((size_t)nr);
    uint32_t before = 0, after = 0;
    for (int k = 0; k < nr; k++) {
        n[k] = all[4 * k]; off[k + 1] = off[k] + n[k];
        if (k < me) before |= (uint32_t)all[4 * k + 1]; else if (k > me) after |= (uint32_t)all[4 * k + 1];
    }
    char e1[ITX_ERRLEN]; e1[0] = 0;
    int rc1 = ensure_xkeys(cu, off[nr], e1);
    if (rc1 == ITX_OK) rc1 = dedup_export(cu, cu->d_xkeys + off[me], e1);
    if ((rc = agree(cu, ag, rc1, e1, path, all.data(), err))) return rc;
    if (off[nr]) {
        int r = gs();
        for (int k = 0; k < nr && !r; k++) if (n[k]) r = bc(cu->d_xkeys + off[k], cu->d_xkeys + off[k], 2 * n[k], 5 /* ncclUint64 */, k, cu->nccl_comm, cu->stream);
        const int r2 = ge(); if (!r) r = r2;
        if (r != 0 || cudaStreamSynchronize(cu->stream) != cudaSuccess) { snprintf(err, ITX_ERRLEN, "ncclBroadcast of the -R keys failed (%d)", r); return ITX_ENODEV; }
    }
    const double t1 = now_ms();
    rc1 = dedup_admit(cu, cu->d_xkeys, off[me], before, e1);
    if (rc1 == ITX_OK) rc1 = shard_count_rmdup(ix, path, o, me, nr, cu->p1.rep.entry_rel, NULL, cnt, e1);
    if (rc1 == ITX_OK) rc1 = dedup_admit(cu, cu->d_xkeys + off[me + 1], off[nr] - off[me + 1], after, e1);
    const double t2 = now_ms();
    total->decode_ms += ix->prof.decode_ms; total->overlap_ms += ix->prof.overlap_ms; total->n_launches += ix->prof.n_launches;
    total->rmdup_exchange_ms += t1 - t0; total->rmdup_count_ms += t2 - t1; total->rmdup_bcast_bytes += off[nr] * sizeof(itx_k128);
    return agree(cu, ag, rc1, e1, path, all.data(), err);
}
extern "C" int itx_scan_alignments_shard(itx_index *ix, const char *bam_list, const itx_scan_opts *o, uint64_t cnt[13], char err[ITX_ERRLEN]) {
    char lerr[ITX_ERRLEN]; if (!err) err = lerr;
    err[0] = 0;
    itx_cuda *cu = ix->cu;
    if (!cu->nccl_comm) { snprintf(err, ITX_ERRLEN, "itx_comm_init has not been called"); return ITX_EARG; }
    CK(cudaSetDevice(cu->device));
    fn_allgather ag = (fn_allgather)dlsym(cu->nccl_lib, "ncclAllGather");
    if (!ag) { snprintf(err, ITX_ERRLEN, "NCCL symbols missing"); return ITX_ENOTSUP; }
    const int nr = cu->nranks, me = cu->rank, ncclUint64 = 5;
    if (!cu->d_shard) CK(cudaMalloc((void **)&cu->d_shard, 4 * 8 * (size_t)(nr + 1)));
    unsigned long long *all = (unsigned long long *)malloc(4 * 8 * (size_t)nr);
    itx_shard_report *reps = (itx_shard_report *)malloc(sizeof(itx_shard_report) * (size_t)nr);
    char *list = strdup(bam_list), *save = NULL; int rc = ITX_OK, nfile = 0;
    itx_profile total; memset(&total, 0, sizeof total);
    const bool rmdup = o->rmDup && nr > 1;             /* phase 1 in the rounds below, then the exchange and phase 2 */
    for (char *tok = strtok_r(list, ",", &save); tok && rc == ITX_OK; tok = strtok_r(NULL, ",", &save)) {
        if (++nfile > 100) break;                       /* the reference's row[100] */
        uint64_t entry = ITX_SHARD_GUESS;
        const double tk0 = now_ms();
        if ((rc = counters_snapshot(ix, 0, err))) break;
        itx_shard_report rep; memset(&rep, 0, sizeof rep);
        bool need_scan = true;
        /* rounds in lock step: whoever has to, scans; everybody all-gathers; everybody runs the same check on the same reports */
        for (int round = 0; rc == ITX_OK; round++) {
            char e1[ITX_ERRLEN]; e1[0] = 0; int rc1 = ITX_OK;
            if (need_scan) {
                if (round > 0) rc1 = counters_snapshot(ix, 1, e1);
                if (rc1 == ITX_OK) rc1 = rmdup ? shard_dedup_keys(ix, tok, o, me, nr, entry, &rep, NULL, NULL, e1) : itx_scan_shard_file(ix, tok, o, me, nr, entry, &rep, cnt, e1);
                need_scan = false;
                if (round == 0) {
                    total.decode_ms += ix->prof.decode_ms; total.overlap_ms += ix->prof.overlap_ms; total.total_ms += ix->prof.total_ms; total.h2d_ms += ix->prof.h2d_ms;
                    total.inflate_ms += ix->prof.inflate_ms; total.stream_bytes += ix->prof.stream_bytes; total.h2d_bytes += ix->prof.h2d_bytes; total.d2h_bytes += ix->prof.d2h_bytes;
                    total.n_launches += ix->prof.n_launches; total.fused = ix->prof.fused; total.n_replayed_windows += ix->prof.n_replayed_windows;
                } else total.n_bad_chunks++;
            }
            unsigned long long mine[4] = {rep.entry_rel, rep.exit_rel, rep.own_bytes, (unsigned long long)(unsigned)(-rc1)};
            if (cudaMemcpyAsync(cu->d_shard, mine, sizeof mine, cudaMemcpyHostToDevice, cu->stream) != cudaSuccess ||
                ag(cu->d_shard, cu->d_shard + 4, 4, ncclUint64, cu->nccl_comm, cu->stream) != 0 ||
                cudaMemcpyAsync(all, cu->d_shard + 4, 4 * 8 * (size_t)nr, cudaMemcpyDeviceToHost, cu->stream) != cudaSuccess ||
                cudaStreamSynchronize(cu->stream) != cudaSuccess) { snprintf(err, ITX_ERRLEN, "ncclAllGather of the shard reports failed"); rc = ITX_ENODEV; break; }
            int failed = -1;
            for (int k = 0; k < nr; k++) { reps[k].entry_rel = all[4 * k]; reps[k].exit_rel = all[4 * k + 1]; reps[k].own_bytes = all[4 * k + 2]; if (all[4 * k + 3] && failed < 0) failed = k; }
            if (failed >= 0) {
                rc = -(int)(unsigned)all[4 * failed + 3];
                if (failed == me) snprintf(err, ITX_ERRLEN, "%s", e1); else snprintf(err, ITX_ERRLEN, "rank %d failed in %s (status %d)", failed, tok, rc);
                break;
            }
            uint64_t forced = 0;
            const int bad = itx_shard_chain_check(nr, reps, &forced);
            if (bad < 0) break;                                    /* the parts chain: this file is done */
            if (round > nr) { snprintf(err, ITX_ERRLEN, "internal: the parts of %s do not chain after %d rounds", tok, round); rc = ITX_EFORMAT; break; }
            if (bad == me) { entry = forced; need_scan = true; }
        }
        if (rc == ITX_OK && rmdup) {
            total.rmdup_keys_ms += now_ms() - tk0;
            rc = shard_rmdup_exchange_count(ix, tok, o, cnt, &total, err);
        }
    }
    /* this rank's counters as they stand */
    if (rc == ITX_OK) {
        unsigned long long hc[16];
        if (cudaMemcpy(hc, cu->D.cnt, sizeof hc, cudaMemcpyDeviceToHost) != cudaSuccess) { snprintf(err, ITX_ERRLEN, "CUDA error reading the counters"); rc = ITX_ENODEV; }
        else { for (int k = 0; k < 13; k++) ix->cnt[k] = hc[k]; if (cnt) memcpy(cnt, ix->cnt, sizeof ix->cnt); }
    }
    total.n_records = ix->cnt[0] + ix->cnt[1]; total.n_fragments = ix->cnt[6];
    ix->prof = total;
    free(list); free(all); free(reps);
    return rc;
}
extern "C" void itx_get_counters(const itx_index *ix, uint64_t cnt[13]) { memcpy(cnt, ix->cnt, sizeof ix->cnt); }
extern "C" void itx_comm_destroy(itx_index *ix) {
    itx_cuda *cu = ix ? ix->cu : NULL;
    if (!cu || !cu->nccl_comm) return;
    fn_destroy f = (fn_destroy)dlsym(cu->nccl_lib, "ncclCommDestroy");
    if (f) f(cu->nccl_comm);
    cu->nccl_comm = NULL;
}
