/* itx_kernels.cuh -- the sm_100a kernels of the iteres hot path.
 *
 *   k_scan      K1+K2+K3  the product path: record boundaries, bam1_core_t unpack, fragment logic, interval overlap,
 *                    "last ascent" selection, XA:Z alternate test and accumulation in ONE pass; nothing but counters
 *                    is written.  The stream is cut into spans; a warp takes a span, GUESSES its first record start
 *                    out of the span's first staged bytes (32 offsets per step, branch-free structural test), then
 *                    carries the block_size chain through the span stage by stage: each 4 KiB stage (+1 KiB margin)
 *                    lands in the warp's shared memory through one 1-D TMA bulk copy (cp.async.bulk + mbarrier) while
 *                    the next stage's bytes are asked into L2; the chain of a stage is walked with run prediction on
 *                    the span's dominant record size; every lane then decodes one record per round and looks its
 *                    fragment up in a 32-entry window of the interval table that sits in shared memory (fetched a
 *                    stage ahead with cp.async).  The spans' entries and exits are logged and checked by the last
 *                    CTA; a failed guess is undone exactly (sign = -1) and replayed through the tuple path.
 *                                                              replaces bam_read1 / bam_calend / bam_aux_get /
 *                                                              binKeeperFind / getCov / mapped2diffSubfam / the counters
 *   k_decode_span K1  the same front half writing 16-byte tuples (one coalesced 512-byte store per 32 records): the
 *                    tuple path, taken when something needs the tuples (-R, ordered outputs, traces).
 *   k_verify / k_fixup  the entry a span assumed must equal the chain exit of the previous span; otherwise the
 *                    span is re-walked from its true entry.  The tuples are therefore exactly the sequential
 *                    chain, whatever the guesses were.
 *   k_decode         the same contract, one thread per chunk reading global memory (A/B measurement, odd sizes).
 *   k_overlap   K2+K3  one lane per tuple: position bucket + bounded backward walk in place of binKeeperFind,
 *                    "last ascent" selection, XA:Z alternate test, then warp-aggregated counters, a shared-memory
 *                    subfamily/family/class histogram per CTA flushed with u64 reductions, and two u32 reductions
 *                    per coverage difference array.
 *   k_dedup     -R: 128-bit key table, smallest file-order ordinal per key.
 *   k_dedup_export / k_dedup_admit  -R across ranks: a part's keys out of its table, other parts' keys into the run's.
 *   k_finalize  prefix sums of the coverage difference arrays (one warp per subfamily).
 *   k_bedgraph / k_cpg  K4  CpG bedGraph text parsed on the device, rows against the same table (cpgBedGraphOverlapRepeat).
 *   k_query     overlap + selection for explicit queries (property tests).
 */
#ifndef ITX_KERNELS_CUH
#define ITX_KERNELS_CUH
#include "itx_logic.cuh"
#include "itx_inflate.cuh"

struct itx_decode_args {
    const uint8_t *b; unsigned long long len, avail, k0;
    unsigned long long own;             /* record starts at or past this offset are someone else's (<= len; = len unless the scan is one rank's shard of a stream) */
    uint32_t nchunks, C, S;
    const itx_tidinfo *tid; int32_t n_ref;
    itx_dev_opts o;
    itx_tuple *tuples; unsigned long long *entry, *exit_; uint32_t *nrec;
    unsigned long long *carry; uint32_t *winbad; uint32_t *status;
    uint32_t *work;                        /* [0] k_decode_span, [1] k_overlap (both zeroed by k_fixup), [2] k_scan (zeroed by its last CTA) */
};

/* fire-and-forget reductions (RED, no return value) */
__device__ __forceinline__ void itx_red_u32(uint32_t *p, uint32_t v) { asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void itx_red_u64(unsigned long long *p, unsigned long long v) { asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }

/* sequential walk of one chunk from global memory: used by k_decode and by the repair path */
__device__ __forceinline__ void itx_walk_chunk(const itx_decode_args &A, uint32_t i, unsigned long long p) {
    const itx_src_global G{A.b};
    const unsigned long long lo = (A.k0 + i) * (unsigned long long)A.C;
    unsigned long long hi = lo + A.C; if (hi > A.own) hi = A.own;
    itx_tuple *out = A.tuples + (size_t)i * A.S;
    uint32_t n = 0;
    if (p < ITX_OFF_END) {
        while (p < hi) {
            if (p + 36 > A.len) { p = ITX_OFF_END; break; }
            uint32_t x[9]; G.core(p, x);
            if ((int32_t)x[0] < 32 || p + 4 + (unsigned long long)x[0] > A.len) { p = ITX_OFF_END; break; }
            if (p + 4 + (unsigned long long)x[0] > A.avail) atomicOr(&A.status[0], 2u);   /* record longer than the staged window */
            if (n < A.S) out[n] = itx_decode_record(G, p, x, (uint32_t)(p - lo), A.tid, A.n_ref, A.o);
            n++;
            p += 4 + (unsigned long long)x[0];
        }
    }
    A.exit_[i] = p; A.nrec[i] = n < A.S ? n : A.S;
}

__global__ void __launch_bounds__(128) k_decode(const itx_decode_args A) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.nchunks) return;
    unsigned long long lo = (A.k0 + i) * (unsigned long long)A.C, hi = lo + A.C;
    if (hi > A.own) hi = A.own;
    unsigned long long p = ITX_OFF_GUESS;
    if (i == 0) { p = *A.carry; *A.winbad = 0; }
    if (p == ITX_OFF_GUESS) p = itx_speculate_entry(itx_src_global{A.b}, lo, hi, A.len, A.n_ref);
    A.entry[i] = p;
    itx_walk_chunk(A, i, p);
}

/* ------------------------------------------------------------------ K1: one pass, TMA-staged, lane-parallel chain */
#define ITX_DW 8                           /* warps per CTA */
#define ITX_CLAIM 8u                       /* work units claimed per atomic on the work counters */
#define ITX_PART 128u                      /* tuple slots per k_overlap work unit */
#ifndef ITX_MARGIN
#define ITX_MARGIN 1024u                   /* bytes staged past the chunk end for records that straddle it */
#endif
#define ITX_DECODE_SMEM 0

__device__ __forceinline__ uint32_t itx_smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void itx_mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void itx_mbar_expect_tx(uint32_t bar, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ void itx_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ bool itx_mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void itx_cp_async16(void *smem_dst, const void *src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(itx_smem_addr(smem_dst)), "l"(src) : "memory"); }
__device__ __forceinline__ void itx_cp_async8(void *smem_dst, const void *src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(itx_smem_addr(smem_dst)), "l"(src) : "memory"); }
__device__ __forceinline__ void itx_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void itx_prefetch_l2(const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
/* bounded wait with back-off: a copy that never lands sets status bit 4 instead of hanging the device */
__device__ __noinline__ bool itx_mbar_wait_slow(uint32_t bar, uint32_t parity, uint32_t *status) {
    for (uint32_t spin = 0; spin < (1u << 22); spin++) { if (itx_mbar_try_wait(bar, parity)) return true; __nanosleep(64); }
    atomicOr(&status[0], 4u);
    return false;
}
__device__ __forceinline__ bool itx_mbar_wait(uint32_t bar, uint32_t parity, uint32_t *status) {
    if (itx_mbar_try_wait(bar, parity)) return true;
    return itx_mbar_wait_slow(bar, parity, status);
}
/* stream bytes [base, base + nb) staged linearly in shared memory; anything beyond comes from global memory */
/* Offsets are taken relative to the stage in 32 bits: a record is shorter than 2^31 bytes and starts inside the stage,
 * so the true distance always fits, and anything at or past nb goes to global memory. */
struct itx_src_stage {
    const uint8_t *buf; const uint8_t *g; unsigned long long base; uint32_t nb;
    __device__ __forceinline__ uint8_t u8(uint64_t off) const {
        const uint32_t d = (uint32_t)off - (uint32_t)base;
        return d < nb ? buf[d] : __ldg(g + off);
    }
    __device__ __forceinline__ uint32_t w32(uint64_t aligned_off) const {
        const uint32_t d = (uint32_t)aligned_off - (uint32_t)base;
        return d < (nb > 3u ? nb - 3u : 0u) ? *reinterpret_cast<const uint32_t *>(buf + d) : __ldg(reinterpret_cast<const uint32_t *>(g + aligned_off));
    }
    __device__ __forceinline__ uint32_t u32(uint64_t off) const {
        const uint64_t a = off & ~3ull; const uint32_t sh = (uint32_t)(off & 3) * 8;
        return itx_funnel_r(w32(a), w32(a + 4), sh);
    }
    __device__ __forceinline__ void core(uint64_t p, uint32_t x[9]) const {
        const uint64_t a = p & ~3ull; const uint32_t sh = (uint32_t)(p & 3) * 8;
        const uint32_t d = (uint32_t)a - (uint32_t)base;
        uint32_t w[10];
        if (d < (nb > 39u ? nb - 39u : 0u)) {
            const uint32_t *q = reinterpret_cast<const uint32_t *>(buf + d);
#pragma unroll
            for (int i = 0; i < 10; i++) w[i] = q[i];
        } else {
#pragma unroll
            for (int i = 0; i < 10; i++) w[i] = w32(a + 4u * i);
        }
#pragma unroll
        for (int j = 0; j < 9; j++) x[j] = itx_funnel_r(w[j], w[j + 1], sh);
    }
};
/* A warp per span (= "chunk" of the bookkeeping, A.C bytes, a multiple of ITX_STAGE).  Only the span's first
 * record start is GUESSED (out of the span's first stage, checked against the previous span by k_verify / k_fixup);
 * inside the span the chain is carried from one 4 KiB stage to the next.  Each stage (+1 KiB margin) arrives
 * in shared memory through one TMA bulk copy; the warp walks the block_size chain of the stage out of shared
 * memory with run prediction, then every lane decodes one record per round out of shared memory and the warp
 * stores 32 tuples with one coalesced 512-byte store. */
#define ITX_STAGE 4096u
#define ITX_POS_SLOTS 128u                 /* > ITX_STAGE / 36 record starts per stage */
#undef ITX_DECODE_SMEM
#define ITX_DECODE_SMEM (ITX_DW * (ITX_STAGE + ITX_MARGIN) + ITX_DW * ITX_POS_SLOTS * 2u + ITX_DW * 8)

__global__ void __launch_bounds__(ITX_DW * 32) k_decode_span(const itx_decode_args A) {
    extern __shared__ __align__(128) uint8_t itx_smem[];
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    constexpr uint32_t STG = ITX_STAGE + ITX_MARGIN;
    uint8_t *buf = itx_smem + w * STG;
    uint16_t *pos = reinterpret_cast<uint16_t *>(itx_smem + ITX_DW * STG) + w * ITX_POS_SLOTS;
    const uint32_t buf_s = itx_smem_addr(buf);
    const uint32_t bar_s = itx_smem_addr(itx_smem + ITX_DW * STG + ITX_DW * ITX_POS_SLOTS * 2u) + w * 8;
    if (lane == 0) {
        itx_mbar_init(bar_s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    if (blockIdx.x == 0 && threadIdx.x == 0) *A.winbad = 0;
    uint32_t parity = 0;
    bool dead = false;
    for (;;) {
        uint32_t i = 0;
        if (lane == 0) i = atomicAdd(&A.work[0], 1u);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= A.nchunks || dead) break;
        /* span-relative 32-bit offsets, sentinels 0xfffffffe (chain ended) / 0xffffffff (no guess), as in k_scan */
        const unsigned long long lo = (A.k0 + i) * (unsigned long long)A.C;
        const uint32_t hi = A.own - lo < A.C ? (uint32_t)(A.own - lo) : A.C;
        uint32_t p = 0xffffffffu;
        bool guess = i != 0;
        if (!guess) {
            const unsigned long long p0 = *A.carry;
            if (p0 == ITX_OFF_GUESS) guess = true;             /* the scan starts in the middle of a stream (a rank's shard) */
            else {
                if (lane == 0) A.entry[i] = p0;
                p = p0 >= ITX_OFF_END ? (uint32_t)p0 : (p0 - lo < 0xfffffff0ull ? (uint32_t)(p0 - lo) : 0xfffffffeu);
            }
        }
        itx_tuple *out = A.tuples + (size_t)i * A.S;
        uint32_t n_out = 0, staged = 0xffffffffu, nb = 0, szd = 0;
        for (;;) {
            if (guess ? hi == 0u : !(p < hi)) { if (guess && lane == 0) A.entry[i] = ITX_OFF_NONE; break; }
            const uint32_t c_lo = guess ? 0u : p & ~(ITX_STAGE - 1u);
            const uint32_t c_hi = c_lo + ITX_STAGE < hi ? c_lo + ITX_STAGE : hi;
            const unsigned long long rest = A.len - lo - c_lo;
            if (staged != c_lo) {
                nb = rest > STG ? STG : (uint32_t)rest;
                const uint32_t bytes = (nb + 15u) & ~15u;     /* the buffer's 64 bytes of slack cover the round-up */
                __syncwarp();                                  /* every lane is done reading the previous stage */
                if (lane == 0) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    itx_mbar_expect_tx(bar_s, bytes);
                    itx_bulk_g2s(buf_s, A.b + lo + c_lo, bytes, bar_s);
                    if (c_lo + ITX_STAGE < hi && rest >= STG + ITX_STAGE) itx_prefetch_l2(A.b + lo + c_lo + STG, ITX_STAGE);
                }
                if (!itx_mbar_wait(bar_s, parity, A.status)) { dead = true; break; }
                parity ^= 1u;
                staged = c_lo;
            }
            if (guess) {
                /* the span's first record start, guessed out of its first stage: itx_plausible2's test on 32 offsets per step */
                const itx_src_stage S0{buf, A.b, lo, nb};
                for (uint32_t base = 0; base < hi; base += 32) {
                    const uint32_t d = base + lane;
                    const unsigned long long q = lo + d;
                    bool ok = false;
                    if (d < hi && q + 36 <= A.len) {
                        uint32_t x[9];
                        S0.core(q, x);
                        ok = itx_plausible2_core(S0, x, q, A.len, A.n_ref);
                    }
                    const uint32_t m = __ballot_sync(0xffffffffu, ok);
                    if (m) { p = base + (uint32_t)__ffs((int)m) - 1; break; }
                }
                if (lane == 0) A.entry[i] = p == 0xffffffffu ? ITX_OFF_NONE : lo + p;
                guess = false;
                continue;
            }
            /* the chain of this stage (see k_scan): run prediction with the span's dominant record size */
            uint32_t n = 0;
            uint32_t q = p - c_lo;
            {
                const uint32_t qh = c_hi - c_lo;
                const uint32_t room32 = rest > 0x7fffffffull ? 0x7fffffffu : (uint32_t)rest;
                uint32_t q_end = q;
                while (q < qh) {
                    q_end = q;
                    if (q + 36u > room32) { q = 0xffffffffu; break; }
                    const uint32_t bs0 = itx_buf_u32(buf, q);
                    const uint32_t sz0 = bs0 + 4u;
                    if ((int32_t)bs0 < 32 || sz0 > room32 - q) { q = 0xffffffffu; break; }
                    const uint32_t szp = szd ? szd : sz0;
                    uint32_t run = 1u, pk = q;
                    if ((sz0 | szp) < 0x10000u) {
                        const bool same = itx_chain_lane(buf, q, sz0, szp, lane, qh, room32, &pk);
                        const uint32_t m = __ballot_sync(0xffffffffu, same);
                        run = m == 0xffffffffu ? 32u : (uint32_t)__ffs((int)~m) - 1u;
                    }
                    if (lane < run && n + lane < ITX_POS_SLOTS) pos[n + lane] = (uint16_t)pk;
                    n += run;
                    q += sz0 + (run - 1u) * szp;
                    szd = run >= 2u ? szp : 0u;
                }
                if (q != 0xffffffffu) q_end = q;
                if (lane == 0 && A.avail < lo + c_lo + q_end) atomicOr(&A.status[0], 2u);
            }
            __syncwarp();
            const unsigned long long c_lo64 = lo + c_lo;
            const itx_src_stage S{buf, A.b, c_lo64, nb};
            for (uint32_t j = lane; j < n; j += 32) {
                const uint32_t ro = pos[j];
                uint32_t x[9]; S.core(c_lo64 + ro, x);
                const itx_tuple T = itx_decode_record(S, c_lo64 + ro, x, c_lo + ro, A.tid, A.n_ref, A.o);
                if (n_out + j < A.S) __stcs(reinterpret_cast<uint4 *>(out + n_out + j), make_uint4(T.start, T.end, T.info, T.rec_off));
            }
            n_out += n;
            if (q == 0xffffffffu) { p = 0xfffffffeu; break; }
            p = c_lo + q;
        }
        if (lane == 0) { A.exit_[i] = p >= 0xfffffffeu ? (0xffffffff00000000ull | p) : lo + p; A.nrec[i] = n_out < A.S ? n_out : A.S; }
    }
}

/* The exit that counts for span i is that of the last span before it that holds a record start (a span a long record runs
 * over logs NONE for entry and exit); NONE all the way down means that nothing is known yet (a scan that starts in the
 * middle of a stream and has not met a record start so far). */
__device__ __forceinline__ unsigned long long itx_prev_exit(const unsigned long long *exit_, uint32_t j) {
    unsigned long long x = exit_[j];
    while (x == ITX_OFF_NONE && j > 0) { j--; x = exit_[j]; }
    return x;
}
__device__ __forceinline__ bool itx_span_consistent(const itx_decode_args &A, uint32_t i) {
    const unsigned long long en = A.entry[i], ex = itx_prev_exit(A.exit_, i - 1);
    if (en == ex || ex == ITX_OFF_NONE) return true;
    if (en != ITX_OFF_NONE) return false;
    const unsigned long long span_end = (A.k0 + i) * (unsigned long long)A.C + A.C;
    return ex == ITX_OFF_END || (ex < ITX_OFF_GUESS && ex >= (span_end < A.own ? span_end : A.own));
}
__global__ void k_verify(const itx_decode_args A) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 || i >= A.nchunks) return;
    if (!itx_span_consistent(A, i)) atomicAdd(A.winbad, 1u);
}

/* one warp; a no-op when every guess was right */
__global__ void k_fixup(const itx_decode_args A) {
    const uint32_t lane = threadIdx.x, n = A.nchunks;
    if (*A.winbad != 0) {
        uint32_t i = 1;
        while (i < n) {
            uint32_t idx = i + lane;
            bool bad = idx < n && !itx_span_consistent(A, idx);
            uint32_t m = __ballot_sync(0xffffffffu, bad);
            if (!m) { i += 32; continue; }
            uint32_t j = i + (uint32_t)__ffs((int)m) - 1;
            if (lane == 0) {
                unsigned long long e = itx_prev_exit(A.exit_, j - 1);
                A.entry[j] = e;
                itx_walk_chunk(A, j, e);
                atomicAdd(&A.status[1], 1u);
                __threadfence();
            }
            __syncwarp();
            i = j + 1;
        }
    }
    __syncwarp();
    if (lane == 0) {
        unsigned long long x = itx_prev_exit(A.exit_, n - 1);
        if (x == ITX_OFF_NONE && *A.carry == ITX_OFF_GUESS) x = ITX_OFF_GUESS;      /* still no record start met */
        *A.carry = x; A.work[0] = 0; A.work[1] = 0;
    }
}

/* ------------------------------------------------------------------ -R: duplicate removal */
/* An open-addressing table of 128-bit keys (claimed with one 128-bit compare-and-swap) beside an array with the
 * smallest file-order ordinal seen for each key.  Per window, k_dedup<false> enters every unique fragment, then
 * k_dedup<true> sets ITX_F_DUP on the fragments that are not their key's first: windows are processed in file
 * order and a later window can only bring larger ordinals, so a window's verdicts are final when it is marked. */
struct __align__(16) itx_k128 { unsigned long long lo, hi; };
__device__ __forceinline__ itx_k128 itx_cas128(itx_k128 *p, itx_k128 cmp, itx_k128 val) {
    itx_k128 old;
    asm volatile("{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\tatom.global.cas.b128 o, [%6], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(old.lo), "=l"(old.hi) : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(p) : "memory");
    return old;
}
#define ITX_DUP_EMPTY 0xffffffffffffffffull
struct itx_dedup_args {
    const uint8_t *b; unsigned long long k0; uint32_t nchunks, C, S;
    itx_tuple *tuples; const uint32_t *nrec; const itx_tidinfo *tid; int32_t n_ref;
    unsigned long long ord_base;                     /* ordinal of slot 0 of chunk 0 of this file */
    itx_k128 *keys; unsigned long long *ords; unsigned long long mask;      /* capacity - 1 (a power of two) */
    unsigned long long *mins;                        /* [0] smallest ordinal of a unique fragment, [1] of any other fragment, [2] keys in the table */
    uint32_t *status;                                /* [4] set when the table is full */
};
__device__ __forceinline__ bool itx_dup_enter(const itx_dedup_args &A, unsigned long long lo, unsigned long long hi, unsigned long long ord) {
    unsigned long long h = itx_dup_hash(lo, hi) & A.mask;
    const itx_k128 key{lo, hi}, empty{ITX_DUP_EMPTY, ITX_DUP_EMPTY};
    for (unsigned long long probes = 0; probes <= A.mask; probes++, h = (h + 1) & A.mask) {
        const itx_k128 old = itx_cas128(A.keys + h, empty, key);
        const bool fresh = old.lo == ITX_DUP_EMPTY && old.hi == ITX_DUP_EMPTY;
        if (fresh) atomicAdd(A.mins + 2, 1ull);
        if (fresh || (old.lo == lo && old.hi == hi)) { atomicMin(A.ords + h, ord); return true; }
    }
    return false;
}
__device__ __forceinline__ unsigned long long itx_dup_first(const itx_dedup_args &A, unsigned long long lo, unsigned long long hi) {
    unsigned long long h = itx_dup_hash(lo, hi) & A.mask;
    for (unsigned long long probes = 0; probes <= A.mask; probes++, h = (h + 1) & A.mask) {
        const itx_k128 k = A.keys[h];
        if (k.lo == lo && k.hi == hi) return A.ords[h];
        if (k.lo == ITX_DUP_EMPTY && k.hi == ITX_DUP_EMPTY) break;
    }
    return ITX_DUP_EMPTY;
}
template <bool MARK>
__global__ void __launch_bounds__(256) k_dedup(const itx_dedup_args A) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t w0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const itx_src_global G{A.b};
    unsigned long long mu = ITX_DUP_EMPTY, mn = ITX_DUP_EMPTY;
    if (MARK) { mu = A.mins[0]; mn = A.mins[1]; }
    for (uint32_t i = w0; i < A.nchunks; i += nw) {
        const uint32_t nr = A.nrec[i];
        const unsigned long long lo_b = (A.k0 + i) * (unsigned long long)A.C;
        itx_tuple *tp = A.tuples + (size_t)i * A.S;
        for (uint32_t j = lane; j < nr; j += 32) {
            const itx_tuple T = tp[j];
            if (!(T.info & ITX_F_FRAG)) continue;
            const unsigned long long ord = A.ord_base + (A.k0 + i) * (unsigned long long)A.S + j;
            if (T.info & ITX_F_UNIQ) {
                const int32_t t = (int32_t)G.u32(lo_b + T.rec_off + 4);
                const int32_t csid = (t >= 0 && t < A.n_ref) ? A.tid[t].csid : -1;
                unsigned long long klo, khi; itx_dup_key(csid, (T.info & ITX_F_MINUS) != 0, T.start, T.end, &klo, &khi);
                if (!MARK) { if (!itx_dup_enter(A, klo, khi, ord)) atomicOr(&A.status[4], 1u); if (ord < mu) mu = ord; }
                else if (itx_dup_first(A, klo, khi) != ord) tp[j].info = T.info | ITX_F_DUP;
            } else {
                if (!MARK) { if (ord < mn) mn = ord; }
                else if (!itx_dup_nonunique_kept(ord, mu, mn)) tp[j].info = T.info | ITX_F_DUP;
            }
        }
    }
    if (!MARK) {
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            const unsigned long long a = __shfl_xor_sync(0xffffffffu, mu, d), c = __shfl_xor_sync(0xffffffffu, mn, d);
            if (a < mu) mu = a;
            if (c < mn) mn = c;
        }
        if (lane == 0) { if (mu != ITX_DUP_EMPTY) atomicMin(A.mins, mu); if (mn != ITX_DUP_EMPTY) atomicMin(A.mins + 1, mn); }
    }
}
/* move every key of a full table into a larger one */
__global__ void k_dedup_rehash(const itx_k128 *old_keys, const unsigned long long *old_ords, unsigned long long old_cap, itx_dedup_args A) {
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < old_cap; s += (unsigned long long)gridDim.x * blockDim.x) {
        const itx_k128 k = old_keys[s];
        if (k.lo == ITX_DUP_EMPTY && k.hi == ITX_DUP_EMPTY) continue;
        if (!itx_dup_enter(A, k.lo, k.hi, old_ords[s])) atomicOr(&A.status[4], 1u);
    }
}
/* -R across ranks: the keys of one rank's part of a file, compacted out of its table into a dense array (one atomic per warp;
 * the order is arbitrary -- admission does not depend on it).  *n_out starts at 0. */
__global__ void k_dedup_export(const itx_k128 *keys, unsigned long long cap, itx_k128 *out, unsigned long long *n_out) {
    const uint32_t lane = threadIdx.x & 31;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long base = (unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < cap; base += stride) {
        const unsigned long long s = base + lane;
        itx_k128 k{ITX_DUP_EMPTY, ITX_DUP_EMPTY};
        if (s < cap) k = keys[s];
        const bool has = !(k.lo == ITX_DUP_EMPTY && k.hi == ITX_DUP_EMPTY);
        const uint32_t m = __ballot_sync(0xffffffffu, has);
        if (!m) continue;
        unsigned long long at = 0;
        if (lane == 0) at = atomicAdd(n_out, (unsigned long long)__popc(m));
        at = __shfl_sync(0xffffffffu, at, 0);
        if (has) out[at + __popc(m & ((1u << lane) - 1u))] = k;
    }
}
/* the keys of other ranks' parts entered into this rank's table with ONE ordinal `ord`, and the parts' flags (bit 0: a unique
 * fragment, bit 1: any other fragment) lowering mins[0] / mins[1] to it -- so that k_dedup<true> judges this rank's reads as if
 * those parts had been scanned here at that place in file order */
__global__ void k_dedup_admit(const itx_k128 *keys, unsigned long long n, unsigned long long ord, uint32_t flags, itx_dedup_args A) {
    const unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i0 == 0) {
        if (flags & 1u) atomicMin(A.mins, ord);
        if (flags & 2u) atomicMin(A.mins + 1, ord);
    }
    for (unsigned long long i = i0; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const itx_k128 k = keys[i];
        if (!itx_dup_enter(A, k.lo, k.hi, ord)) atomicOr(&A.status[4], 1u);
    }
}

/* ------------------------------------------------------------------ overlap + accumulate */
struct itx_overlap_args {
    itx_dev_index D;
    const uint8_t *b; unsigned long long k0; uint32_t nchunks, C, S;
    const itx_tuple *tuples; const uint32_t *nrec;
    itx_dev_opts o;
    itx_trace *trace; unsigned long long trace_cap; const unsigned long long *rec_base;   /* trace != 0: per-record trace */
    long long *sel_out;                                                                  /* != 0: selected element per tuple slot */
    uint32_t *work;
    const itx_dev_index *Dg;                                                             /* D in global memory, for the out-of-line selection of long hit lists */
};

#define ITX_WIN 32u                      /* table entries per warp window */
#define ITX_WIN_BYTES (ITX_WIN * (16u + 16u + 8u))
/* table loads of a walk: the warp's window when the index falls into it, global memory otherwise (same values either way) */
struct itx_iv_window {
    const itx_dev_index &D; const int4 *win; uint32_t base, n;
    __device__ __forceinline__ itx_iv operator()(uint32_t i) const {
        const uint32_t d = i - base;
        if (d < n) { const int4 v = win[d]; itx_iv e; e.start = v.x; e.end = v.y; e.pmax = v.z; e.row = (uint32_t)v.w; return e; }
        return itx_ld_iv(D, i);
    }
};
#define ITX_OVL_WIN_SMEM (8u * ITX_WIN_BYTES)          /* k_overlap: a table window per warp, behind the histogram */
template <bool SMEM_HIST>
__global__ void __launch_bounds__(256, 4) k_overlap(const itx_overlap_args A) {
    extern __shared__ __align__(16) uint32_t sh_hist[];
    __shared__ unsigned long long sh_cnt[13];
    const itx_dev_index &D = A.D;
    const uint32_t nh = SMEM_HIST ? 2u * (uint32_t)(D.n_sub + D.n_fam + D.n_cla) : 0u;
    for (uint32_t t = threadIdx.x; t < nh; t += blockDim.x) sh_hist[t] = 0;
    if (threadIdx.x < 13) sh_cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    /* the warp's table window (as k_scan's): tuples are in file order, so the 32 fragments of a round walk the same few table entries --
     * the entries around the highest bucket end any lane starts from are loaded once, coalesced, with their metadata, and the walks and
     * the accumulation read them out of shared memory (global memory outside the window: same values).  A window is kept while the
     * rounds that follow still start inside it. */
    uint8_t *win_b = reinterpret_cast<uint8_t *>(sh_hist) + ((nh * 4u + 15u) & ~15u) + (threadIdx.x >> 5) * ITX_WIN_BYTES;
    int4 *win_iv = reinterpret_cast<int4 *>(win_b);
    uint4 *win_meta = reinterpret_cast<uint4 *>(win_iv + ITX_WIN);
    int2 *win_meta2 = reinterpret_cast<int2 *>(win_meta + ITX_WIN);
    uint32_t wbase = 0, wn = 0;
    const uint32_t n_elem32 = D.n_elem > 0xffffffffll ? 0xffffffffu : (uint32_t)D.n_elem;
    uint32_t c[13];
#pragma unroll
    for (int k = 0; k < 13; k++) c[k] = 0;
    const bool stat = A.o.filter == 0 && D.stat_mode;
    const itx_src_global G{A.b};
    /* work unit = ITX_PART consecutive tuple slots of one chunk; a warp claims ITX_CLAIM units per atomic */
    const uint32_t ppc = (A.S + ITX_PART - 1) / ITX_PART, n_units = A.nchunks * ppc;
    uint32_t u = 0, u_end = 0;
    for (;; u++) {
        if (u >= u_end) {
            if (lane == 0) u = atomicAdd(A.work, ITX_CLAIM);
            u = __shfl_sync(0xffffffffu, u, 0);
            if (u >= n_units) break;
            u_end = u + ITX_CLAIM < n_units ? u + ITX_CLAIM : n_units;
        }
        const uint32_t i = u / ppc, part = u - i * ppc;
        const uint32_t nr = A.nrec[i];
        if (part * ITX_PART >= nr) { u += ppc - part - 1; continue; }       /* the rest of this chunk's units are empty */
        const uint32_t n = nr < (part + 1) * ITX_PART ? nr : (part + 1) * ITX_PART;
        const itx_tuple *tp = A.tuples + (size_t)i * A.S;
        const unsigned long long lo = (A.k0 + i) * (unsigned long long)A.C;
        for (uint32_t j0 = part * ITX_PART; j0 < n; j0 += 32) {
            const uint32_t j = j0 + lane; const bool valid = j < n;
            itx_tuple T; T.start = T.end = T.rec_off = 0; T.info = 0;
            if (valid) { const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(tp + j)); T.start = v.x; T.end = v.y; T.info = v.z; T.rec_off = v.w; }
            const uint32_t info = T.info;
            const bool slot2 = info & ITX_F_SLOT2, frag = info & ITX_F_FRAG, uniq = info & ITX_F_UNIQ, live = frag && !(info & ITX_F_DUP);
            const uint32_t m_valid = __ballot_sync(0xffffffffu, valid), m_slot2 = __ballot_sync(0xffffffffu, slot2);
            const uint32_t m_map = __ballot_sync(0xffffffffu, info & ITX_F_MAPPED), m_used = __ballot_sync(0xffffffffu, info & ITX_F_USED);
            const uint32_t m_frag = __ballot_sync(0xffffffffu, frag), m_uniq = __ballot_sync(0xffffffffu, uniq);
            c[0] += __popc(m_valid & ~m_slot2); c[1] += __popc(m_slot2);
            c[2] += __popc(m_map & ~m_slot2);   c[3] += __popc(m_map & m_slot2);
            c[4] += __popc(m_used & ~m_slot2);  c[5] += __popc(m_used & m_slot2);
            c[6] += __popc(m_frag);
            c[7] += __popc(m_frag & m_uniq);
            c[11] += __popc(__ballot_sync(0xffffffffu, live) & m_uniq);       /* unique reads that survive -R (generic.c:921-922) */
            if ((info & ITX_F_UNKNOWN) && T.start < ITX_MAX_TID_SEEN) D.tid_unknown_seen[T.start] = 1u;
            long long sel = -1; bool diffsub = false; itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
            const uint32_t chrom = info & ITX_CHROM_MASK;
            itx_query Q; Q.fs = Q.fe = 0; Q.lo = Q.top = 0;
            const bool q_ok = live && chrom != ITX_CHROM_NONE && itx_query_open(D, (int32_t)chrom, T.start, T.end, &Q);
            {
                const uint32_t tmax = __reduce_max_sync(0xffffffffu, q_ok ? Q.top : 0u);
                if (tmax && !(wn && tmax >= wbase + 8u && tmax <= wbase + wn)) {
                    __syncwarp();                              /* the previous rounds' readers are done */
                    wbase = tmax > 24u ? tmax - 24u : 0u;
                    wn = n_elem32 - wbase < ITX_WIN ? n_elem32 - wbase : ITX_WIN;
                    if (lane < wn) {
                        win_iv[lane] = __ldg(reinterpret_cast<const int4 *>(D.iv + wbase + lane));
                        if (stat) {
                            win_meta[lane] = __ldg(reinterpret_cast<const uint4 *>(D.meta + wbase + lane));
                            win_meta2[lane] = __ldg(reinterpret_cast<const int2 *>(D.meta2 + wbase + lane));
                        }
                    }
                    __syncwarp();
                }
            }
            if (q_ok) {
                int32_t nhit = 0; float tcov = 0.0f;
                sel = itx_select_walk(D, Q, itx_iv_window{D, win_iv, wbase, wn}, T.start, T.end, A.o.minCoverage, &nhit, &tcov, &e);
                if (sel == ITX_SEL_LONG) {
                    const itx_sel_cov r = itx_select_multi(*A.Dg, Q, T.start, T.end, nhit);
                    sel = r.sel; tcov = r.cov;
                    if (sel >= 0) e = itx_ld_iv(D, (uint32_t)sel);
                }
                if (sel >= 0 && tcov < A.o.minCoverage) sel = -1;
                if (sel >= 0 && A.o.diffSubfam && (info & ITX_F_HASXA)) {
                    const unsigned long long p = lo + T.rec_off;
                    uint32_t x[9]; G.core(p, x);
                    uint32_t bad = 0;
                    if (itx_mapped_to_diff_subfam(*A.Dg, G, p, x, (int32_t)__ldg(&D.ivf[sel].row), (int32_t)(T.end - T.start), &bad)) diffsub = true;      /* (the index in global memory: an out-of-line walk handed the parameter copy would make every thread copy it to its stack) */
                    if (bad) atomicAdd(&D.status[2], bad);
                }
            }
            const bool counted = sel >= 0 && !diffsub;
            const uint32_t m_cnt = __ballot_sync(0xffffffffu, counted);
            c[12] += __popc(__ballot_sync(0xffffffffu, diffsub));
            c[9] += __popc(m_cnt); c[10] += __popc(m_cnt & m_uniq);
            if (counted) {
                if (stat) {
                    const uint32_t wd = (uint32_t)sel - wbase;
                    uint4 mv; int2 m2v;
                    if (wd < wn) { mv = win_meta[wd]; m2v = win_meta2[wd]; }
                    else { mv = __ldg(reinterpret_cast<const uint4 *>(D.meta + sel)); m2v = __ldg(reinterpret_cast<const int2 *>(D.meta2 + sel)); }
                    itx_meta m; m.cons_start = mv.x; m.cons_end = mv.y; m.row = mv.z; m.sub = mv.w;
                    itx_meta2 m2; m2.fam = m2v.x; m2.cla = m2v.y;
                    const uint32_t hs = 2u * m.sub, hf = 2u * (uint32_t)(D.n_sub + m2.fam), hc = 2u * (uint32_t)(D.n_sub + D.n_fam + m2.cla);
                    if (SMEM_HIST) {
                        atomicAdd(&sh_hist[hs], 1u); atomicAdd(&sh_hist[hf], 1u); atomicAdd(&sh_hist[hc], 1u);
                        if (uniq) { atomicAdd(&sh_hist[hs + 1], 1u); atomicAdd(&sh_hist[hf + 1], 1u); atomicAdd(&sh_hist[hc + 1], 1u); }
                    } else {
                        itx_red_u64(&D.grp[hs], 1ull); itx_red_u64(&D.grp[hf], 1ull); itx_red_u64(&D.grp[hc], 1ull);
                        if (uniq) { itx_red_u64(&D.grp[hs + 1], 1ull); itx_red_u64(&D.grp[hf + 1], 1ull); itx_red_u64(&D.grp[hc + 1], 1ull); }
                    }
                    const uint4 sv = __ldg(reinterpret_cast<const uint4 *>(D.sinfo + m.sub));      /* {len, fold, bp_off} */
                    const uint32_t L = sv.x;
                    uint32_t ja, jb;
                    if (L && itx_cov_range(T.start, T.end - T.start, e.start, e.end, m.cons_start, m.cons_end, L, &ja, &jb)) {
                        const unsigned long long off = (unsigned long long)sv.z | ((unsigned long long)sv.w << 32);
                        itx_red_u32(&D.bp_diff[off + ja], 1u); itx_red_u32(&D.bp_diff[off + jb], 0xffffffffu);
                        if (uniq) { itx_red_u32(&D.bp_diff_u[off + ja], 1u); itx_red_u32(&D.bp_diff_u[off + jb], 0xffffffffu); }
                    }
                } else if (A.o.filter) {
                    itx_red_u32(&D.el_cnt[sel], 1u);
                    if (uniq) itx_red_u32(&D.el_cnt_u[sel], 1u);
                }
            }
            if (A.sel_out && valid) A.sel_out[(size_t)i * A.S + j] = counted ? sel : -1;
            if (A.trace && valid) {
                const unsigned long long r = A.rec_base[i] + j;
                if (r < A.trace_cap) {
                    itx_trace t;
                    t.start = live ? T.start : 0; t.end = live ? T.end : 0;
                    t.tid = (int32_t)G.u32(lo + T.rec_off + 4);
                    t.sel_row = sel >= 0 ? (int32_t)e.row : -1;
                    t.flags = (live ? ITX_T_FRAGMENT : 0u) | (live && uniq ? ITX_T_UNIQ : 0u) | ((live && (info & ITX_F_MINUS)) ? ITX_T_MINUS : 0u) |
                              ((live && (info & ITX_F_HASXA)) ? ITX_T_HAS_XA : 0u) | (diffsub ? ITX_T_DIFFSUB : 0u) | (counted ? ITX_T_COUNTED : 0u) |
                              ((info & ITX_F_DUP) ? ITX_T_DUP : 0u);
                    A.trace[r] = t;
                }
            }
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 13; k++) if (c[k]) atomicAdd(&sh_cnt[k], (unsigned long long)c[k]);
    }
    __syncthreads();
    if (threadIdx.x < 13 && sh_cnt[threadIdx.x]) itx_red_u64(&D.cnt[threadIdx.x], sh_cnt[threadIdx.x]);
    for (uint32_t t = threadIdx.x; t < nh; t += blockDim.x) { const uint32_t v = sh_hist[t]; if (v) itx_red_u64(&D.grp[t], (unsigned long long)v); }
}

/* ------------------------------------------------------------------ K1+K2+K3 in one pass */
/* k_scan: the span kernel's streaming walk (TMA-staged stages, run-predicted chain) with every decoded record going
 * straight into overlap / selection / accumulation, so no tuple ever leaves the SM: the stream is read once and
 * nothing but counters is written.  A span's first record start is still a guess, and a wrong guess would by now
 * have been counted; so the spans' entries and exits are logged, the LAST CTA to finish checks the chain
 * (entry[i] == the exit of the last span before it that held a record start) and notes the first window that fails,
 * and the host -- at the end of the scan, when it reads the counters anyway -- replays every window from the first bad
 * one with sign = -1 (the same guesses, the same additions, negated: integer sums, so the undo is exact) and runs the
 * tuple path (k_decode_span, k_verify, k_fixup, k_overlap) over them instead.  No guess has failed on any generated or
 * converted stream; the path exists for exactness. */
struct itx_scan_args {
    itx_decode_args A;                   /* stream, spans, reference table, options, entry / exit logs, carry, status, work[2] */
    itx_dev_index D;
    const itx_dev_index *Dg;             /* the same in global memory: what the out-of-line functions are handed, so that D stays in the parameter bank */
    int32_t sign;                        /* +1: count; -1: take back what the same call counted */
    uint32_t window;                     /* index of this launch in the scan */
    unsigned long long *carry_log;       /* [window] the carry the window started from (the undo pass starts from it too) */
    uint32_t *first_bad;                 /* smallest window index whose chain check failed; [1] CTAs done; [2] status bits of this launch (folded into
                                          * status[0] by the last CTA only when the launch will not be replayed: what a wrongly guessed span reports is garbage);
                                          * [4..5] (u64) the first record start a scan that began mid-stream settled on */
    uint32_t flags;                      /* ITX_SCAN_* (A/B switches; every combination gives the same counts) */
    /* reads that carry XA:Z and are about to be counted are not decided here: their record offsets are queued for k_xa, which
     * tests the alternates (mapped2diffSubfam) and does their accumulation.  xa_n[0] = entries so far (k_xa zeroes it) */
    unsigned long long *xa_q; uint32_t *xa_n; unsigned long long xa_cap;
};
#define ITX_SCAN_PREFETCH 1u             /* the next stage's bytes are asked into L2 while this stage is worked on */
#define ITX_SCAN_DOMSIZE  2u             /* chain walk predicts with the span's dominant record size, so an odd record costs one step, not two */
#define ITX_SCAN_WINDOW   4u             /* the 32 table entries under the warp's highest bucket end are staged in shared memory, metadata included */
#define ITX_SCAN_WINAHEAD 8u             /* the window the NEXT round will most likely need is fetched with cp.async while this round's tail and the next stage's
                                          * copy, chain walk and decode go on (coordinate-sorted reads move up the table a few entries per round) */
#define ITX_SCAN_EARLY    16u            /* the next stage's bulk copy is issued as soon as the last round of this stage has taken what it needs out of the
                                          * staged bytes (core, CIGAR, aux tags): it flies while the warp does the table walk, selection and accumulation */
#define ITX_SCAN_EVICT    32u            /* stream bytes carry an L2 evict-first hint: they are used once, the interval table and the counters are not */
#define ITX_SCAN_XACOOP   64u            /* XA:Z alternates are tested one LANE per alternate (all alternates of a round side by side) instead of one lane per read */
#define ITX_SCAN_EVICT_PF 128u           /* the evict-first hint on the L2 prefetches too */
#define ITX_SCAN_CARRY    256u           /* the margin of the stage in place becomes the head of the next one inside shared memory: it is not fetched twice */
#define ITX_SCAN_PACK     512u           /* stages start AT a record (16-byte granule) instead of on a 4 KiB boundary and hold up to 32 whole records, one
                                          * round each: with 4 KiB of record starts per stage a 232-byte record (PE-100) fills 18 lanes of a round, packed it
                                          * fills 22; the tail of the buffer behind the last whole record is carried inside shared memory.  Measured SLOWER
                                          * (SE-50 2.23 -> 2.53 ms, PE-100 3.16 -> 3.50 ms): kept as a switch (ITX_SCAN_PACK=1), not the product's choice */
#define ITX_SCAN_SERIAL   1024u          /* a span whose records keep defeating the size prediction (fewer than 2.5 records accepted per step: XA lists, long
                                          * read names of every length) walks the rest of its stages record by record -- 18 instructions per record, all
                                          * lanes alike, against 45 per step of the predicted walk.  A/B switch only: compiled into the product it gains the
                                          * SE-75 + XA stream 3 % and costs SE-50 / PE-100 4 % (a register spilled, a longer loop) */
#define ITX_SCAN_DEFAULT  (ITX_SCAN_DOMSIZE | ITX_SCAN_WINDOW | ITX_SCAN_WINAHEAD | ITX_SCAN_EARLY | ITX_SCAN_XACOOP)
#define ITX_XA_BLK 128u                  /* k_scan -> k_xa queue: a warp reserves this many entries at a time (one atomic on the queue's counter per block, not
                                          * per round: a million and more same-address atomics per launch queued up in L2 and cost cfg 3 two milliseconds);
                                          * what a warp leaves unused of its last block is marked empty (all ones) */
#ifndef ITX_SCAN_NW
#define ITX_SCAN_NW 14                    /* warps per k_scan CTA */
#endif
/* shared memory of a k_scan CTA of NW warps: stages, record-start slots, mbarriers, table windows; the histogram follows */
/* one contiguous block per warp (every pointer is the warp's base plus a constant) */
#define ITX_SCAN_WARP_BYTES (ITX_STAGE + ITX_MARGIN + ITX_POS_SLOTS * 2u + 16u + ITX_WIN_BYTES)
#define ITX_SCAN_SMEM_BASE(NW) ((NW) * ITX_SCAN_WARP_BYTES)
#define ITX_SCAN_CTAS(NW) ((NW) <= 8 ? 3 : ((NW) >= 32 ? 1 : 2))          /* 8 warps x 3 CTAs (80 registers) or 14 warps x 2 CTAs (72 registers) per SM */

__device__ __forceinline__ unsigned long long itx_policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void itx_bulk_g2s_hint(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, unsigned long long pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ void itx_prefetch_l2_hint(const void *src, uint32_t bytes, unsigned long long pol) {
    asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(src), "r"(bytes), "l"(pol) : "memory");
}


/* The chain check of a launch group, by its last CTA (k_scan) -- also what the sharded scan's host side applies between ranks.
 * A span that holds no record start at all (a record longer than a span runs over it) logs NONE for both its entry and its exit:
 * the exit that counts for span i is that of the last span before it which has one.  Span i is consistent when its guessed entry
 * IS that exit -- or, if it found no plausible start, when the chain does run over it entirely (or had already ended). */
__device__ __forceinline__ unsigned long long itx_effective_exit(const unsigned long long *exit_, uint32_t j) {
    unsigned long long x = __ldcg(exit_ + j);
    while (x == ITX_OFF_NONE && j > 0) { j--; x = __ldcg(exit_ + j); }
    return x;
}

/* A span's first record start, guessed out of its first staged bytes (itx_plausible2's test, 32 offsets per step: the core of every
 * offset comes out of the stage with plain shared-memory loads and is tested without branches; the second record is looked at for
 * the survivors).  Once per span, so it is kept out of line: the stage loop is bound by instruction fetch as much as by issue, and
 * these few hundred instructions are not part of it.  Returns the span-relative offset or 0xffffffff. */
__device__ __noinline__ uint32_t itx_guess_span(const uint8_t *buf, const uint8_t *g, unsigned long long lo, uint32_t hi, uint32_t nb, unsigned long long len, int32_t n_ref) {
    const uint32_t lane = threadIdx.x & 31;
    const itx_src_stage S0{buf, g, lo, nb};
    uint32_t p = 0xffffffffu;
    for (uint32_t base = 0; base < hi; base += 32) {
        const uint32_t d = base + lane;
        const unsigned long long q = lo + d;
        bool ok = false;
        if (d < hi && q + 36 <= len) {
            uint32_t x[9];
            if (base + 32u + 40u <= nb) {                     /* warp-uniform: every lane's core lies in the stage */
                const uint32_t *wq = reinterpret_cast<const uint32_t *>(buf + (d & ~3u)); const uint32_t sh = (d & 3u) * 8u;
                uint32_t wv[10];
#pragma unroll
                for (int k = 0; k < 10; k++) wv[k] = wq[k];
#pragma unroll
                for (int k = 0; k < 9; k++) x[k] = itx_funnel_r(wv[k], wv[k + 1], sh);
            } else S0.core(q, x);
            ok = itx_plausible2_core(S0, x, q, len, n_ref);
        }
        const uint32_t m = __ballot_sync(0xffffffffu, ok);
        if (m) { p = base + (uint32_t)__ffs((int)m) - 1; break; }
    }
    return p;
}
/* a record that runs past the staged bytes (longer than the margin): decoded with the bounds-tested source, out of line */
__device__ __noinline__ itx_tuple itx_decode_long(const uint8_t *buf, const uint8_t *g, unsigned long long c_lo64, uint32_t nb, uint32_t rec_rel,
                                                  const itx_tidinfo *tid, int32_t n_ref, const itx_dev_opts o) {
    const itx_src_stage S{buf, g, c_lo64, nb};
    uint32_t x[9]; S.core(c_lo64 + rec_rel, x);
    return itx_decode_record<itx_src_stage, false>(S, c_lo64 + rec_rel, x, 0u, tid, n_ref, o);
}
/* the XA tag of one record (its type byte, relative to the stage; 0: none): bam_aux_get's walk over the aux area, out of line --
 * only records whose aux area can hold a list at all get here */
__device__ __noinline__ uint32_t itx_find_xa_tag(const uint8_t *buf, const uint8_t *g, unsigned long long c_lo64, uint32_t nb, uint32_t rec_rel, uint32_t aux_rel, uint32_t rec_bytes) {
    const itx_src_stage S{buf, g, c_lo64, nb};
    const uint64_t rp = c_lo64 + rec_rel, a0 = rp + aux_rel, aend = rp + rec_bytes;
    const uint64_t xa = itx_aux_find(S, a0, aend, 'X', 'A');
    return (xa && xa < aend) ? (uint32_t)(xa - c_lo64) : 0u;
}
/* the 13 report counters of a warp (8-bit fields of three registers per lane) into the CTA's totals: every 255 rounds, out of line */
__device__ __noinline__ void itx_flush_counters(uint32_t pa, uint32_t pb, uint32_t pc, unsigned long long *sh_cnt) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t a0_ = __reduce_add_sync(0xffffffffu, pa & 0x00ff00ffu), a1_ = __reduce_add_sync(0xffffffffu, (pa >> 8) & 0x00ff00ffu);
    const uint32_t b0_ = __reduce_add_sync(0xffffffffu, pb & 0x00ff00ffu), b1_ = __reduce_add_sync(0xffffffffu, (pb >> 8) & 0x00ff00ffu);
    const uint32_t c0_ = __reduce_add_sync(0xffffffffu, pc & 0x00ff00ffu), c1_ = __reduce_add_sync(0xffffffffu, (pc >> 8) & 0x00ff00ffu);
    if (lane == 0) {
        if (a0_ & 0xffffu) atomicAdd(&sh_cnt[0], (unsigned long long)(a0_ & 0xffffu));
        if (a1_ & 0xffffu) atomicAdd(&sh_cnt[1], (unsigned long long)(a1_ & 0xffffu));
        if (a0_ >> 16) atomicAdd(&sh_cnt[2], (unsigned long long)(a0_ >> 16));
        if (a1_ >> 16) atomicAdd(&sh_cnt[3], (unsigned long long)(a1_ >> 16));
        if (b0_ & 0xffffu) atomicAdd(&sh_cnt[4], (unsigned long long)(b0_ & 0xffffu));
        if (b1_ & 0xffffu) atomicAdd(&sh_cnt[5], (unsigned long long)(b1_ & 0xffffu));
        if (b0_ >> 16) atomicAdd(&sh_cnt[6], (unsigned long long)(b0_ >> 16));
        if (b1_ >> 16) { atomicAdd(&sh_cnt[7], (unsigned long long)(b1_ >> 16)); atomicAdd(&sh_cnt[11], (unsigned long long)(b1_ >> 16)); }
        if (c0_ & 0xffffu) atomicAdd(&sh_cnt[9], (unsigned long long)(c0_ & 0xffffu));
        if (c1_ & 0xffffu) atomicAdd(&sh_cnt[10], (unsigned long long)(c1_ & 0xffffu));
        if (c0_ >> 16) atomicAdd(&sh_cnt[12], (unsigned long long)(c0_ >> 16));
    }
}
/* AB = false: the product build -- the switches above are compile-time constants (ITX_SCAN_PRODUCT), so the paths they would
 * select between are not in the loop at all (the loop is bound by instruction issue AND fetch: every instruction that is not
 * there helps); AB = true: the switches are read from P.flags (tests and measurements: every combination gives the same counts) */
#ifndef ITX_SCAN_PRODUCT
#define ITX_SCAN_PRODUCT (ITX_SCAN_DEFAULT | ITX_SCAN_EVICT | ITX_SCAN_CARRY)      /* not ITX_SCAN_PACK, not ITX_SCAN_SERIAL: measured slower (DESIGN.md 6) */
#endif
template <bool SMEM_HIST, int NW, bool AB, bool PACK = false>
__global__ void __launch_bounds__(NW * 32, ITX_SCAN_CTAS(NW)) k_scan(const itx_scan_args P) {
    extern __shared__ __align__(128) uint8_t itx_smem[];
    __shared__ unsigned long long sh_cnt[13];
    __shared__ uint32_t sh_last;
    const itx_decode_args &A = P.A; const itx_dev_index &D = P.D;
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    constexpr uint32_t STG = ITX_STAGE + ITX_MARGIN;
    uint8_t *buf = itx_smem + w * ITX_SCAN_WARP_BYTES;
    uint16_t *pos = reinterpret_cast<uint16_t *>(buf + STG);
    const uint32_t buf_s = itx_smem_addr(buf);
    const uint32_t bar_s = buf_s + STG + ITX_POS_SLOTS * 2u;
    int4 *win_iv = reinterpret_cast<int4 *>(buf + STG + ITX_POS_SLOTS * 2u + 16u);
    uint4 *win_meta = reinterpret_cast<uint4 *>(win_iv + ITX_WIN);
    int2 *win_meta2 = reinterpret_cast<int2 *>(win_meta + ITX_WIN);
    uint32_t *sh_hist = reinterpret_cast<uint32_t *>(itx_smem + ITX_SCAN_SMEM_BASE(NW));
    const uint32_t nh = SMEM_HIST ? 2u * (uint32_t)(D.n_sub + D.n_fam + D.n_cla) : 0u;
    for (uint32_t t = threadIdx.x; t < nh; t += blockDim.x) sh_hist[t] = 0;
    if (threadIdx.x < 13) sh_cnt[threadIdx.x] = 0;
    if (lane == 0) { itx_mbar_init(bar_s, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    uint32_t *xa_blk = reinterpret_cast<uint32_t *>(buf + STG + ITX_POS_SLOTS * 2u + 8u);      /* the warp's block of the XA queue: [0] first entry, [1] entries used (beside the mbarrier) */
    if (lane == 0) { xa_blk[0] = 0u; xa_blk[1] = ITX_XA_BLK; }
    __syncthreads();
    const bool neg = P.sign < 0;
#define one (neg ? 0xffffffffu : 1u)
#define minus_one (neg ? 1u : 0xffffffffu)
#define one64 (neg ? ~0ull : 1ull)
    const bool stat = A.o.filter == 0 && D.stat_mode;
    const uint32_t flags = AB ? P.flags : (uint32_t)(ITX_SCAN_PRODUCT | (PACK ? ITX_SCAN_PACK : 0u));
    const bool f_pack = flags & ITX_SCAN_PACK, f_serial = flags & ITX_SCAN_SERIAL;
    const bool f_prefetch = flags & ITX_SCAN_PREFETCH, f_dom = flags & ITX_SCAN_DOMSIZE, f_win = flags & ITX_SCAN_WINDOW;
    const bool f_ahead = f_win && (flags & ITX_SCAN_WINAHEAD), f_early = flags & ITX_SCAN_EARLY;
    const bool f_evict = flags & ITX_SCAN_EVICT, f_evict_pf = flags & ITX_SCAN_EVICT_PF, f_carry = flags & ITX_SCAN_CARRY;
#define n_elem32 (D.n_elem > 0xffffffffll ? 0xffffffffu : (uint32_t)D.n_elem)
    uint32_t wspec = 0xffffffffu;                               /* first table entry of the window fetched ahead (none yet) */
    /* the 13 report counters: every lane counts its own records in 8-bit fields of three registers (no votes, no
     * popcounts); the fields are summed over the warp and added to the CTA's totals before any of them can reach 256 */
    uint32_t pa = 0, pb = 0, pc = 0, n_rounds = 0;
    /* one stage into shared memory: a TMA bulk copy of ITX_STAGE + ITX_MARGIN bytes (less at the end of the stream), and what
     * the stage after it adds on its way into L2 meanwhile; the caller has made sure that every lane is done with the old bytes */
#define ITX_SCAN_ISSUE(c_lo_, rest_, nb_out_, carry_) do { \
        nb_out_ = (rest_) > STG ? STG : (uint32_t)(rest_); \
        /* the stage that follows the one in place begins with that one's margin: those bytes are moved inside shared memory (32 per \
         * lane) and only the rest comes over from L2 / HBM -- the margin is not fetched twice */ \
        const bool carry__ = f_carry && (carry_) && nb_out_ > ITX_MARGIN; \
        if (carry__) { \
            const uint4 t0_ = *reinterpret_cast<const uint4 *>(buf + ITX_STAGE + lane * 32u), t1_ = *reinterpret_cast<const uint4 *>(buf + ITX_STAGE + lane * 32u + 16u); \
            *reinterpret_cast<uint4 *>(buf + lane * 32u) = t0_; *reinterpret_cast<uint4 *>(buf + lane * 32u + 16u) = t1_; \
        } \
        __syncwarp(); \
        if (lane == 0) { \
            const uint32_t skip_ = carry__ ? ITX_MARGIN : 0u; \
            const uint32_t bytes_ = ((nb_out_ + 15u) & ~15u) - skip_;     /* the buffer's 64 bytes of slack cover the round-up */ \
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); \
            itx_mbar_expect_tx(bar_s, bytes_); \
            if (f_evict) itx_bulk_g2s_hint(buf_s + skip_, A.b + lo + (c_lo_) + skip_, bytes_, bar_s, itx_policy_evict_first()); else itx_bulk_g2s(buf_s + skip_, A.b + lo + (c_lo_) + skip_, bytes_, bar_s); \
            if (f_prefetch && (c_lo_) + ITX_STAGE < hi && (rest_) >= STG + ITX_STAGE) { \
                if (f_evict_pf) itx_prefetch_l2_hint(A.b + lo + (c_lo_) + STG, ITX_STAGE, itx_policy_evict_first()); else itx_prefetch_l2(A.b + lo + (c_lo_) + STG, ITX_STAGE); \
            } \
        } \
    } while (0)
    /* the packed geometry's issue: `tail_` bytes at the end of the buffer in place (a multiple of 16; 0: none) are the head of the new
     * stage -- moved to the front, 16 bytes per lane and step, every step read by all lanes before any of them writes -- and the
     * bulk copy brings what follows them */
#define ITX_SCAN_ISSUE_PACK(c_lo_, rest_, nb_prev_, nb_out_, tail_) do { \
        const uint32_t nbp__ = (nb_prev_); \
        nb_out_ = (rest_) > STG ? STG : (uint32_t)(rest_); \
        uint32_t tl__ = (tail_); \
        if (!(f_carry && nb_out_ > tl__)) tl__ = 0u; \
        for (uint32_t b__ = 0; b__ < tl__; b__ += 512u) { \
            const uint32_t c__ = b__ + lane * 16u; \
            uint4 t__ = make_uint4(0u, 0u, 0u, 0u); \
            if (c__ < tl__) t__ = *reinterpret_cast<const uint4 *>(buf + (nbp__ - tl__) + c__); \
            __syncwarp(); \
            if (c__ < tl__) *reinterpret_cast<uint4 *>(buf + c__) = t__; \
        } \
        __syncwarp(); \
        if (lane == 0) { \
            const uint32_t bytes__ = ((nb_out_ + 15u) & ~15u) - tl__; \
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); \
            itx_mbar_expect_tx(bar_s, bytes__); \
            if (f_evict) itx_bulk_g2s_hint(buf_s + tl__, A.b + lo + (c_lo_) + tl__, bytes__, bar_s, itx_policy_evict_first()); else itx_bulk_g2s(buf_s + tl__, A.b + lo + (c_lo_) + tl__, bytes__, bar_s); \
        } \
    } while (0)
    uint32_t parity = 0;
    bool dead = false;
    for (;;) {
        uint32_t i = 0;
        if (lane == 0) i = atomicAdd(&A.work[2], 1u);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= A.nchunks || dead) break;
        /* Inside a span everything is kept relative to its first byte, in 32 bits (a span is at most 1 MiB and a record
         * shorter than 2^31 bytes); the two chain sentinels keep their low words (0xfffffffe ended, 0xffffffff none). */
        const unsigned long long lo = (A.k0 + i) * (unsigned long long)A.C;
        /* record starts at or past A.own belong to whoever scans the stream from there on (the next rank of a sharded scan) */
        const uint32_t hi = A.own - lo < A.C ? (uint32_t)(A.own - lo) : A.C;
        /* the span's first record start: known for the window's first span (unless the scan starts in the middle of a stream:
         * ITX_OFF_GUESS); otherwise guessed out of the span's first stage, which is needed in shared memory anyway */
        uint32_t p = 0xffffffffu;
        bool guess = i != 0;
        if (!guess) {
            unsigned long long p0;
            if (neg) p0 = P.carry_log[P.window];
            else { p0 = *A.carry; if (lane == 0) P.carry_log[P.window] = p0; }
            if (p0 == ITX_OFF_GUESS) guess = true;
            else {
                if (lane == 0) A.entry[i] = p0;
                p = p0 >= ITX_OFF_END ? (uint32_t)p0 : (p0 - lo < 0xfffffff0ull ? (uint32_t)(p0 - lo) : 0xfffffffeu);
            }
        }
        uint32_t staged = 0xffffffffu;                         /* span offset of the stage now in shared memory */
        uint32_t inflight = 0xffffffffu;                       /* span offset of the stage whose copy was issued early (none) */
        uint32_t nb = 0;
        uint32_t szd = 0;                                      /* the span's dominant record size (0: none yet) */
        bool guessed = false;                                  /* packed geometry: the stage the guess was made in is kept for the first records */
        bool ser = false;                                      /* the size prediction does badly in this span: walk record by record */
        for (;;) {
            if (guess ? hi == 0u : !(p < hi)) { if (guess && lane == 0) A.entry[i] = ITX_OFF_NONE; break; }
            /* packed: a stage starts at the 16-byte granule of its first record (the span's first stage, staged for the guess, is kept
             * when the guess lies in its first 512 bytes); otherwise on a 4 KiB boundary */
            const uint32_t c_lo = guess ? 0u : (f_pack ? ((guessed && p < 512u) ? 0u : p & ~15u) : p & ~(ITX_STAGE - 1u));
            guessed = false;
            const uint32_t c_hi = f_pack ? hi : (c_lo + ITX_STAGE < hi ? c_lo + ITX_STAGE : hi);
            const unsigned long long rest = A.len - lo - c_lo;                 /* bytes of the stream from this stage on */
            if (staged != c_lo) {
                if (inflight == c_lo) nb = rest > STG ? STG : (uint32_t)rest;      /* on its way since the last round of the previous stage */
                else if (f_pack) {
                    const uint32_t tail = (staged != 0xffffffffu && nb == STG && c_lo > staged && c_lo - staged < STG) ? staged + STG - c_lo : 0u;
                    ITX_SCAN_ISSUE_PACK(c_lo, rest, nb, nb, tail);
                }
                else ITX_SCAN_ISSUE(c_lo, rest, nb, staged + ITX_STAGE == c_lo && nb == STG);      /* (every lane is done reading the previous stage: the macro's __syncwarp ... */
                if (!itx_mbar_wait(bar_s, parity, A.status)) { dead = true; break; }
                parity ^= 1u;
                staged = c_lo; inflight = 0xffffffffu;
            }
            if (guess) {
                p = itx_guess_span(buf, A.b, lo, hi, nb, A.len, A.n_ref);
                if (lane == 0) A.entry[i] = p == 0xffffffffu ? ITX_OFF_NONE : lo + p;
                guess = false; guessed = true;
                continue;
            }
            /* the chain of this stage, out of shared memory.  Lane 0 holds the record at q; lane k >= 1 looks where record k
             * would start if records 1.. had the dominant size, and the run of lanes that find that size there is accepted
             * in one step (each accepted start is the previous record's start + its verified size: the exact chain).
             * Offsets are stage-relative and 32 bits wide; records of 64 KiB and more are stepped over one at a time.
             * q ends as the offset of the next stage's first record, or as 0xffffffff when the chain ends here. */
            uint32_t n = 0;
            uint32_t q = p - c_lo;
            {
                const uint32_t qh = c_hi - c_lo;
                const uint32_t room32 = rest > 0x7fffffffull ? 0x7fffffffu : (uint32_t)rest;
                uint32_t q_end = q;                                                /* where the last whole record of the stage ends */
                if (f_pack) {
                    /* packed: up to 32 records that lie in the staged bytes as a whole (one round); the stage after this one starts at
                     * the first record left over.  A record longer than the buffer is taken alone, at the head of a stage of its own
                     * (its core is staged, the rest comes from global memory: itx_decode_long). */
                    while (q < qh && n < 32u) {
                        q_end = q;
                        if (q + 36u > nb) { if (q + 36u > room32) q = 0xffffffffu; break; }      /* the stream ends inside the core: the chain does; else: the next stage starts here */
                        const uint32_t bs0 = itx_buf_u32(buf, q);
                        const uint32_t sz0 = bs0 + 4u;
                        if ((int32_t)bs0 < 32 || sz0 > room32 - q) { q = 0xffffffffu; break; }
                        if (sz0 > nb - q) {                                            /* not whole in the staged bytes */
                            if (n == 0u && q < 16u) { if (lane == 0) pos[0] = (uint16_t)q; n = 1u; q += sz0; szd = 0u; }
                            break;
                        }
                        const uint32_t szp = szd ? szd : sz0;
                        uint32_t run = 1u, pk = q;
                        if ((sz0 | szp) < 0x10000u) {                                  /* warp-uniform */
                            const bool same = itx_chain_lane(buf, q, sz0, szp, lane, qh, nb, &pk);      /* (nb <= room32: predicted records end inside the staged bytes) */
                            const uint32_t m = __ballot_sync(0xffffffffu, same);       /* bit 0 is always set */
                            run = m == 0xffffffffu ? 32u : (uint32_t)__ffs((int)~m) - 1u;
                        }
                        szd = (f_dom && run >= 2u) ? szp : 0u;
                        if (run > 32u - n) run = 32u - n;
                        if (lane < run) pos[n + lane] = (uint16_t)pk;
                        n += run;
                        q += sz0 + (run - 1u) * szp;
                    }
                } else if (f_serial && ser) {
                    /* record by record, every lane the same walk (the lane whose turn it is notes the start) */
                    while (q < qh) {
                        q_end = q;
                        if (q + 36u > room32) { q = 0xffffffffu; break; }
                        const uint32_t bs0 = itx_buf_u32(buf, q);
                        if ((int32_t)bs0 < 32 || bs0 + 4u > room32 - q) { q = 0xffffffffu; break; }
                        if ((n & 31u) == lane && n < ITX_POS_SLOTS) pos[n] = (uint16_t)q;
                        n++;
                        q += bs0 + 4u;
                    }
                } else {
                uint32_t steps = 0;
                while (q < qh) {
                    q_end = q;
                    steps++;
                    if (q + 36u > room32) { q = 0xffffffffu; break; }
                    const uint32_t bs0 = itx_buf_u32(buf, q);
                    const uint32_t sz0 = bs0 + 4u;
                    if ((int32_t)bs0 < 32 || sz0 > room32 - q) { q = 0xffffffffu; break; }
                    const uint32_t szp = szd ? szd : sz0;
                    uint32_t run = 1u, pk = q;
                    if ((sz0 | szp) < 0x10000u) {                                  /* warp-uniform */
                        const bool same = itx_chain_lane(buf, q, sz0, szp, lane, qh, room32, &pk);
                        const uint32_t m = __ballot_sync(0xffffffffu, same);       /* bit 0 is always set */
                        run = m == 0xffffffffu ? 32u : (uint32_t)__ffs((int)~m) - 1u;
                    }
                    if (lane < run && n + lane < ITX_POS_SLOTS) pos[n + lane] = (uint16_t)pk;
                    n += run;
                    q += sz0 + (run - 1u) * szp;
                    szd = (f_dom && run >= 2u) ? szp : 0u;
                }
                if (f_serial && n >= 8u && steps * 5u > n * 2u) ser = true;
                }
                if (q != 0xffffffffu) q_end = q;
                if (lane == 0 && A.avail < lo + c_lo + q_end) atomicOr(P.first_bad + 2, 2u);              /* a record longer than the staged window */
            }
            __syncwarp();
            const unsigned long long c_lo64 = lo + c_lo;
            const itx_src_stage S{buf, A.b, c_lo64, nb};
            uint32_t tmax_last = 0;                            /* highest table entry any round of this stage started from */
            for (uint32_t j0 = 0; j0 < n; j0 += 32) {
                const uint32_t j = j0 + lane; const bool valid = j < n;
                /* ---- everything this round needs out of the staged bytes: core, CIGAR, the XA / NM tags */
                itx_tuple T; T.start = T.end = T.rec_off = 0; T.info = 0;
                uint32_t xa_rel = 0;                                               /* stage-relative offset of the XA tag's type byte (0: the read carries no XA) */
                if (valid) {
                    const unsigned long long rp = c_lo64 + pos[j];
                    uint32_t x[9];
                    {   /* the chain walk has made sure that the 36 bytes of the core lie inside the stream, and a record starts inside the
                         * stage: they are in the staged bytes -- no bounds test, no path to global memory */
                        const uint32_t d = pos[j];
                        const uint32_t *wq = reinterpret_cast<const uint32_t *>(buf + (d & ~3u)); const uint32_t sh = (d & 3u) * 8u;
                        uint32_t wv[10];
#pragma unroll
                        for (int k = 0; k < 10; k++) wv[k] = wq[k];
#pragma unroll
                        for (int k = 0; k < 9; k++) x[k] = itx_funnel_r(wv[k], wv[k + 1], sh);
                    }
                    /* a record that lies inside the staged bytes (all but the ones longer than the margin) is read without bounds
                     * tests; XA is looked for right here, below */
                    if (pos[j] + 4u + x[0] <= nb) T = itx_decode_record<itx_src_flat, false>(itx_src_flat{buf, c_lo64}, rp, x, 0u, A.tid, A.n_ref, A.o);
                    else T = itx_decode_long(buf, A.b, c_lo64, nb, pos[j], A.tid, A.n_ref, A.o);
                    if (A.o.diffSubfam && (T.info & ITX_F_FRAG) && (T.info & ITX_CHROM_MASK) != ITX_CHROM_NONE) {
                        /* "XA" + type + at least one character + NUL: a shorter aux area cannot hold a list of alternates */
                        const uint32_t lq = x[3] & 0xffu, nc = x[4] & 0xffffu; const int32_t ls = (int32_t)x[5];
                        const int64_t fixed = 36ll + lq + 4ll * nc + (int64_t)ls + (int64_t)((ls + 1) / 2);
                        if (fixed >= 36 && fixed + 5 <= 4ll + (int64_t)x[0]) xa_rel = itx_find_xa_tag(buf, A.b, c_lo64, nb, pos[j], (uint32_t)fixed, x[0] + 4u);
                    }
                }
                /* the last round of a stage is done with the staged bytes: the next stage's copy starts now */
                if (f_early && j0 + 32u >= n && q != 0xffffffffu && c_lo + q < hi) {
                    const uint32_t c_nx = f_pack ? (c_lo + q) & ~15u : (c_lo + q) & ~(ITX_STAGE - 1u);
                    const unsigned long long rest_nx = A.len - lo - c_nx;
                    uint32_t nb_nx;
                    if (f_pack) {
                        const uint32_t tail = (nb == STG && c_nx > c_lo && c_nx - c_lo < STG) ? c_lo + STG - c_nx : 0u;
                        ITX_SCAN_ISSUE_PACK(c_nx, rest_nx, nb, nb_nx, tail);
                    } else ITX_SCAN_ISSUE(c_nx, rest_nx, nb_nx, c_nx == c_lo + ITX_STAGE && nb == STG);
                    (void)nb_nx;
                    inflight = c_nx;
                }
                const uint32_t info = T.info;
                const bool frag = info & ITX_F_FRAG, uniq = info & ITX_F_UNIQ;
                {   /* read_end1/2, *_mapped, *_used, reads_mapped, reads_mapped_unique (= reads_nonredundant_unique without -R) */
                    const uint32_t s2 = (info >> 28) & 1u, ns2 = s2 ^ 1u, mp = (info >> 29) & 1u, us = (info >> 30) & 1u, fr = (info >> 24) & 1u, uq = (info >> 25) & 1u;
                    pa += ((valid ? 1u : 0u) & ns2) | (s2 << 8) | ((mp & ns2) << 16) | ((mp & s2) << 24);
                    pb += (us & ns2) | ((us & s2) << 8) | (fr << 16) | ((fr & uq) << 24);
                }
                /* marks of THIS launch: the last CTA folds them into the scan's marks only if the launch stands (a plain store: every
                 * read of such a chromosome hits the same word, and reductions on one address serialise in L2) */
                if ((info & ITX_F_UNKNOWN) && T.start < ITX_MAX_TID_SEEN) D.tid_unknown_seen[ITX_MAX_TID_SEEN + T.start] = 1u;
                long long sel = -1; const bool diffsub = false; itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
                const uint32_t chrom = info & ITX_CHROM_MASK;
                itx_query Q; Q.fs = Q.fe = 0; Q.lo = Q.top = 0;
                const bool q_ok = frag && chrom != ITX_CHROM_NONE && itx_query_open(D, (int32_t)chrom, T.start, T.end, &Q);
                /* the table window of this round: the ITX_WIN entries below the highest bucket end any lane starts from
                 * (coordinate-sorted reads walk the same few entries), loaded once, coalesced, with their metadata */
                uint32_t wbase = 0, wn = 0, tmax = 0;
                if (f_win) {
                    tmax = __reduce_max_sync(0xffffffffu, q_ok ? Q.top : 0u);
                    if (tmax) {
                        if (wspec != 0xffffffffu) itx_cp_async_wait_all();
                        __syncwarp();                          /* the window fetched ahead has landed; the previous round's readers are done */
                        if (wspec != 0xffffffffu && tmax >= wspec + 8u && tmax <= wspec + ITX_WIN) {
                            wbase = wspec; wn = n_elem32 - wspec < ITX_WIN ? n_elem32 - wspec : ITX_WIN;     /* it covers this round */
                        } else {
                            wbase = tmax > ITX_WIN ? tmax - ITX_WIN : 0u; wn = tmax - wbase;
                            if (lane < wn) {
                                win_iv[lane] = __ldg(reinterpret_cast<const int4 *>(D.iv + wbase + lane));
                                if (stat) {
                                    win_meta[lane] = __ldg(reinterpret_cast<const uint4 *>(D.meta + wbase + lane));
                                    win_meta2[lane] = __ldg(reinterpret_cast<const int2 *>(D.meta2 + wbase + lane));
                                }
                            }
                            wspec = 0xffffffffu;
                            __syncwarp();
                        }
                    }
                }
                int32_t nhit = 0; float tcov = 0.0f;
                if (q_ok) sel = itx_select_walk(D, Q, itx_iv_window{D, win_iv, wbase, wn}, T.start, T.end, A.o.minCoverage, &nhit, &tcov, &e);
                /* the out-of-line paths (hit lists longer than four, XA alternates) sit in regions of their own: a call inside
                 * the region above would make every lane that leaves it wait for a spilled convergence barrier */
                if (sel == ITX_SEL_LONG) {
                    const itx_sel_cov r = itx_select_multi(*P.Dg, Q, T.start, T.end, nhit);
                    sel = r.sel; tcov = r.cov;
                    if (sel >= 0) e = itx_ld_iv(D, (uint32_t)sel);
                }
                if (sel >= 0 && tcov < A.o.minCoverage) sel = -1;
                /* ---- reads with XA:Z alternates that are about to be counted go to k_xa (mapped2diffSubfam + their accumulation) */
                {
                    const bool xa_go = sel >= 0 && xa_rel != 0u;
                    const uint32_t m_xa = __ballot_sync(0xffffffffu, xa_go);
                    if (m_xa) {
                        const uint32_t cnt = (uint32_t)__popc(m_xa);
                        uint32_t qb = xa_blk[0], used = xa_blk[1];
                        if (used + cnt > ITX_XA_BLK) {         /* the block cannot take this round: its rest is marked empty, the next one reserved */
                            if (qb + ITX_XA_BLK <= P.xa_cap) for (uint32_t t = used + lane; t < ITX_XA_BLK; t += 32u) P.xa_q[qb + t] = ~0ull;
                            if (lane == 0) qb = atomicAdd(P.xa_n, ITX_XA_BLK);
                            qb = __shfl_sync(0xffffffffu, qb, 0); used = 0u;
                        }
                        if (xa_go) {
                            if (qb + ITX_XA_BLK <= P.xa_cap) P.xa_q[qb + used + (uint32_t)__popc(m_xa & ((1u << lane) - 1u))] = c_lo64 + pos[j];
                            else atomicOr(&A.status[0], 8u);       /* cannot happen: the queue holds one entry per 42 bytes of stream and a block per warp on top */
                            sel = -1;
                        }
                        __syncwarp();
                        if (lane == 0) { xa_blk[0] = qb; xa_blk[1] = used + cnt; }
                        __syncwarp();
                    }
                }
                const bool counted = sel >= 0 && !diffsub;
                pc += (counted ? 1u : 0u) | ((counted && uniq ? 1u : 0u) << 8) | ((diffsub ? 1u : 0u) << 16);      /* reads_repeat, reads_repeat_unique, reads_diff_subfam */
                if (++n_rounds == 255u) { itx_flush_counters(pa, pb, pc, sh_cnt); pa = pb = pc = 0; n_rounds = 0; }
                if (counted) {
                    if (stat) {
                        const uint32_t wd = (uint32_t)sel - wbase;
                        uint4 mv; int2 m2v;
                        if (wd < wn) { mv = win_meta[wd]; m2v = win_meta2[wd]; }
                        else { mv = __ldg(reinterpret_cast<const uint4 *>(D.meta + sel)); m2v = __ldg(reinterpret_cast<const int2 *>(D.meta2 + sel)); }
                        itx_meta m; m.cons_start = mv.x; m.cons_end = mv.y; m.row = mv.z; m.sub = mv.w;
                        const uint32_t hs = 2u * m.sub, hf = 2u * (uint32_t)(D.n_sub + m2v.x), hc = 2u * (uint32_t)(D.n_sub + D.n_fam + m2v.y);
                        if (SMEM_HIST) {
                            atomicAdd(&sh_hist[hs], 1u); atomicAdd(&sh_hist[hf], 1u); atomicAdd(&sh_hist[hc], 1u);
                            if (uniq) { atomicAdd(&sh_hist[hs + 1], 1u); atomicAdd(&sh_hist[hf + 1], 1u); atomicAdd(&sh_hist[hc + 1], 1u); }
                        } else {
                            itx_red_u64(&D.grp[hs], one64); itx_red_u64(&D.grp[hf], one64); itx_red_u64(&D.grp[hc], one64);
                            if (uniq) { itx_red_u64(&D.grp[hs + 1], one64); itx_red_u64(&D.grp[hf + 1], one64); itx_red_u64(&D.grp[hc + 1], one64); }
                        }
                        const uint4 sv = __ldg(reinterpret_cast<const uint4 *>(D.sinfo + m.sub));
                        const uint32_t L = sv.x;
                        uint32_t ja, jb;
                        if (L && itx_cov_range(T.start, T.end - T.start, e.start, e.end, m.cons_start, m.cons_end, L, &ja, &jb)) {
                            const unsigned long long off = (unsigned long long)sv.z | ((unsigned long long)sv.w << 32);
                            itx_red_u32(&D.bp_diff[off + ja], one); itx_red_u32(&D.bp_diff[off + jb], minus_one);
                            if (uniq) { itx_red_u32(&D.bp_diff_u[off + ja], one); itx_red_u32(&D.bp_diff_u[off + jb], minus_one); }
                        }
                    } else if (A.o.filter) {
                        itx_red_u32(&D.el_cnt[sel], one);
                        if (uniq) itx_red_u32(&D.el_cnt_u[sel], one);
                    }
                }
                if (tmax) tmax_last = tmax;
            }
            /* the window the next stage will most likely need, unless the one in place still has room above this stage's
             * highest entry (issued out here, after the rounds: a spilled register reloaded right behind these copies
             * would wait for them) */
            if (f_ahead && tmax_last && !(wspec != 0xffffffffu && tmax_last + 8u <= wspec + ITX_WIN)) {
                const uint32_t nbase = tmax_last > 20u ? tmax_last - 20u : 0u;
                __syncwarp();                                  /* the last round's readers are done */
                if (nbase + lane < n_elem32) {
                    itx_cp_async16(win_iv + lane, D.iv + nbase + lane);
                    if (stat) { itx_cp_async16(win_meta + lane, D.meta + nbase + lane); itx_cp_async8(win_meta2 + lane, D.meta2 + nbase + lane); }
                }
                wspec = nbase;
            }
            if (q == 0xffffffffu) { p = 0xfffffffeu; break; }
            p = c_lo + q;
        }
        if (lane == 0) A.exit_[i] = p >= 0xfffffffeu ? (0xffffffff00000000ull | p) : lo + p;
    }
    itx_cp_async_wait_all();                                   /* a window fetched ahead and never used */
    {   /* what is left of the warp's block of the XA queue is marked empty */
        const uint32_t qb = xa_blk[0], used = xa_blk[1];
        if (used < ITX_XA_BLK && qb + ITX_XA_BLK <= P.xa_cap) for (uint32_t t = used + lane; t < ITX_XA_BLK; t += 32u) P.xa_q[qb + t] = ~0ull;
    }
    itx_flush_counters(pa, pb, pc, sh_cnt);
    __syncthreads();
    if (threadIdx.x < 13 && sh_cnt[threadIdx.x]) itx_red_u64(&D.cnt[threadIdx.x], neg ? 0ull - sh_cnt[threadIdx.x] : sh_cnt[threadIdx.x]);
    for (uint32_t t = threadIdx.x; t < nh; t += blockDim.x) { const uint32_t v = sh_hist[t]; if (v) itx_red_u64(&D.grp[t], neg ? 0ull - (unsigned long long)v : (unsigned long long)v); }
    /* the last CTA out checks the chain of the whole window and hands the carry on */
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) sh_last = atomicAdd(P.first_bad + 1, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (sh_last) {
        __threadfence();
        uint32_t bad = 0;
        for (uint32_t i = 1 + threadIdx.x; i < A.nchunks; i += blockDim.x) {
            const unsigned long long en = __ldcg(A.entry + i), ex = itx_effective_exit(A.exit_, i - 1);
            bool ok = en == ex || ex == ITX_OFF_NONE;          /* NONE all the way down: a scan that starts mid-stream has met no record start yet */
            if (!ok && en == ITX_OFF_NONE) {                   /* the span found no record start: right if the chain runs over it, or has ended */
                const unsigned long long span_end = (A.k0 + i) * (unsigned long long)A.C + A.C;
                ok = ex == ITX_OFF_END || (ex < ITX_OFF_GUESS && ex >= (span_end < A.own ? span_end : A.own));
            }
            bad |= ok ? 0u : 1u;
        }
        bad = __syncthreads_or((int)bad) ? 1u : 0u;
        {   /* this launch's unknown-chromosome marks: kept if the launch stands, dropped with it otherwise (the replay marks for itself) */
            const bool stands = !neg && !bad && __ldcg(P.first_bad) == 0xffffffffu;
            const uint32_t nt = (uint32_t)(A.n_ref < ITX_MAX_TID_SEEN ? A.n_ref : ITX_MAX_TID_SEEN);
            for (uint32_t t = threadIdx.x; t < nt; t += blockDim.x)
                if (__ldcg(D.tid_unknown_seen + ITX_MAX_TID_SEEN + t)) { if (stands) D.tid_unknown_seen[t] = 1u; D.tid_unknown_seen[ITX_MAX_TID_SEEN + t] = 0u; }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            if (!neg) {
                if (bad) atomicMin(P.first_bad, P.window);
                unsigned long long x = itx_effective_exit(A.exit_, A.nchunks - 1);
                if (x == ITX_OFF_NONE && __ldcg(P.carry_log + P.window) == ITX_OFF_GUESS) x = ITX_OFF_GUESS;
                *A.carry = x;
                /* what this launch reported about the stream counts only if the launch stands (windows are launched in order, so
                 * first_bad is final for every window up to this one) */
                const uint32_t st = __ldcg(P.first_bad + 2);
                if (st && __ldcg(P.first_bad) == 0xffffffffu) atomicOr(&A.status[0], st);
            }
            if (!neg && P.window == 0 && __ldcg(P.carry_log) == ITX_OFF_GUESS) {
                /* a scan that started mid-stream: the record start it settled on (the caller checks it against the scan before) */
                unsigned long long fe = ITX_OFF_NONE;
                for (uint32_t i = 0; i < A.nchunks && fe == ITX_OFF_NONE; i++) fe = __ldcg(A.entry + i);
                *reinterpret_cast<unsigned long long *>(P.first_bad + 4) = fe;
            }
            A.work[2] = 0; P.first_bad[1] = 0; P.first_bad[2] = 0;
        }
    }
#undef one
#undef minus_one
#undef one64
#undef n_elem32
}

/* ------------------------------------------------------------------ XA:Z alternates (mapped2diffSubfam) */
/* k_xa: the reads k_scan queued -- they carry XA:Z and were about to be counted.  One lane per read re-derives its fragment and
 * the selected element (the same functions, out of global memory), then the warp walks the alternates of its 32 reads one LANE
 * per ALTERNATE: every owner counts the pieces of its own list, the pieces of the 32 reads are numbered across the warp and handed
 * out 32 at a time -- whichever read they belong to -- so that parsing, chromosome lookup and the table walk of all alternates
 * run side by side; the verdicts go back to the owners with two ballots (the first alternate that answers yes ends a read's
 * walk; malformed ones before it are counted).  Reads that stay are accumulated here, with the sign of the k_scan launch. */
struct itx_xa_args {
    itx_dev_index D; const itx_dev_index *Dg;                                  /* Dg: the same in global memory, for the out-of-line one-lane walk */
    const uint8_t *b; const itx_tidinfo *tid; int32_t n_ref; itx_dev_opts o;
    const unsigned long long *q; uint32_t *q_n; unsigned long long q_cap;      /* q_n: [0] entries, [1] CTAs done (the last one zeroes both) */
    int32_t sign; uint32_t flags;
    uint32_t hist_fc;                                                          /* 1: the CTA keeps the family / class counts in shared memory (behind the pools) */
};
#ifndef ITX_XA_OCC
#define ITX_XA_OCC 4                 /* 64 registers, 32 warps per SM: the kernel waits on scattered table and record reads (11.2 -> 9.3 ms per 30 M reads of cfg 3 against 24 warps at 80 registers; 48 registers spill and lose again) */
#endif
#ifndef ITX_XA_POOL
#define ITX_XA_POOL 6144u            /* bytes of shared memory per warp for the aux areas of its 32 reads (192 per read; what does not fit waits for the next pass) */
#endif
#define ITX_XA_SMEM (8u * ITX_XA_POOL + 64u)          /* + slack: itx_xa_piece_fast loads whole words up to 60 bytes past a piece's start */
__device__ __forceinline__ void itx_cp_async16_cg(void *smem_dst, const void *src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(itx_smem_addr(smem_dst)), "l"(src) : "memory"); }
/* The aux areas are parsed out of SHARED memory.  Round 2's first k_xa read them byte by byte with __ldg (1.4 G sector requests
 * and 2.9 G warp-instructions per 9 M reads, most of them waiting on L1): here the warp first brings the aux areas of its reads
 * over with 16-byte cp.async -- packed one behind the other in the warp's pool, as many reads per pass as fit -- and every parser
 * (tag walk, piece count, field split, strtol, chromosome name) then runs on itx_src_flat, without bounds tests and without a
 * global load.  An aux area larger than the pool takes the one-lane walk over global memory. */
__global__ void __launch_bounds__(256, ITX_XA_OCC) k_xa(const itx_xa_args A) {
    extern __shared__ __align__(16) uint8_t itx_xa_smem[];
    const itx_dev_index &D = A.D;
    __shared__ uint32_t sh_c[3];
    if (threadIdx.x < 3) sh_c[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    uint8_t *pool = itx_xa_smem + (threadIdx.x >> 5) * ITX_XA_POOL;
    /* the family and class counters are a few dozen addresses that every counted read would hit: per CTA in shared memory, flushed once
     * (reductions on one address queue up in L2); the subfamily counters -- a thousand and more addresses -- go straight to global memory */
    uint32_t *sh_fc = reinterpret_cast<uint32_t *>(itx_xa_smem + ITX_XA_SMEM);
    const uint32_t n_fc = A.hist_fc ? 2u * (uint32_t)(D.n_fam + D.n_cla) : 0u;
    for (uint32_t t = threadIdx.x; t < n_fc; t += blockDim.x) sh_fc[t] = 0u;
    __syncthreads();
    const unsigned long long n = __ldcg(A.q_n) < A.q_cap ? __ldcg(A.q_n) : A.q_cap;
    const bool neg = A.sign < 0, stat = A.o.filter == 0 && D.stat_mode, coop = A.flags & ITX_SCAN_XACOOP;
    const uint32_t one = neg ? 0xffffffffu : 1u, minus_one = neg ? 1u : 0xffffffffu;
    const unsigned long long one64 = neg ? ~0ull : 1ull;
    const itx_src_global G{A.b};
    uint32_t c_rep = 0, c_rep_u = 0, c_diff = 0;
    const unsigned long long w0 = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    for (unsigned long long i0 = w0 * 32ull; i0 < n; i0 += nw * 32ull) {
        const unsigned long long idx = i0 + lane;
        bool go = idx < n;
        itx_tuple T; T.start = T.end = T.rec_off = 0; T.info = 0;
        long long sel = -1; itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
        uint64_t a0 = 0, aend = 0; int32_t fold = 0;
        unsigned long long rp = ~0ull;
        if (go) { rp = __ldcs(A.q + idx); go = rp != ~0ull; }      /* all ones: an entry of a block that its warp did not fill */
        if (go) {
            uint32_t x[9]; G.core(rp, x);
            T = itx_decode_record<itx_src_global, false>(G, rp, x, 0u, A.tid, A.n_ref, A.o);
            int32_t nhit = 0; float tcov = 0.0f;
            itx_query Q;
            if (itx_query_open(D, (int32_t)(T.info & ITX_CHROM_MASK), T.start, T.end, &Q)) {
                sel = itx_select_walk(D, Q, itx_iv_global{D}, T.start, T.end, A.o.minCoverage, &nhit, &tcov, &e);
                if (sel == ITX_SEL_LONG) {                       /* out of line, on the copy of the index in global memory (no local copy of D) */
                    const itx_sel_cov r = itx_select_multi(*A.Dg, Q, T.start, T.end, nhit);
                    sel = r.sel; tcov = r.cov;
                    if (sel >= 0) e = itx_ld_iv(D, (uint32_t)sel);
                }
            }
            if (sel >= 0 && tcov < A.o.minCoverage) sel = -1;
            itx_aux_range(rp, x, &a0, &aend);
            go = sel >= 0 && a0 < aend;                            /* always true: k_scan queued the read because it is counted and carries XA */
            if (go) fold = (int32_t)__ldg(&D.ivf[sel].row);
        }
        const int32_t qlen = (int32_t)(T.end - T.start);
        /* the aux area, 16-byte granules around it (stream buffers are 16-byte aligned and carry 64 bytes of slack) */
        const uint64_t base = a0 & ~15ull;
        const uint32_t need = go ? (uint32_t)((aend - base + 15ull) & ~15ull) : 0u;
        /* inside the pool offsets are 32 bits wide and relative to `base` (the parsers do half the work per byte of a 64-bit walk) */
        const uint32_t a0r = (uint32_t)(a0 - base), aendr = go ? (uint32_t)(aend - base) : 0u;
        bool big = go && (!coop || aend - base > (uint64_t)(ITX_XA_POOL - 16u));
        bool pending = go && !big, diffsub = false;
        uint32_t n_bad = 0;
        while (__any_sync(0xffffffffu, pending)) {
            /* this pass: the pending reads whose aux areas fit the pool, in lane order */
            const uint32_t nd = pending ? need : 0u;
            uint32_t incl_b = nd;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl_b, d); if (lane >= (uint32_t)d) incl_b += t; }
            const bool in = pending && incl_b <= ITX_XA_POOL;
            const uint32_t off = incl_b - nd;
            __syncwarp();                                          /* the readers of the previous pass are done with the pool */
            /* every lane brings its own read's aux area (16 bytes per copy: the sectors are the same however the lanes share them out, and a
             * loop over the reads with the warp copying each one together cost a shuffle round per read) */
            if (in) for (uint32_t c = 0; c < nd; c += 16u) itx_cp_async16_cg(pool + off + c, A.b + base + c);
            itx_cp_async_wait_all();
            __syncwarp();
            /* every owner: XA and NM (bam_aux_get), the pieces of its list counted */
            uint32_t np = 0, sp0 = 0, sp1 = 0, packed = 0, zs = 0, ze = 0; int32_t nm = 0;
            if (in) {
                const itx_src_flat S{pool + off, 0ull};
                const uint32_t xa = itx_aux_find(S, a0r, aendr, 'X', 'A');
                const uint32_t nmo = xa == 0xffffffffu ? xa : itx_aux_find(S, a0r, aendr, 'N', 'M');
                if (xa == 0xffffffffu || nmo == 0xffffffffu) big = true;   /* a corrupt array count in the aux area: the 64-bit walk over global memory decides */
                else if (xa && xa < aendr) {
                    nm = itx_aux2i(S, nmo, aendr);
                    const uint8_t ty = S.u8(xa);
                    if (ty == 'Z' || ty == 'H') { uint32_t sp[2]; bool pk; zs = xa + 1u; np = itx_xa_count_pack(S, zs, aendr, &ze, sp, &pk); sp0 = sp[0]; sp1 = sp[1]; packed = pk ? 1u : 0u; }
                } else go = false;                                 /* (never: k_scan saw the tag) */
            }
            /* the pieces of the pass are numbered across the warp and handed out 32 at a time, one lane per alternate */
            uint32_t incl = np;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (uint32_t)d) incl += t; }
#ifdef ITX_XA_EXPERIMENT                                         /* timing experiments only (tools/build_variant.sh): 1 = no alternate is looked at */
            const uint32_t total = 0u, pbase = incl - np;
#else
            const uint32_t total = __shfl_sync(0xffffffffu, incl, 31), pbase = incl - np;
#endif
            bool found = false;
            for (uint32_t b0 = 0; b0 < total; b0 += 32u) {
                const uint32_t gi = b0 + lane;                     /* this lane's piece of the batch */
                /* its owner: the first lane whose running count exceeds gi (the counts never decrease along the warp) */
                uint32_t ow = 0;
#pragma unroll
                for (uint32_t st = 16; st; st >>= 1) { const uint32_t v = __shfl_sync(0xffffffffu, incl, (int)(ow + st - 1u)); if (v <= gi) ow += st; }
                ow &= 31u;
                const uint32_t o_base = __shfl_sync(0xffffffffu, pbase, (int)ow), o_off = __shfl_sync(0xffffffffu, off, (int)ow);
                const uint32_t o_zs = __shfl_sync(0xffffffffu, zs, (int)ow), o_ze = __shfl_sync(0xffffffffu, ze, (int)ow);
                const int32_t o_nm = __shfl_sync(0xffffffffu, nm, (int)ow), o_fold = __shfl_sync(0xffffffffu, fold, (int)ow), o_qlen = __shfl_sync(0xffffffffu, qlen, (int)ow);
                const uint32_t o_np = __shfl_sync(0xffffffffu, np, (int)ow), o_packed = __shfl_sync(0xffffffffu, packed, (int)ow);
                uint32_t o_sp[2]; o_sp[0] = __shfl_sync(0xffffffffu, sp0, (int)ow); o_sp[1] = __shfl_sync(0xffffffffu, sp1, (int)ow);
                bool hit = false, mal = false;
                if (gi < total) {
                    const itx_src_flat So{pool + o_off, 0ull};
                    uint32_t ps, pe;
                    const uint32_t k = gi - o_base;
                    if (o_packed && k < 8u) itx_xa_piece_bounds(o_zs, o_ze, o_np, o_sp, k, &ps, &pe);      /* the owner noted where its first ';' are */
                    else itx_xa_kth(So, o_zs, o_ze, k, &ps, &pe);
                    if (pe > ps) hit = itx_xa_piece_fast(D, So, ps, pe, o_nm, o_qlen, o_fold, &mal);
                }
                const uint32_t m_hit = __ballot_sync(0xffffffffu, hit), m_mal = __ballot_sync(0xffffffffu, mal);
                if (np && !found && pbase < b0 + 32u && incl > b0) {
                    const uint32_t lo_b = pbase > b0 ? pbase - b0 : 0u, hi_b = incl - b0 < 32u ? incl - b0 : 32u;
                    const uint32_t range = (hi_b >= 32u ? 0xffffffffu : (1u << hi_b) - 1u) & ~((1u << lo_b) - 1u);
                    const uint32_t h = m_hit & range;
                    if (h) { found = true; n_bad += (uint32_t)__popc(m_mal & range & ((1u << ((uint32_t)__ffs((int)h) - 1u)) - 1u)); }
                    else n_bad += (uint32_t)__popc(m_mal & range);
                }
            }
            if (in) { diffsub = found; pending = false; }
        }
        if (big && go) {                                           /* an aux area that does not fit the pool (or the A/B switch): one lane, global memory */
            const uint64_t xa = itx_aux_find(G, a0, aend, 'X', 'A');
            if (xa && xa < aend) {
                const int32_t nm = itx_aux2i(G, itx_aux_find(G, a0, aend, 'N', 'M'), aend);
                diffsub = itx_xa_walk(*A.Dg, G, xa, aend, nm, fold, qlen, &n_bad);
            } else go = false;
        }
        if (n_bad) atomicAdd(&D.status[2], neg ? 0u - n_bad : n_bad);
        const bool uniq = T.info & ITX_F_UNIQ, counted = go && !diffsub;
        const uint32_t m_cnt = __ballot_sync(0xffffffffu, counted);
        c_diff += (uint32_t)__popc(__ballot_sync(0xffffffffu, go && diffsub));
        c_rep += (uint32_t)__popc(m_cnt); c_rep_u += (uint32_t)__popc(m_cnt & __ballot_sync(0xffffffffu, uniq));
        if (counted) {
            if (stat) {
                const itx_meta m = D.meta[sel]; const itx_meta2 m2 = D.meta2[sel];
                const uint32_t hs = 2u * m.sub, hf = 2u * (uint32_t)(D.n_sub + m2.fam), hc = 2u * (uint32_t)(D.n_sub + D.n_fam + m2.cla);
                itx_red_u64(&D.grp[hs], one64);
                if (uniq) itx_red_u64(&D.grp[hs + 1], one64);
                if (n_fc) {
                    const uint32_t lf = 2u * (uint32_t)m2.fam, lc = 2u * (uint32_t)(D.n_fam + m2.cla);
                    atomicAdd(&sh_fc[lf], 1u); atomicAdd(&sh_fc[lc], 1u);
                    if (uniq) { atomicAdd(&sh_fc[lf + 1], 1u); atomicAdd(&sh_fc[lc + 1], 1u); }
                } else {
                    itx_red_u64(&D.grp[hf], one64); itx_red_u64(&D.grp[hc], one64);
                    if (uniq) { itx_red_u64(&D.grp[hf + 1], one64); itx_red_u64(&D.grp[hc + 1], one64); }
                }
                const uint4 sv = __ldg(reinterpret_cast<const uint4 *>(D.sinfo + m.sub));
                const uint32_t L = sv.x;
                uint32_t ja, jb;
                if (L && itx_cov_range(T.start, T.end - T.start, e.start, e.end, m.cons_start, m.cons_end, L, &ja, &jb)) {
                    const unsigned long long off = (unsigned long long)sv.z | ((unsigned long long)sv.w << 32);
                    itx_red_u32(&D.bp_diff[off + ja], one); itx_red_u32(&D.bp_diff[off + jb], minus_one);
                    if (uniq) { itx_red_u32(&D.bp_diff_u[off + ja], one); itx_red_u32(&D.bp_diff_u[off + jb], minus_one); }
                }
            } else if (A.o.filter) {
                itx_red_u32(&D.el_cnt[sel], one);
                if (uniq) itx_red_u32(&D.el_cnt_u[sel], one);
            }
        }
    }
    if (lane == 0) { if (c_rep) atomicAdd(&sh_c[0], c_rep); if (c_rep_u) atomicAdd(&sh_c[1], c_rep_u); if (c_diff) atomicAdd(&sh_c[2], c_diff); }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < n_fc; t += blockDim.x) { const uint32_t v = sh_fc[t]; if (v) itx_red_u64(&D.grp[2u * (uint32_t)D.n_sub + t], neg ? 0ull - (unsigned long long)v : (unsigned long long)v); }
    if (threadIdx.x == 0) {
        if (sh_c[0]) itx_red_u64(&D.cnt[9], neg ? 0ull - sh_c[0] : (unsigned long long)sh_c[0]);
        if (sh_c[1]) itx_red_u64(&D.cnt[10], neg ? 0ull - sh_c[1] : (unsigned long long)sh_c[1]);
        if (sh_c[2]) itx_red_u64(&D.cnt[12], neg ? 0ull - sh_c[2] : (unsigned long long)sh_c[2]);
        __threadfence();
        if (atomicAdd(A.q_n + 1, 1u) == gridDim.x - 1) { A.q_n[0] = 0; A.q_n[1] = 0; }      /* every CTA has read the count: the queue is empty again */
    }
}

/* prefix sums of the coverage difference arrays: one warp per subfamily */
__global__ void k_finalize(const itx_dev_index D, uint32_t *bp, uint32_t *bp_u) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t s = w; s < (uint32_t)D.n_sub; s += nw) {
        const uint32_t L = D.sub_len[s];
        if (!L) continue;
        const unsigned long long off = D.sub_bp_off[s];
        uint32_t carry = 0, carry_u = 0;
        for (uint32_t j0 = 0; j0 <= L; j0 += 32) {
            const uint32_t j = j0 + lane;
            uint32_t v = j <= L ? D.bp_diff[off + j] : 0u, u = j <= L ? D.bp_diff_u[off + j] : 0u;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t tv = __shfl_up_sync(0xffffffffu, v, d), tu = __shfl_up_sync(0xffffffffu, u, d);
                if (lane >= (uint32_t)d) { v += tv; u += tu; }
            }
            v += carry; u += carry_u;
            if (j <= L) { bp[off + j] = v; bp_u[off + j] = u; }
            carry = __shfl_sync(0xffffffffu, v, 31); carry_u = __shfl_sync(0xffffffffu, u, 31);
        }
    }
}

/* exclusive scan of nrec over one window (trace only): one block */
__global__ void k_rec_base(const uint32_t *nrec, uint32_t n, unsigned long long *rec_base, unsigned long long *running) {
    __shared__ unsigned long long part[1024];
    const uint32_t t = threadIdx.x, per = (n + blockDim.x - 1) / blockDim.x;
    const uint32_t a = t * per < n ? t * per : n, b = a + per < n ? a + per : n;
    unsigned long long s = 0;
    for (uint32_t i = a; i < b; i++) s += nrec[i];
    part[t] = s;
    __syncthreads();
    if (t == 0) { unsigned long long acc = *running; for (uint32_t k = 0; k < blockDim.x; k++) { const unsigned long long v = part[k]; part[k] = acc; acc += v; } *running = acc; }
    __syncthreads();
    s = part[t];
    for (uint32_t i = a; i < b; i++) { rec_base[i] = s; s += nrec[i]; }
}

__global__ void k_query(const itx_dev_index D, int32_t chrom, const uint32_t *start, const uint32_t *end, long long n, float min_cov,
                        int32_t *sel_row, int32_t *n_hits) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t nh; float tcov; itx_iv e; e.row = 0;
    long long sel = itx_find_select(D, chrom, start[i], end[i], min_cov, &nh, &tcov, &e);
    if (sel >= 0 && tcov < min_cov) sel = -1;
    sel_row[i] = sel >= 0 ? (int32_t)e.row : -1;
    if (n_hits) n_hits[i] = nh;
}

/* ------------------------------------------------------------------ CpG rows */
struct itx_cpg_args {
    itx_dev_index D;
    const int32_t *chrom; const uint32_t *start, *end; const double *score; long long n; int32_t filter;
    unsigned long long *in_repeat;
};
__global__ void __launch_bounds__(256) k_cpg(const itx_cpg_args A) {
    const itx_dev_index &D = A.D;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long sel = -1; double sc = 0.0; uint32_t st = 0; itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
    if (i < A.n) {
        const int32_t c = A.chrom[i];
        if (c >= 0) { st = A.start[i]; sel = itx_find_head(D, c, st, A.end[i], &e); sc = A.score[i]; }
    }
    const uint32_t m = __popc(__ballot_sync(0xffffffffu, sel >= 0));
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(A.in_repeat, (unsigned long long)m);
    if (sel < 0) return;
    if (A.filter) { atomicAdd(&D.el_cpg[sel], 1u); atomicAdd(&D.el_cpg_score[sel], sc); return; }
    if (!D.stat_mode) return;
    const itx_meta mt = D.meta[sel]; const itx_meta2 m2 = D.meta2[sel];
    const uint32_t gs = mt.sub, gf = (uint32_t)(D.n_sub + m2.fam), gc = (uint32_t)(D.n_sub + D.n_fam + m2.cla);
    atomicAdd(&D.grp_cpg[gs], 1u); atomicAdd(&D.grp_cpg_score[gs], sc);
    atomicAdd(&D.grp_cpg[gf], 1u); atomicAdd(&D.grp_cpg_score[gf], sc);
    atomicAdd(&D.grp_cpg[gc], 1u); atomicAdd(&D.grp_cpg_score[gc], sc);
    const uint32_t L = D.sub_len[mt.sub];
    uint32_t ja, jb;
    if (L && itx_cov_range(st, 2u, e.start, e.end, mt.cons_start, mt.cons_end, L, &ja, &jb)) {
        const unsigned long long off = D.sub_bp_off[mt.sub];
        for (uint32_t j = ja; j < jb; j++) atomicAdd(&D.bp_cpg[off + j], sc);
    }
}

/* ------------------------------------------------------------------ CpG bedGraph text on the device */
/* k_bedgraph: the text of a bedGraph file, whole lines, in device memory.  A thread per byte: the thread whose byte
 * starts a line parses it (v2: a CTA per 4 KiB tile lists its line starts first, then a thread per line) -- skip blank and '#' lines, chop on white space, chromosome by name, strtol start / end,
 * strtod score (lineFileNextReal + chopByWhite + generic.c:1069-1076) -- and counts it exactly as k_cpg does.  Lines
 * with fewer than four fields (the reference aborts at the first one) and scores outside the exact fast path of
 * itx_strtod_fast are reported by file offset for the host. */
#define ITX_BG_SH 512u                     /* families + classes gathered per CTA in shared memory */
struct itx_bedgraph_args {
    itx_dev_index D;
    const uint8_t *text; unsigned long long n;
    int32_t filter;
    unsigned long long *counts;          /* [0] lines, [1] CpG sites in repeats, [2] smallest offset of a malformed line, [3] lines left to the host */
    uint32_t *fallback; unsigned long long fallback_cap;      /* offsets (in this text) of the lines whose score the host must parse */
};
#define ITX_BG_TILE 4096u                  /* text bytes per CTA */
__global__ void __launch_bounds__(256) k_bedgraph(const itx_bedgraph_args A) {
    /* family and class sums are a few dozen addresses hit by every row: they are gathered per CTA in shared memory first */
    __shared__ double sh_sc[ITX_BG_SH]; __shared__ uint32_t sh_cn[ITX_BG_SH];
    __shared__ uint16_t sh_start[ITX_BG_TILE + 1]; __shared__ uint32_t sh_n, sh_lines, sh_inrep;
    const itx_dev_index &D = A.D;
    const uint32_t n_fc = (uint32_t)(D.n_fam + D.n_cla);
    const bool sh_ok = !A.filter && D.stat_mode && n_fc <= ITX_BG_SH;
    if (sh_ok) for (uint32_t t = threadIdx.x; t < n_fc; t += blockDim.x) { sh_sc[t] = 0.0; sh_cn[t] = 0; }
    if (threadIdx.x == 0) { sh_n = 0; sh_lines = 0; sh_inrep = 0; }
    __syncthreads();
    /* pass 1: the tile's line feeds, 16 bytes per thread; the line after each of them is this CTA's (it may run into the
     * next tile: the parse reads global memory), and the first CTA also owns the line at offset 0 */
    const unsigned long long base = (unsigned long long)blockIdx.x * ITX_BG_TILE;
    {
        const unsigned long long q0 = base + threadIdx.x * 16ull;
        if (q0 < A.n) {
            uint32_t w[4] = {0, 0, 0, 0};
            if (q0 + 16 <= A.n) { const uint4 v = __ldg(reinterpret_cast<const uint4 *>(A.text + q0)); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
            else for (uint32_t j = 0; q0 + j < A.n; j++) w[j >> 2] |= (uint32_t)A.text[q0 + j] << (8 * (j & 3));
#pragma unroll
            for (uint32_t j = 0; j < 16; j++)
                if (((w[j >> 2] >> (8 * (j & 3))) & 0xffu) == '\n' && q0 + j + 1 < A.n) sh_start[atomicAdd(&sh_n, 1u)] = (uint16_t)(threadIdx.x * 16u + j + 1u);
        }
        if (blockIdx.x == 0 && threadIdx.x == 0 && A.n) sh_start[atomicAdd(&sh_n, 1u)] = 0;
    }
    __syncthreads();
    const itx_src_global G{A.text};
    /* pass 2: a thread per line */
    for (uint32_t k = threadIdx.x; k < sh_n; k += blockDim.x) {
        const unsigned long long p = base + sh_start[k];
        unsigned long long q = p, le = p;
        while (le < A.n && A.text[le] != '\n') le++;
        while (q < le && itx_is_space(A.text[q])) q++;
        if (q >= le || A.text[q] == '#') continue;
        /* up to four words; a fifth and later ones do not matter */
        unsigned long long ws[4], we[4]; int nw = 0;
        while (nw < 4 && q < le) {
            ws[nw] = q; while (q < le && !itx_is_space(A.text[q])) q++;
            we[nw] = q; nw++;
            while (q < le && itx_is_space(A.text[q])) q++;
        }
        if (nw < 4) { atomicMin(A.counts + 2, p); continue; }
        bool exact;
        const double sc = itx_strtod_fast(G, ws[3], we[3], &exact);
        if (!exact) {
            const unsigned long long f = atomicAdd(A.counts + 3, 1ull);
            if (f < A.fallback_cap) A.fallback[f] = (uint32_t)p;
            continue;
        }
        atomicAdd(&sh_lines, 1u);
        const uint32_t st = (uint32_t)itx_strtol_int(G, ws[1], we[1]), en = (uint32_t)itx_strtol_int(G, ws[2], we[2]);
        const int32_t c = itx_chrom_by_name(D, G, ws[0], we[0]);
        itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
        const long long sel = c >= 0 ? itx_find_head(D, c, st, en, &e) : -1;
        if (sel < 0) continue;
        atomicAdd(&sh_inrep, 1u);
        if (A.filter) { atomicAdd(&D.el_cpg[sel], 1u); atomicAdd(&D.el_cpg_score[sel], sc); continue; }
        if (!D.stat_mode) continue;
        const itx_meta mt = D.meta[sel]; const itx_meta2 m2 = D.meta2[sel];
        const uint32_t gs = mt.sub, gf = (uint32_t)(D.n_sub + m2.fam), gc = (uint32_t)(D.n_sub + D.n_fam + m2.cla);
        atomicAdd(&D.grp_cpg[gs], 1u); atomicAdd(&D.grp_cpg_score[gs], sc);
        if (sh_ok) {
            atomicAdd(&sh_cn[m2.fam], 1u); atomicAdd(&sh_sc[m2.fam], sc);
            atomicAdd(&sh_cn[D.n_fam + m2.cla], 1u); atomicAdd(&sh_sc[D.n_fam + m2.cla], sc);
        } else {
            atomicAdd(&D.grp_cpg[gf], 1u); atomicAdd(&D.grp_cpg_score[gf], sc);
            atomicAdd(&D.grp_cpg[gc], 1u); atomicAdd(&D.grp_cpg_score[gc], sc);
        }
        const uint32_t L = D.sub_len[mt.sub];
        uint32_t ja, jb;
        if (L && itx_cov_range(st, 2u, e.start, e.end, mt.cons_start, mt.cons_end, L, &ja, &jb)) {
            const unsigned long long off = D.sub_bp_off[mt.sub];
            for (uint32_t j = ja; j < jb; j++) atomicAdd(&D.bp_cpg[off + j], sc);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) { if (sh_lines) atomicAdd(A.counts, (unsigned long long)sh_lines); if (sh_inrep) atomicAdd(A.counts + 1, (unsigned long long)sh_inrep); }
    if (sh_ok) for (uint32_t t = threadIdx.x; t < n_fc; t += blockDim.x) if (sh_cn[t]) { atomicAdd(&D.grp_cpg[D.n_sub + t], sh_cn[t]); atomicAdd(&D.grp_cpg_score[D.n_sub + t], sh_sc[t]); }
}

/* ------------------------------------------------------------------ BGZF inflate on the device */
/* One thread per BGZF block, one warp per CTA, 2^LG of the warp's lanes decoding 2^LG blocks in lock step (the others idle).
 * A thread's look-up tables (ITX_LUT_CELLS 16-bit cells) live in shared memory as 32-bit words interleaved across the
 * active lanes -- word w of lane l at index w * 2^LG + l -- so every lane owns a bank whatever cell it reads; 20 KiB per
 * warp of 32 blocks.  The symbol arrays of the long codes live in global memory, interleaved by 32 (cell j of lane l at
 * tabs[warp][j * 32 + l]).  A warp takes the groups of 2^LG blocks blockIdx.x, blockIdx.x + gridDim.x, ...
 * Fewer blocks per warp = fewer ways for a round to diverge = a shorter round: 32 blocks per warp is the densest packing,
 * 8 the lowest latency per block (what the last groups of a file want: nothing hides their latency). */
template <uint32_t LG>
struct itx_tab_dev {
    uint16_t *g, *s;
    __device__ __forceinline__ uint16_t operator()(uint32_t j) const { return g[j * 32u]; }
    __device__ __forceinline__ void set(uint32_t j, uint16_t v) const { g[j * 32u] = v; }
    __device__ __forceinline__ uint16_t lut(uint32_t j) const { return s[((j >> 1) << (LG + 1u)) | (j & 1u)]; }
    __device__ __forceinline__ void lut_set(uint32_t j, uint16_t v) const { s[((j >> 1) << (LG + 1u)) | (j & 1u)] = v; }
};
struct itx_inflate_args {
    const uint8_t *file;                 /* the compressed bytes on the device (a ring: coff is an offset into it, not into the file) */
    const itx_bgzf_block *blk;           /* coff, csize, isize, uoff per block */
    unsigned long long b0, nblk;         /* blocks [b0, b0 + nblk) */
    uint8_t *out;                        /* uncompressed stream: block b goes to out + blk[b].uoff */
    uint32_t *status;                    /* [5] number of blocks that failed, [6] index of one of them */
    uint16_t *tabs;                      /* 32 * ITX_T_CELLS cells per warp of the grid */
    /* deferred matches: block g0 of the launch owns m_pl[g0 * m_cap ..] / m_d[g0 * m_cap ..]; m_n[g0] = entries or ITX_M_NONE */
    uint32_t *m_pl; uint16_t *m_d; uint32_t *m_n; uint32_t m_cap;
    uint32_t fuse_lz;                    /* the decoding warp resolves the matches of its own blocks (itx_lzw_resolve): no second kernel */
};
#define ITX_INF_THREADS 32
#define ITX_INF_SMEM(LG) (ITX_LUT_CELLS * 2u * (1u << (LG)))
/* First pass over every block of the launch: Huffman decoding, literals stored, matches listed (m_cap != 0) or
 * copied in line (m_cap == 0).  The host sizes the lists for the worst case (ITX_M_WORST entries: a match is at
 * least three bytes long), so a list cannot overflow. */
#define ITX_M_WORST 21848u
/* The second pass of one block by the 32 lanes of the warp that decoded it: windows of W bytes; W 16-bit src cells and the window's
 * bytes in the warp's shared memory (its look-up tables, dead once the batch is decoded).  The list is in output order and its matches
 * do not overlap, so the entries of a window are a run of the list; an entry cut by a window's end is visited by both windows.
 * A window comes in with 16-byte loads (ld.cg: the bytes were stored by other lanes of this warp, L2 is where stores land), bytes whose
 * source lies before the window are gathered from L2 eight loads at a time per lane, the others out of shared memory, and the window
 * goes back with 16-byte stores. */
template <uint32_t W>
__device__ __forceinline__ void itx_lzw_resolve(uint8_t *out, uint32_t isize, const uint32_t *pl, const uint16_t *md, uint32_t n, uint16_t *src, uint8_t *data, uint32_t lane) {
    uint32_t k0 = 0;
    for (uint32_t w0 = 0; w0 < isize && k0 < n; w0 += W) {
        const uint32_t w1 = w0 + W < isize ? w0 + W : isize, cnt = w1 - w0;
        if ((__ldcg(pl + k0) & 0xffffu) >= w1) continue;                    /* nothing but literals in this window */
        const uint32_t skew = (uint32_t)(reinterpret_cast<uintptr_t>(out + w0) & 15u);
        uint8_t *a0 = out + w0 - skew;                                       /* 16-byte aligned; the stream buffer has slack on both sides */
        const uint32_t span = (skew + cnt + 15u) & ~15u;
        for (uint32_t i = lane * 16u; i < span; i += 512u) *reinterpret_cast<uint4 *>(data + i) = __ldcg(reinterpret_cast<const uint4 *>(a0 + i));
        itx_lzw_init(src, w0, cnt, lane);
        __syncwarp();
        for (uint32_t k = k0;; k += 32u) {
            const bool in = k + lane < n;
            const uint32_t e = in ? __ldcg(pl + k + lane) : 0xffffu;
            const uint32_t pos = e & 0xffffu, len = e >> 16;
            if (in && pos < w1) itx_lzw_scatter(src, w0, w1, pos, len, (uint32_t)__ldcg(md + k + lane));
            const uint32_t c = (uint32_t)__popc(__ballot_sync(0xffffffffu, in && pos + len <= w1));       /* finished for good: a prefix of the batch */
            k0 = k + c;
            if (c < 32u) break;
        }
        __syncwarp();
        while (__any_sync(0xffffffffu, itx_lzw_jump(src, w0, cnt, lane))) { }
        uint8_t *dw = data + skew;
        const uint32_t cnt_r = (cnt + 255u) & ~255u;                        /* cells past the window's end are their own sources (itx_lzw_init) */
        for (uint32_t i0 = lane; i0 < cnt_r; i0 += 256u) {
            uint32_t sv[8]; uint8_t b[8];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) sv[u] = (uint32_t)src[i0 + 32u * u];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) b[u] = sv[u] < w0 ? __ldcg(out + sv[u]) : dw[sv[u] - w0];       /* a literal reads itself; a literal of the window is never changed here */
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) dw[i0 + 32u * u] = b[u];
        }
        __syncwarp();
        for (uint32_t i = lane * 16u; i < span; i += 512u) {
            if (i >= skew && i + 16u <= skew + cnt) *reinterpret_cast<uint4 *>(a0 + i) = *reinterpret_cast<const uint4 *>(data + i);
            else for (uint32_t j = 0; j < 16u; j++) if (i + j >= skew && i + j < skew + cnt) a0[i + j] = data[i + j];
        }
        __syncwarp();
    }
}
#ifndef ITX_LZW_W5
#define ITX_LZW_W5 6144u
#define ITX_LZW_W4 3072u
#define ITX_LZW_W3 1536u
#endif
#ifndef ITX_INF_OCC4
#define ITX_INF_OCC4 18             /* 96 registers: 18 warps of 16 blocks per SM measured 4 % faster end to end than 16 warps at 112 */
#endif
#ifndef ITX_INF_OCC5
#define ITX_INF_OCC5 10
#endif
template <uint32_t LG>
__global__ void __launch_bounds__(ITX_INF_THREADS, LG == 5 ? ITX_INF_OCC5 : ITX_INF_OCC4) k_inflate(const itx_inflate_args A) {
    extern __shared__ __align__(16) uint8_t itx_inf_smem[];
    constexpr uint32_t NL = 1u << LG;
    const uint32_t lane = threadIdx.x;
    itx_inflater<itx_tab_dev<LG> > I;
    I.tab.g = A.tabs + (size_t)blockIdx.x * (32u * ITX_T_CELLS) + lane;
    I.tab.s = reinterpret_cast<uint16_t *>(itx_inf_smem) + (lane & (NL - 1u)) * 2u;
    for (unsigned long long g0 = (unsigned long long)blockIdx.x * NL; g0 < A.nblk; g0 += (unsigned long long)gridDim.x * NL) {
        const unsigned long long g = g0 + lane, b = A.b0 + g;
        const bool mine = lane < NL && g < A.nblk;
        I.state = ITX_ST_DONE; I.err = ITX_INF_OK; I.m_cap = 0; I.n_match = 0;
        if (mine) {
            const itx_bgzf_block B = A.blk[b];
            I.out = A.out + B.uoff; I.out_cap = B.isize;
            if (A.m_cap) { I.m_cap = A.m_cap; I.m_pl = A.m_pl + g * A.m_cap; I.m_d = A.m_d + g * A.m_cap; }
            I.begin(A.file + B.coff + 18, B.csize - 18 - 8, B.isize);          /* header 18, footer CRC32 + ISIZE */
        }
        /* the warp's blocks step together, one round (a few symbols, or a header with its table build) per lane per
         * iteration.  A table build is thousands of instructions: a lane that reaches a header waits there until most
         * of the others have reached theirs, so that the builds run side by side instead of one after the other
         * (blocks written by the same compressor change tables after about the same number of symbols). */
        for (;;) {
            const bool run = I.running(), hdr = run && I.state == ITX_ST_HEADER;
            const uint32_t m_run = __ballot_sync(0xffffffffu, run), m_hdr = __ballot_sync(0xffffffffu, hdr);
            if (!m_run) break;
            const bool hdr_go = m_hdr == m_run || (uint32_t)__popc(m_hdr) >= (3u * NL) / 4u;
            if (run && (!hdr || hdr_go)) I.advance();
        }
        if (mine) {
            if (A.m_cap) A.m_n[g] = I.state == ITX_ST_DONE ? I.n_match : ITX_M_NONE;
            if (I.state != ITX_ST_DONE) { atomicAdd(&A.status[5], 1u); A.status[6] = (uint32_t)b; }
        }
        __syncwarp();
        if (A.fuse_lz && A.m_cap) {
            /* the warp's blocks one after the other, all 32 lanes on each */
            constexpr uint32_t W = LG == 5 ? ITX_LZW_W5 : (LG == 4 ? ITX_LZW_W4 : ITX_LZW_W3);      /* 2 W bytes of cells + W + 32 bytes of data in the warp's 640 << LG */
            const uint32_t nm = mine && I.state == ITX_ST_DONE ? I.n_match : 0u;
            const unsigned long long op = reinterpret_cast<unsigned long long>(I.out);
            for (uint32_t l = 0; l < NL; l++) {
                const uint32_t n_l = __shfl_sync(0xffffffffu, nm, (int)l);
                if (!n_l) continue;
                const uint32_t isz = __shfl_sync(0xffffffffu, I.out_pos, (int)l);
                uint8_t *o_l = reinterpret_cast<uint8_t *>(__shfl_sync(0xffffffffu, op, (int)l));
                itx_lzw_resolve<W>(o_l, isz, A.m_pl + (g0 + l) * A.m_cap, A.m_d + (g0 + l) * A.m_cap, n_l, reinterpret_cast<uint16_t *>(itx_inf_smem), itx_inf_smem + 2u * W, lane);
            }
        }
    }
}

/* Second pass: a CTA per block.  The block (literals in place, holes where matches go) is read into shared memory
 * with 16-byte loads, warp 0 copies the listed matches there -- 32 list entries at a time, a few cycles per byte of
 * history instead of a trip to L2 or DRAM -- and the finished block goes back with 16-byte stores.  Meanwhile the
 * other warps pull the next block's list and bytes into L2. */
#define ITX_LZ_THREADS 128
#define ITX_LZ_SMEM (65536u + 32u)
#define ITX_LZ_NB 4                        /* list batches (of 32 entries) kept in registers ahead of the copy loop */
__device__ __forceinline__ void itx_prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__global__ void __launch_bounds__(ITX_LZ_THREADS) k_lz_resolve(const itx_inflate_args A) {
    extern __shared__ __align__(16) uint8_t itx_lz_buf[];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (unsigned long long g = blockIdx.x; g < A.nblk; g += gridDim.x) {
        const uint32_t n = A.m_n[g];
        if (n == ITX_M_NONE || n == 0) continue;                       /* failed (reported by k_inflate) or nothing to copy */
        const itx_bgzf_block B = A.blk[A.b0 + g];
        uint8_t *base = A.out + B.uoff;
        const uint32_t skew = (uint32_t)(reinterpret_cast<uintptr_t>(base) & 15u);
        const uint8_t *a0 = base - skew;                               /* 16-byte aligned; never before the stream buffer */
        const uint32_t span = (skew + B.isize + 15u) & ~15u;           /* <= 65536 + 16; the stream buffer carries slack past its end */
        const uint32_t *pl = A.m_pl + g * A.m_cap; const uint16_t *md = A.m_d + g * A.m_cap;
        for (uint32_t i = tid * 16u; i < span; i += ITX_LZ_THREADS * 16u) *reinterpret_cast<uint4 *>(itx_lz_buf + i) = __ldcs(reinterpret_cast<const uint4 *>(a0 + i));
        __syncthreads();
        if (warp == 0) {
            uint8_t *sm = itx_lz_buf + skew;
            uint32_t e_nx[ITX_LZ_NB], d_nx[ITX_LZ_NB];
#pragma unroll
            for (uint32_t b = 0; b < ITX_LZ_NB; b++) { const uint32_t k = 32u * b + lane; e_nx[b] = k < n ? __ldcs(pl + k) : 0u; d_nx[b] = k < n ? (uint32_t)__ldcs(md + k) : 0u; }
            for (uint32_t c0 = 0; c0 < n; c0 += 32u * ITX_LZ_NB) {
                uint32_t e_cu[ITX_LZ_NB], d_cu[ITX_LZ_NB];
#pragma unroll
                for (uint32_t b = 0; b < ITX_LZ_NB; b++) {
                    e_cu[b] = e_nx[b]; d_cu[b] = d_nx[b];
                    const uint32_t k = c0 + 32u * (ITX_LZ_NB + b) + lane;                      /* the next chunk's entries are on their way */
                    if (k < n) { e_nx[b] = __ldcs(pl + k); d_nx[b] = (uint32_t)__ldcs(md + k); }
                }
#pragma unroll
                for (uint32_t b = 0; b < ITX_LZ_NB; b++) {
                    const uint32_t k0 = c0 + 32u * b;
                    if (k0 < n) {
                        const uint32_t pos = e_cu[b] & 0xffffu, len = e_cu[b] >> 16, dist = d_cu[b];
                        uint32_t undone = __ballot_sync(0xffffffffu, k0 + lane < n);
                        while (undone) {
                            const uint32_t m = (uint32_t)__ffs((int)undone) - 1u;
                            const uint32_t pm = __shfl_sync(0xffffffffu, pos, (int)m);
                            const bool go = ((undone >> lane) & 1u) && itx_lz_ready(pos, len, dist, lane == m, pm);
                            if (go) itx_lz_copy<false>(sm + pos, len, dist);
                            __syncwarp();
                            undone &= ~__ballot_sync(0xffffffffu, go);
                        }
                    }
                }
            }
        } else {
            /* the next block of this CTA: its list and its bytes towards L2 */
            const unsigned long long g2 = g + gridDim.x;
            if (g2 < A.nblk) {
                const uint32_t n2 = A.m_n[g2];
                if (n2 != ITX_M_NONE && n2 != 0) {
                    const uint8_t *q0 = reinterpret_cast<const uint8_t *>(A.m_pl + g2 * A.m_cap), *q1 = reinterpret_cast<const uint8_t *>(A.m_d + g2 * A.m_cap);
                    const itx_bgzf_block B2 = A.blk[A.b0 + g2];
                    const uint8_t *q2 = A.out + B2.uoff;
                    const uint32_t t = tid - 32u, nt = ITX_LZ_THREADS - 32u;
                    for (uint32_t i = t * 128u; i < n2 * 4u; i += nt * 128u) itx_prefetch_l2(q0 + i);
                    for (uint32_t i = t * 128u; i < n2 * 2u; i += nt * 128u) itx_prefetch_l2(q1 + i);
                    for (uint32_t i = t * 128u; i < B2.isize; i += nt * 128u) itx_prefetch_l2(q2 + i);
                }
            }
        }
        __syncthreads();
        const uint32_t lo = skew, hi = skew + B.isize;
        for (uint32_t i = tid * 16u; i < span; i += ITX_LZ_THREADS * 16u) {
            if (i >= lo && i + 16u <= hi) *reinterpret_cast<uint4 *>(const_cast<uint8_t *>(a0) + i) = *reinterpret_cast<const uint4 *>(itx_lz_buf + i);
            else for (uint32_t j = 0; j < 16u; j++) if (i + j >= lo && i + j < hi) const_cast<uint8_t *>(a0)[i + j] = itx_lz_buf[i + j];
        }
        __syncthreads();
    }
}

/* Second pass, data-parallel: a CTA per block, EVERY thread busy.  A byte of the block is either a literal (already in place) or
 * belongs to a listed match, i.e. it is a copy of the byte `dist` before it -- which may itself be a copy.  src[i] = where byte i comes
 * from (itself for a literal); following src to its fixed point names the literal every byte finally equals, and the chains are
 * shortened by pointer jumping (src[i] = src[src[i]], all bytes at once), so the number of passes is the LOGARITHM of the longest
 * chain -- a handful for BAM blocks, 16 at worst (a run of one byte repeated through the whole block).  No ordering between matches
 * is ever needed, so nothing waits: the block is in and out of shared memory in tens of microseconds.
 * Shared memory: the block (64 KiB + alignment slack) and src as 16-bit indices (128 KiB): one CTA per SM. */
#define ITX_LZ2_THREADS 512
#define ITX_LZ2_SMEM (65536u + 32u + 131072u)
__global__ void __launch_bounds__(ITX_LZ2_THREADS, 1) k_lz_jump(const itx_inflate_args A) {
    extern __shared__ __align__(16) uint8_t itx_lz_buf[];
    uint8_t *data = itx_lz_buf;
    uint16_t *src = reinterpret_cast<uint16_t *>(itx_lz_buf + 65536u + 32u);
    const uint32_t tid = threadIdx.x;
    for (unsigned long long g = blockIdx.x; g < A.nblk; g += gridDim.x) {
        const uint32_t n = A.m_n[g];
        if (n == ITX_M_NONE || n == 0) continue;                       /* failed (reported by k_inflate) or nothing to copy */
        const itx_bgzf_block B = A.blk[A.b0 + g];
        uint8_t *base = A.out + B.uoff;
        const uint32_t skew = (uint32_t)(reinterpret_cast<uintptr_t>(base) & 15u);
        const uint8_t *a0 = base - skew;                               /* 16-byte aligned; never before the stream buffer */
        const uint32_t span = (skew + B.isize + 15u) & ~15u;           /* <= 65536 + 16; the stream buffer carries slack past its end */
        const uint32_t isize = B.isize;
        const uint32_t *pl = A.m_pl + g * A.m_cap; const uint16_t *md = A.m_d + g * A.m_cap;
        for (uint32_t i = tid * 16u; i < span; i += ITX_LZ2_THREADS * 16u) *reinterpret_cast<uint4 *>(data + i) = __ldcs(reinterpret_cast<const uint4 *>(a0 + i));
        for (uint32_t i = tid * 2u; i < isize; i += ITX_LZ2_THREADS * 2u) *reinterpret_cast<uint32_t *>(src + i) = i | ((i + 1u) << 16);      /* every byte its own source */
        __syncthreads();
        /* the listed matches: byte pos + j comes from pos + j - dist (a match that overlaps itself chains through its own bytes) */
        for (uint32_t k = tid; k < n; k += ITX_LZ2_THREADS) {
            const uint32_t e = __ldcs(pl + k), d = (uint32_t)__ldcs(md + k);
            const uint32_t pos = e & 0xffffu, len = e >> 16;
            for (uint32_t j = 0; j < len; j++) src[pos + j] = (uint16_t)(pos + j - d);
        }
        __syncthreads();
        /* pointer jumping until every byte points at a literal */
        for (;;) {
            bool changed = false;
            for (uint32_t i = tid; i < isize; i += ITX_LZ2_THREADS) {
                const uint32_t s = src[i];
                if (s != i) { const uint32_t ss = src[s]; if (ss != s) { src[i] = (uint16_t)ss; changed = true; } }
            }
            if (!__syncthreads_or(changed ? 1 : 0)) break;
        }
        uint8_t *sm = data + skew;
        for (uint32_t i = tid; i < isize; i += ITX_LZ2_THREADS) { const uint32_t s = src[i]; if (s != i) sm[i] = sm[s]; }      /* a literal is never written here */
        __syncthreads();
        const uint32_t lo = skew, hi = skew + isize;
        for (uint32_t i = tid * 16u; i < span; i += ITX_LZ2_THREADS * 16u) {
            if (i >= lo && i + 16u <= hi) *reinterpret_cast<uint4 *>(const_cast<uint8_t *>(a0) + i) = *reinterpret_cast<const uint4 *>(data + i);
            else for (uint32_t j = 0; j < 16u; j++) if (i + j >= lo && i + j < hi) const_cast<uint8_t *>(a0)[i + j] = data[i + j];
        }
        __syncthreads();
    }
}

__global__ void k_fill_u32(uint32_t *p, unsigned long long n, uint32_t v) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) p[i] = v;
}
#endif
