/* itx_emu.cpp -- TEST-ONLY host emulation of the device logic (never part of libiteres_gpu.so).
 *
 * iteres_b200/csrc/itx_logic.cuh is written as __host__ __device__ code; this file compiles it with
 * g++ and drives it the way the kernels in itx_kernels.cuh do -- chunked speculative record-boundary
 * discovery, chain verification / repair, then one "lane" per tuple -- but sequentially.  It lets
 * the `-m "not gpu"` suite check the per-record logic against the oracle on a box without a GPU.
 * The product has no CPU path: nothing under iteres_b200/ links or loads this file.
 */
#include <stdint.h>
static uint64_t g_xa_fast[2];                              /* pieces of XA lists that took itx_xa_piece_fast's register path / the general one */
#define ITX_XA_FAST_NOTE(i) (g_xa_fast[i]++)
static int64_t g_xa_walk[5];                               /* the last question an alternate's parser asked the table: chromosome, start, end, fold; [4] how many so far */
#define ITX_XA_WALK_NOTE(c, s, e, fold) (g_xa_walk[0] = (c), g_xa_walk[1] = (s), g_xa_walk[2] = (e), g_xa_walk[3] = (fold), g_xa_walk[4]++)
#include "../../iteres_b200/csrc/itx_logic.cuh"
#include "../../iteres_b200/csrc/itx_inflate.cuh"
#include "../../iteres_b200/csrc/itx_ordered.h"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <vector>
#include <string>
#include <cmath>

struct emu_index {
    itx_index ix;
    itx_dev_index D;
    std::vector<uint32_t> cname_slot, cname_off; std::vector<char> cname_pool;
    std::vector<unsigned long long> u64; std::vector<uint32_t> bp_diff, bp_diff_u, el_cnt, el_cnt_u, tid_seen, status;
    std::vector<uint32_t> grp_cpg, el_cpg; std::vector<double> grp_cpg_score, bp_cpg, el_cpg_score;
    std::vector<itx_trace> trace; uint64_t n_bad, ring_checked, ring_mismatch, tile_checked, tile_mismatch, tile_entry_miss;
    uint32_t *cname32 = nullptr;
    uint64_t xa_checked = 0, xa_mismatch = 0;             /* reads with XA put through the lane-per-alternate decomposition of k_scan; verdicts that differed from the one-lane walk */
    /* -R: smallest ordinal per key, of the unique and of the other fragments; persists across the files of a run */
    std::map<std::pair<unsigned long long, unsigned long long>, unsigned long long> dup_first;
    unsigned long long dup_min_unique = ~0ull, dup_min_other = ~0ull, dup_ord_base = 0;
};

extern "C" {

void emu_reset(emu_index *E) {
    std::fill(E->u64.begin(), E->u64.end(), 0ull);
    std::fill(E->bp_diff.begin(), E->bp_diff.end(), 0u); std::fill(E->bp_diff_u.begin(), E->bp_diff_u.end(), 0u);
    std::fill(E->el_cnt.begin(), E->el_cnt.end(), 0u); std::fill(E->el_cnt_u.begin(), E->el_cnt_u.end(), 0u);
    std::fill(E->grp_cpg.begin(), E->grp_cpg.end(), 0u); std::fill(E->el_cpg.begin(), E->el_cpg.end(), 0u);
    std::fill(E->grp_cpg_score.begin(), E->grp_cpg_score.end(), 0.0); std::fill(E->bp_cpg.begin(), E->bp_cpg.end(), 0.0);
    std::fill(E->el_cpg_score.begin(), E->el_cpg_score.end(), 0.0);
    std::fill(E->status.begin(), E->status.end(), 0u);
    E->dup_first.clear(); E->dup_min_unique = E->dup_min_other = ~0ull; E->dup_ord_base = 0;
    E->trace.clear(); E->n_bad = 0; E->ring_checked = E->ring_mismatch = 0; E->tile_checked = E->tile_mismatch = E->tile_entry_miss = 0; E->xa_checked = E->xa_mismatch = 0;
}

emu_index *emu_build(const char *chrom_sizes, const char *rep_sizes, const char *rmsk, int filter_field, const char *filter_name, char *err) {
    emu_index *E = new emu_index();
    memset(&E->ix, 0, sizeof E->ix);
    if (itx_host_index_load(&E->ix, chrom_sizes, rep_sizes, rmsk, filter_field, filter_name, err) != ITX_OK) { itx_host_index_free(&E->ix); delete E; return NULL; }
    itx_index &ix = E->ix; itx_dev_index &D = E->D;
    const int32_t nc = ix.chroms.n, ns = ix.subs.n, nf = ix.fams.n, ncl = ix.clas.n; const size_t ne = (size_t)ix.n_elem, ng = (size_t)(ns + nf + ncl);
    uint32_t nslot = 16; while (nslot < (uint32_t)nc * 2u + 2u) nslot <<= 1;
    E->cname_slot.assign(nslot, 0); E->cname_off.assign((size_t)nc + 1, 0);
    for (int32_t c = 0; c < nc; c++) {
        const char *nm = ix.chroms.names[c]; size_t l = strlen(nm);
        E->cname_off[c] = (uint32_t)E->cname_pool.size(); E->cname_pool.insert(E->cname_pool.end(), nm, nm + l + 1);
        uint32_t i = itx_fnv1a(nm, l) & (nslot - 1);
        while (E->cname_slot[i]) i = (i + 1) & (nslot - 1);
        E->cname_slot[i] = (uint32_t)c + 1;
    }
    E->cname_pool.push_back(0);
    E->u64.assign(16 + 2 * ng, 0); E->bp_diff.assign(ix.bp_len + 1, 0); E->bp_diff_u.assign(ix.bp_len + 1, 0);
    E->el_cnt.assign(ne + 1, 0); E->el_cnt_u.assign(ne + 1, 0); E->tid_seen.assign(ITX_MAX_TID_SEEN, 0); E->status.assign(8, 0);
    E->grp_cpg.assign(ng + 1, 0); E->el_cpg.assign(ne + 1, 0); E->grp_cpg_score.assign(ng + 1, 0.0); E->bp_cpg.assign(ix.bp_len + 1, 0.0); E->el_cpg_score.assign(ne + 1, 0.0);
    D.iv = ix.iv; D.ivf = ix.ivf; D.bucket = ix.bucket; D.chrom_bucket = ix.chrom_bucket; D.meta = ix.meta; D.meta2 = ix.meta2; D.chrom_off = ix.chrom_off; D.chrom_size = ix.chrom_size;
    D.n_chrom = nc; D.n_elem = ix.n_elem;
    D.cname_slot = E->cname_slot.data(); D.cname_nslot = nslot; D.cname_off = E->cname_off.data(); D.cname_pool = E->cname_pool.data(); E->cname32 = itx_names32(ix.chroms.names, nc); D.cname32 = E->cname32;
    D.n_sub = ns; D.n_fam = nf; D.n_cla = ncl; D.stat_mode = ix.stat_mode;
    D.sub_len = ix.sub_len; D.sub_bp_off = ix.sub_bp_off; D.sub_fold = ix.sub_fold; D.cinfo = ix.cinfo; D.sinfo = ix.sinfo;
    D.cnt = E->u64.data(); D.grp = D.cnt + 16; D.bp_diff = E->bp_diff.data(); D.bp_diff_u = E->bp_diff_u.data();
    D.el_cnt = E->el_cnt.data(); D.el_cnt_u = E->el_cnt_u.data();
    D.grp_cpg = E->grp_cpg.data(); D.el_cpg = E->el_cpg.data(); D.grp_cpg_score = E->grp_cpg_score.data(); D.bp_cpg = E->bp_cpg.data(); D.el_cpg_score = E->el_cpg_score.data();
    D.tid_unknown_seen = E->tid_seen.data(); D.status = E->status.data();
    E->n_bad = 0; E->ring_checked = E->ring_mismatch = 0; E->tile_checked = E->tile_mismatch = E->tile_entry_miss = 0;
    return E;
}
void emu_free(emu_index *E) { if (!E) return; itx_host_index_free(&E->ix); free(E->cname32); delete E; }
itx_index *emu_host_index(emu_index *E) { return &E->ix; }

/* the ring the TMA decode kernel reads records from: 4 tiles of 2 KiB addressed by (offset & 8191) */
static const uint32_t EMU_TILE = 2048, EMU_RING = 8192;
static void walk_chunk(emu_index *E, const uint8_t *b, uint64_t len, uint64_t lo, uint32_t C, uint64_t p, const itx_bam_header &h, const itx_dev_opts &o,
                       std::vector<itx_tuple> &out, uint64_t *exit_, uint64_t own = ~0ull) {
    const itx_src_global G{b};
    alignas(16) static thread_local uint8_t ring[EMU_RING];
    const itx_src_ring R{ring, EMU_RING - 1};
    uint64_t ring_t0 = ~0ull;
    uint64_t hi = lo + C; if (hi > len) hi = len; if (hi > own) hi = own;
    out.clear();
    if (p < ITX_OFF_END) {
        while (p < hi) {
            if (p + 36 > len) { p = ITX_OFF_END; break; }
            uint32_t x[9]; G.core(p, x);
            if ((int32_t)x[0] < 32 || p + 4 + (uint64_t)x[0] > len) { p = ITX_OFF_END; break; }
            const itx_tuple T = itx_decode_record(G, p, x, (uint32_t)(p - lo), h.tid, h.n_ref, o);
            out.push_back(T);
            /* cross-check: the same record decoded out of the shared-memory ring layout */
            const uint64_t t0 = p / EMU_TILE, F = (t0 + 2) * EMU_TILE;
            if (p + 4 + (uint64_t)x[0] <= F) {
                if (t0 != ring_t0) {
                    for (uint64_t t = t0; t < t0 + 2; t++) {
                        const uint64_t off = t * EMU_TILE; if (off >= len + 64) break;
                        uint64_t nb = len + 64 - off; if (nb > EMU_TILE) nb = EMU_TILE;
                        memcpy(ring + (off & (EMU_RING - 1)), b + off, nb);
                    }
                    ring_t0 = t0;
                }
                uint32_t y[9]; R.core(p, y);
                const itx_tuple T2 = itx_decode_record(R, p, y, (uint32_t)(p - lo), h.tid, h.n_ref, o);
                E->ring_checked++;
                if (memcmp(x, y, sizeof x) != 0 || memcmp(&T, &T2, sizeof T) != 0 || R.u32(p) != x[0]) E->ring_mismatch++;
            }
            p += 4 + (uint64_t)x[0];
        }
    }
    *exit_ = p;
}

/* The span kernels' chain (k_scan / k_decode_span), simulated lane by lane with the very functions the kernels call
 * (itx_plausible2_core for the span guess, itx_buf_u32 / itx_chain_lane for a step of the walk): the span's first record
 * start is guessed 32 offsets per step out of the span's first bytes, then the chain is carried stage by stage
 * (ITX_EMU_STAGE bytes, as the kernels' ITX_STAGE) with run prediction on the span's dominant record size.  Offsets are
 * span-relative and 32 bits wide, sentinels 0xfffffffe (chain ended) / 0xffffffff (no guess) as in the kernels.
 * Returns the entry, the record starts and the exit, to be compared with the sequential chain. */
#define ITX_EMU_STAGE 4096u
static void span_chain(const uint8_t *b, uint64_t len, uint64_t lo, uint32_t C, int32_t n_ref, bool first, uint64_t carry,
                       uint64_t *entry0, std::vector<uint64_t> *starts, uint64_t *exitX) {
    const itx_src_global G{b};
    const uint32_t hi = len - lo < C ? (uint32_t)(len - lo) : C;
    uint32_t p = 0xffffffffu;
    if (first) p = carry >= ITX_OFF_END ? (uint32_t)carry : (carry - lo < 0xfffffff0ull ? (uint32_t)(carry - lo) : 0xfffffffeu);
    else {
        for (uint32_t base = 0; base < hi && p == 0xffffffffu; base += 32) {
            uint32_t m = 0;
            for (uint32_t lane = 0; lane < 32; lane++) {
                const uint32_t d = base + lane; const uint64_t q = lo + d;
                bool ok = false;
                if (d < hi && q + 36 <= len) { uint32_t x[9]; G.core(q, x); ok = itx_plausible2_core(G, x, q, len, n_ref); }
                if (ok) m |= 1u << lane;
            }
            if (m) p = base + (uint32_t)__builtin_ctz(m);
        }
    }
    *entry0 = p >= 0xfffffffeu ? (0xffffffff00000000ull | p) : lo + p;
    starts->clear();
    uint32_t szd = 0;
    while (p < hi) {
        const uint32_t c_lo = p & ~(ITX_EMU_STAGE - 1u), c_hi = c_lo + ITX_EMU_STAGE < hi ? c_lo + ITX_EMU_STAGE : hi;
        const uint64_t rest = len - lo - c_lo;
        const uint8_t *buf = b + lo + c_lo;
        uint32_t q = p - c_lo;
        const uint32_t qh = c_hi - c_lo, room32 = rest > 0x7fffffffull ? 0x7fffffffu : (uint32_t)rest;
        while (q < qh) {
            if (q + 36u > room32) { q = 0xffffffffu; break; }
            const uint32_t bs0 = itx_buf_u32(buf, q), sz0 = bs0 + 4u;
            if ((int32_t)bs0 < 32 || sz0 > room32 - q) { q = 0xffffffffu; break; }
            const uint32_t szp = szd ? szd : sz0;
            uint32_t run = 1u, pks[32]; pks[0] = q;
            if ((sz0 | szp) < 0x10000u) {
                uint32_t m = 0;
                for (uint32_t lane = 0; lane < 32; lane++) if (itx_chain_lane(buf, q, sz0, szp, lane, qh, room32, &pks[lane])) m |= 1u << lane;
                run = m == 0xffffffffu ? 32u : (uint32_t)__builtin_ctz(~m);
            }
            for (uint32_t lane = 0; lane < run; lane++) starts->push_back(lo + c_lo + pks[lane]);
            q += sz0 + (run - 1u) * szp;
            szd = run >= 2u ? szp : 0u;
        }
        if (q == 0xffffffffu) { p = 0xfffffffeu; break; }
        p = c_lo + q;
    }
    *exitX = p >= 0xfffffffeu ? (0xffffffff00000000ull | p) : lo + p;
}

/* k_scan's XA walk for ONE read, composed exactly as the kernel composes it: the pieces are counted (itx_xa_count), handed out
 * 32 at a time -- one per lane -- each lane finds its piece (itx_xa_kth) and tests it (itx_xa_piece); the first alternate that
 * answers yes ends the walk and the malformed ones before it are counted. */
static bool xa_lanes(const itx_dev_index &D, const itx_src_global &G, uint64_t p, const uint32_t x[9], int32_t fold, int32_t qlen, uint32_t *malformed) {
    uint64_t a0, aend; itx_aux_range(p, x, &a0, &aend);
    if (aend - a0 < 5) return false;
    const uint64_t xa = itx_aux_find(G, a0, aend, 'X', 'A');
    if (!xa || xa >= aend) return false;
    const int32_t nm = itx_aux2i(G, itx_aux_find(G, a0, aend, 'N', 'M'), aend);
    const uint8_t ty = G.u8(xa);
    if (ty != 'Z' && ty != 'H') return false;
    uint64_t ze, ze2; const uint64_t zs = xa + 1;
    uint32_t sp[2]; bool packed;
    const uint32_t np = itx_xa_count_pack(G, zs, aend, &ze, sp, &packed);
    if (np != itx_xa_count(G, zs, aend, &ze2) || ze != ze2) return !*malformed && false;      /* (never: the two counters agree) */
    bool found = false;
    for (uint32_t b0 = 0; b0 < np && !found; b0 += 32) {
        uint32_t m_hit = 0, m_mal = 0;
        for (uint32_t lane = 0; lane < 32 && b0 + lane < np; lane++) {
            uint64_t ps, pe; bool mal = false, hit = false;
            const uint32_t k = b0 + lane;
            if (packed && k < 8u) {                              /* as k_xa: bounds out of the owner's notes, checked here against the scan */
                uint64_t ps2, pe2;
                itx_xa_piece_bounds(zs, ze, np, sp, k, &ps, &pe);
                itx_xa_kth(G, zs, ze, k, &ps2, &pe2);
                if (ps != ps2 || pe != pe2) { *malformed += 1000000u; }
            } else itx_xa_kth(G, zs, ze, k, &ps, &pe);
            if (pe > ps) hit = itx_xa_piece(D, G, ps, pe, nm, qlen, fold, &mal);
            if (hit) m_hit |= 1u << lane;
            if (mal) m_mal |= 1u << lane;
        }
        if (m_hit) { found = true; *malformed += (uint32_t)__builtin_popcount(m_mal & ((1u << __builtin_ctz(m_hit)) - 1u)); }
        else *malformed += (uint32_t)__builtin_popcount(m_mal);
    }
    return found;
}

/* k_xa as it is now: the aux area of the read is STAGED (16-byte granules around it, as the kernel's cp.async brings them into the
 * warp's pool; everything else in the pool is poisoned here) and parsed with 32-bit pool-relative offsets through itx_src_flat; a
 * read whose aux area does not fit, or whose tag walk meets an array count that leaves the area, takes the one-lane 64-bit walk
 * over global memory -- the kernel's fallback.  Returns the verdict; *malformed as the kernel would count it. */
static const uint32_t EMU_XA_POOL = 6144;
static bool xa_staged(const itx_dev_index &D, const itx_src_global &G, uint64_t p, const uint32_t x[9], int32_t fold, int32_t qlen, uint32_t *malformed, uint32_t pool_off, bool *counted_go) {
    uint64_t a0, aend; itx_aux_range(p, x, &a0, &aend);
    *counted_go = a0 < aend;
    if (!(a0 < aend)) return false;
    const uint64_t base = a0 & ~15ull;
    bool big = aend - base > (uint64_t)(EMU_XA_POOL - 16u);
    bool diffsub = false;
    if (!big) {
        const uint32_t need = (uint32_t)((aend - base + 15ull) & ~15ull);
        if (pool_off + need > EMU_XA_POOL) pool_off = 0;
        alignas(16) static thread_local uint8_t pool[EMU_XA_POOL + 64];
        memset(pool, 0xA5, sizeof pool);
        memcpy(pool + pool_off, G.b + base, need);
        const uint32_t a0r = (uint32_t)(a0 - base), aendr = (uint32_t)(aend - base);
        const itx_src_flat S{pool + pool_off, 0ull};
        const uint32_t xa = itx_aux_find(S, a0r, aendr, (uint8_t)'X', (uint8_t)'A');
        const uint32_t nmo = xa == 0xffffffffu ? xa : itx_aux_find(S, a0r, aendr, (uint8_t)'N', (uint8_t)'M');
        if (xa == 0xffffffffu || nmo == 0xffffffffu) big = true;
        else if (xa && xa < aendr) {
            const int32_t nm = itx_aux2i(S, nmo, aendr);
            const uint8_t ty = S.u8(xa);
            uint32_t np = 0, zs = 0, ze = 0, sp[2] = {0, 0}; bool packed = false;
            if (ty == 'Z' || ty == 'H') { zs = xa + 1u; np = itx_xa_count_pack(S, zs, aendr, &ze, sp, &packed); }
            bool found = false;
            for (uint32_t b0 = 0; b0 < np && !found; b0 += 32) {
                uint32_t m_hit = 0, m_mal = 0;
                for (uint32_t lane = 0; lane < 32 && b0 + lane < np; lane++) {
                    uint32_t ps, pe; bool mal = false, hit = false;
                    const uint32_t k = b0 + lane;
                    if (packed && k < 8u) itx_xa_piece_bounds(zs, ze, np, sp, k, &ps, &pe);
                    else itx_xa_kth(S, zs, ze, k, &ps, &pe);
                    if (pe > ps) hit = itx_xa_piece_fast(D, S, ps, pe, nm, qlen, fold, &mal);
                    if (hit) m_hit |= 1u << lane;
                    if (mal) m_mal |= 1u << lane;
                }
                if (m_hit) { found = true; *malformed += (uint32_t)__builtin_popcount(m_mal & ((1u << __builtin_ctz(m_hit)) - 1u)); }
                else *malformed += (uint32_t)__builtin_popcount(m_mal);
            }
            diffsub = found;
        } else *counted_go = false;
    }
    if (big) {
        const uint64_t xa = itx_aux_find(G, a0, aend, (uint8_t)'X', (uint8_t)'A');
        if (xa && xa < aend) {
            const int32_t nm = itx_aux2i(G, itx_aux_find(G, a0, aend, (uint8_t)'N', (uint8_t)'M'), aend);
            diffsub = itx_xa_walk(D, G, xa, aend, nm, fold, qlen, malformed);
        } else *counted_go = false;
    }
    return diffsub;
}

/* the chain rule of the kernels (itx_span_consistent): the exit that counts for span i is that of the last span before it
 * that holds a record start; a span that met none is right when the chain runs over it or has ended */
static uint64_t prev_exit(const std::vector<uint64_t> &exit_, uint64_t j) { uint64_t x = exit_[j]; while (x == ITX_OFF_NONE && j > 0) { j--; x = exit_[j]; } return x; }
static bool span_consistent(const std::vector<uint64_t> &entry, const std::vector<uint64_t> &exit_, uint64_t i, uint64_t span_end, uint64_t own) {
    const uint64_t en = entry[i], ex = prev_exit(exit_, i - 1);
    if (en == ex || ex == ITX_OFF_NONE) return true;
    if (en != ITX_OFF_NONE) return false;
    return ex == ITX_OFF_END || (ex < ITX_OFF_GUESS && ex >= (span_end < own ? span_end : own));
}

/* bam: uncompressed stream with >= 64 readable bytes after len.  want_trace: keep a per-record trace. */
static int emu_scan_core(emu_index *E, const uint8_t *hdr_bam, uint64_t hdr_bytes, const uint8_t *bam, uint64_t len, uint64_t own, uint64_t carry0, const itx_scan_opts *so,
                         uint32_t chunk, int want_trace, uint64_t cnt[13], uint64_t *entry_out, uint64_t *exit_out, char *err);
int emu_scan_stream(emu_index *E, const uint8_t *bam, uint64_t len, const itx_scan_opts *so, uint32_t chunk, int want_trace, uint64_t cnt[13], char *err) {
    return emu_scan_core(E, bam, len, bam, len, ~0ull, ~0ull, so, chunk, want_trace, cnt, NULL, NULL, err);
}
/* one rank's part of a stream (itx_scan_shard_file on the device): `bam` holds the rank's own bytes [0, own) plus a margin up to len
 * and no header (that comes from hdr_bam, the start of the file); carry0 = ITX_OFF_GUESS or the forced entry */
int emu_scan_shard(emu_index *E, const uint8_t *hdr_bam, uint64_t hdr_bytes, const uint8_t *bam, uint64_t len, uint64_t own, uint64_t carry0, const itx_scan_opts *so,
                   uint32_t chunk, uint64_t cnt[13], uint64_t *entry_rel, uint64_t *exit_rel, char *err) {
    uint64_t en = ITX_OFF_NONE, ex = ITX_OFF_NONE;
    int rc = emu_scan_core(E, hdr_bam, hdr_bytes, bam, len, own, carry0, so, chunk, 0, cnt, &en, &ex, err);
    if (rc) return rc;
    *entry_rel = en;
    *exit_rel = ex >= ITX_OFF_GUESS ? (ex == ITX_OFF_GUESS ? ITX_OFF_NONE : ex) : (ex >= own ? ex - own : 0);
    return ITX_OK;
}
static int emu_scan_core(emu_index *E, const uint8_t *hdr_bam, uint64_t hdr_bytes, const uint8_t *bam, uint64_t len, uint64_t own, uint64_t carry0, const itx_scan_opts *so,
                         uint32_t chunk, int want_trace, uint64_t cnt[13], uint64_t *entry_out, uint64_t *exit_out, char *err) {
    itx_index &ix = E->ix; itx_dev_index &D = E->D;
    itx_bam_header h;
    if (itx_host_parse_bam_header(&ix, hdr_bam, hdr_bytes, so->addChr, &h, err) != ITX_OK) return ITX_EFORMAT;
    if (own > len) own = len;
    if (carry0 == ~0ull) carry0 = h.hdr_len;
    const uint64_t first_byte = carry0 >= ITX_OFF_GUESS ? 0 : carry0;
    itx_dev_opts o; o.mapQ = so->mapQ; o.iSize = so->iSize; o.extension = so->extension; o.minCoverage = so->minCoverage;
    o.filter = so->filter; o.discardWrongEnd = so->discardWrongEnd; o.treat = so->treat; o.diffSubfam = so->diffSubfam;
    const uint32_t C = chunk;
    const uint64_t k0 = first_byte / C, k1 = own > first_byte ? (own + C - 1) / C : k0, n = k1 - k0;
    std::vector<std::vector<itx_tuple>> tup(n);
    std::vector<uint64_t> entry(n), exit_(n);
    /* K1: every chunk guesses its entry independently (chunk 0 knows it, unless the scan starts in the middle of a stream) */
    for (uint64_t i = 0; i < n; i++) {
        uint64_t lo = (k0 + i) * C, hi = lo + C; if (hi > own) hi = own;
        uint64_t p = (i == 0 && carry0 != ITX_OFF_GUESS) ? carry0 : itx_speculate_entry(itx_src_global{bam}, lo, hi, len, h.n_ref);
        entry[i] = p;
        walk_chunk(E, bam, len, lo, C, p, h, o, tup[i], &exit_[i], own);
    }
    /* verify + repair (k_verify / k_fixup) */
    for (uint64_t i = 1; i < n; i++) if (!span_consistent(entry, exit_, i, (k0 + i) * C + C, own)) {
        E->n_bad++;
        entry[i] = prev_exit(exit_, i - 1);
        walk_chunk(E, bam, len, (k0 + i) * C, C, entry[i], h, o, tup[i], &exit_[i], own);
    }
    if (entry_out) { *entry_out = ITX_OFF_NONE; if (carry0 != ITX_OFF_GUESS) *entry_out = carry0; else for (uint64_t i = 0; i < n && *entry_out == ITX_OFF_NONE; i++) *entry_out = entry[i]; }
    if (exit_out) { *exit_out = n ? prev_exit(exit_, n - 1) : carry0; if (*exit_out == ITX_OFF_NONE && carry0 == ITX_OFF_GUESS) *exit_out = ITX_OFF_GUESS; }
    /* the span kernels' chain (staged guess, run-predicted walk), span by span, against the sequential chain */
    if ((C % ITX_EMU_STAGE) == 0 && C <= (1u << 20) && own == len && carry0 == h.hdr_len) {
        for (uint64_t i = 0; i < n; i++) {
            uint64_t e0, ex; std::vector<uint64_t> st;
            span_chain(bam, len, (k0 + i) * C, C, h.n_ref, i == 0, i == 0 ? h.hdr_len : 0, &e0, &st, &ex);
            E->tile_checked++;
            if (e0 != entry[i]) { E->tile_entry_miss++; continue; }     /* a wrong chunk guess: the repair path's business */
            bool same = ex == exit_[i] && st.size() == tup[i].size();
            for (size_t j = 0; same && j < st.size(); j++) same = (uint32_t)(st[j] - (k0 + i) * C) == tup[i][j].rec_off;
            if (!same) E->tile_mismatch++;
        }
    }
    /* -R: the two passes of k_dedup (enter every unique fragment's key, then flag what is not its key's first) */
    if (so->rmDup) {
        const uint64_t S = C / 36 + 1;
        auto key_of = [&](uint64_t i, const itx_tuple &T) {
            const int32_t t = (int32_t)itx_src_global{bam}.u32((k0 + i) * C + T.rec_off + 4);
            unsigned long long lo, hi; itx_dup_key((t >= 0 && t < h.n_ref) ? h.tid[t].csid : -1, (T.info & ITX_F_MINUS) != 0, T.start, T.end, &lo, &hi);
            return std::make_pair(lo, hi);
        };
        for (uint64_t i = 0; i < n; i++) for (size_t j = 0; j < tup[i].size(); j++) {
            const itx_tuple &T = tup[i][j]; if (!(T.info & ITX_F_FRAG)) continue;
            const unsigned long long ord = E->dup_ord_base + (k0 + i) * S + j;
            if (T.info & ITX_F_UNIQ) {
                auto it = E->dup_first.insert(std::make_pair(key_of(i, T), ord)).first;
                if (ord < it->second) it->second = ord;
                if (ord < E->dup_min_unique) E->dup_min_unique = ord;
            } else if (ord < E->dup_min_other) E->dup_min_other = ord;
        }
        for (uint64_t i = 0; i < n; i++) for (size_t j = 0; j < tup[i].size(); j++) {
            itx_tuple &T = tup[i][j]; if (!(T.info & ITX_F_FRAG)) continue;
            const unsigned long long ord = E->dup_ord_base + (k0 + i) * S + j;
            const bool keep = (T.info & ITX_F_UNIQ) ? E->dup_first[key_of(i, T)] == ord : itx_dup_nonunique_kept(ord, E->dup_min_unique, E->dup_min_other);
            if (!keep) T.info |= ITX_F_DUP;
        }
        E->dup_ord_base += (k1 + 1) * S;
    }
    /* ordered side outputs: the same host pass as the product, fed by this run's trace */
    const bool ordered = so->outbed || so->outbed_unique || so->readNames;
    const size_t trace0 = E->trace.size();
    if (ordered) want_trace = 1;
    /* K2 + K3 */
    unsigned long long *c = D.cnt;
    const bool stat = o.filter == 0 && D.stat_mode;
    const itx_src_global G{bam};
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t lo = (k0 + i) * C;
        for (size_t j = 0; j < tup[i].size(); j++) {
            const itx_tuple T = tup[i][j]; const uint32_t info = T.info;
            const bool slot2 = info & ITX_F_SLOT2, frag = info & ITX_F_FRAG, uniq = info & ITX_F_UNIQ, live = frag && !(info & ITX_F_DUP);
            c[slot2 ? 1 : 0]++;
            if (info & ITX_F_MAPPED) c[slot2 ? 3 : 2]++;
            if (info & ITX_F_USED) c[slot2 ? 5 : 4]++;
            if (frag) { c[6]++; if (uniq) { c[7]++; if (live) c[11]++; } }
            if ((info & ITX_F_UNKNOWN) && T.start < ITX_MAX_TID_SEEN) D.tid_unknown_seen[T.start] = 1;
            long long sel = -1; bool diffsub = false; itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
            const uint32_t chrom = info & ITX_CHROM_MASK;
            if (live && chrom != ITX_CHROM_NONE) {
                int32_t nh; float tcov;
                sel = itx_find_select(D, (int32_t)chrom, T.start, T.end, o.minCoverage, &nh, &tcov, &e);
                if (sel >= 0 && tcov < o.minCoverage) sel = -1;
                if (sel >= 0 && o.diffSubfam && (info & ITX_F_HASXA)) {
                    const uint64_t p = lo + T.rec_off; uint32_t x[9]; G.core(p, x); uint32_t bad = 0;
                    if (itx_mapped_to_diff_subfam(D, G, p, x, D.sinfo[D.meta[sel].sub].fold, (int32_t)(T.end - T.start), &bad)) diffsub = true;
                    D.status[2] += bad;
                    uint32_t bad2 = 0;
                    const bool d2 = xa_lanes(D, G, p, x, D.sinfo[D.meta[sel].sub].fold, (int32_t)(T.end - T.start), &bad2);
                    E->xa_checked++;
                    if (d2 != diffsub || bad2 != bad) E->xa_mismatch++;
                    /* and k_xa's staged 32-bit walk, at a pool offset that moves from read to read */
                    uint32_t bad3 = 0; bool go3 = false;
                    const bool d3 = xa_staged(D, G, p, x, D.sinfo[D.meta[sel].sub].fold, (int32_t)(T.end - T.start), &bad3, (uint32_t)((E->xa_checked * 48u) % EMU_XA_POOL) & ~15u, &go3);
                    if (d3 != diffsub || bad3 != bad || !go3) E->xa_mismatch++;
                }
            }
            if (diffsub) c[12]++;
            const bool counted = sel >= 0 && !diffsub;
            if (counted) {
                c[9]++; if (uniq) c[10]++;
                if (stat) {
                    const itx_meta m = D.meta[sel]; const itx_meta2 m2 = D.meta2[sel];
                    const uint32_t hs = 2u * m.sub, hf = 2u * (uint32_t)(D.n_sub + m2.fam), hc = 2u * (uint32_t)(D.n_sub + D.n_fam + m2.cla);
                    D.grp[hs]++; D.grp[hf]++; D.grp[hc]++;
                    if (uniq) { D.grp[hs + 1]++; D.grp[hf + 1]++; D.grp[hc + 1]++; }
                    const uint32_t L = D.sub_len[m.sub]; uint32_t ja, jb;
                    if (L && itx_cov_range(T.start, T.end - T.start, e.start, e.end, m.cons_start, m.cons_end, L, &ja, &jb)) {
                        const unsigned long long off = D.sub_bp_off[m.sub];
                        D.bp_diff[off + ja] += 1u; D.bp_diff[off + jb] += 0xffffffffu;
                        if (uniq) { D.bp_diff_u[off + ja] += 1u; D.bp_diff_u[off + jb] += 0xffffffffu; }
                    }
                } else if (o.filter) { D.el_cnt[sel]++; if (uniq) D.el_cnt_u[sel]++; }
            }
            if (want_trace) {
                itx_trace t;
                t.start = live ? T.start : 0; t.end = live ? T.end : 0; t.tid = (int32_t)G.u32(lo + T.rec_off + 4);
                t.sel_row = sel >= 0 ? (int32_t)e.row : -1;
                t.flags = (live ? ITX_T_FRAGMENT : 0u) | (live && uniq ? ITX_T_UNIQ : 0u) | ((live && (info & ITX_F_MINUS)) ? ITX_T_MINUS : 0u) |
                          ((live && (info & ITX_F_HASXA)) ? ITX_T_HAS_XA : 0u) | (diffsub ? ITX_T_DIFFSUB : 0u) | (counted ? ITX_T_COUNTED : 0u) |
                          ((info & ITX_F_DUP) ? ITX_T_DUP : 0u);
                E->trace.push_back(t);
            }
        }
    }
    if (ordered) {
        itx_ordered_sink K; K.bed = so->outbed ? fopen(so->outbed, "w") : NULL; K.bed_u = so->outbed_unique ? fopen(so->outbed_unique, "w") : NULL;
        K.names = so->readNames != 0; K.mapQ = so->mapQ; K.tname = itx_ordered_tnames(&h); K.n_ref = h.n_ref; K.ix = &ix;
        if (K.names) itx_ordered_names_init(&ix);
        itx_ordered_walk(K, bam + h.hdr_len, len - h.hdr_len, E->trace.data() + trace0, E->trace.size() - trace0);
        if (K.bed) fclose(K.bed);
        if (K.bed_u) fclose(K.bed_u);
        for (int32_t i = 0; i < h.n_ref; i++) free(K.tname[i]);
        free(K.tname);
    }
    for (int k = 0; k < 13; k++) { ix.cnt[k] = c[k]; if (cnt) cnt[k] = c[k]; }
    for (int32_t i = 0; i < h.n_ref; i++) free(h.names[i]);
    free(h.names); free(h.lens); free(h.tid);
    return ITX_OK;
}

/* results -> the host index (what itx_sync_counts does after the device run) */
void emu_sync(emu_index *E) {
    itx_index &ix = E->ix; itx_dev_index &D = E->D;
    const size_t ne = (size_t)ix.n_elem, bl = (size_t)ix.bp_len;
    if (!ix.bp) { ix.bp = (uint32_t *)calloc(bl + 1, 4); ix.bp_u = (uint32_t *)calloc(bl + 1, 4); ix.bp_cpg = (double *)calloc(bl + 1, 8); }
    if (!ix.el_cnt) { ix.el_cnt = (uint32_t *)calloc(ne + 1, 4); ix.el_cnt_u = (uint32_t *)calloc(ne + 1, 4); ix.el_cpg = (uint32_t *)calloc(ne + 1, 4); ix.el_cpg_score = (double *)calloc(ne + 1, 8); }
    for (int32_t s = 0; s < ix.subs.n; s++) {
        uint32_t L = ix.sub_len[s]; if (!L) continue;
        uint64_t off = ix.sub_bp_off[s]; uint32_t a = 0, u = 0;
        for (uint32_t j = 0; j <= L; j++) { a += D.bp_diff[off + j]; u += D.bp_diff_u[off + j]; ix.bp[off + j] = a; ix.bp_u[off + j] = u; }
    }
    memcpy(ix.el_cnt, D.el_cnt, ne * 4); memcpy(ix.el_cnt_u, D.el_cnt_u, ne * 4);
    memcpy(ix.el_cpg, D.el_cpg, ne * 4); memcpy(ix.el_cpg_score, D.el_cpg_score, ne * 8); memcpy(ix.bp_cpg, D.bp_cpg, bl * 8);
    const int32_t ns = ix.subs.n, nf = ix.fams.n, nc = ix.clas.n; const unsigned long long *g = D.grp;
    for (int32_t i = 0; i < ns; i++) { ix.sub[i].read_count = g[2 * i]; ix.sub[i].read_count_unique = g[2 * i + 1]; ix.sub[i].cpg_count = D.grp_cpg[i]; ix.sub[i].cpg_score = D.grp_cpg_score[i]; }
    for (int32_t i = 0; i < nf; i++) { ix.fam[i].read_count = g[2 * (ns + i)]; ix.fam[i].read_count_unique = g[2 * (ns + i) + 1]; ix.fam[i].cpg_count = D.grp_cpg[ns + i]; ix.fam[i].cpg_score = D.grp_cpg_score[ns + i]; }
    for (int32_t i = 0; i < nc; i++) { ix.cla[i].read_count = g[2 * (ns + nf + i)]; ix.cla[i].read_count_unique = g[2 * (ns + nf + i) + 1]; ix.cla[i].cpg_count = D.grp_cpg[ns + nf + i]; ix.cla[i].cpg_score = D.grp_cpg_score[ns + nf + i]; }
}

uint64_t emu_trace(emu_index *E, itx_trace *out, uint64_t cap) {
    uint64_t n = E->trace.size() < cap ? E->trace.size() : cap;
    memcpy(out, E->trace.data(), n * sizeof(itx_trace));
    return E->trace.size();
}
uint64_t emu_n_bad(emu_index *E) { return E->n_bad; }
uint64_t emu_xa_checked(emu_index *E) { return E->xa_checked; }
uint64_t emu_xa_fast(int which) { return g_xa_fast[which & 1]; }
/* itx_xa_piece_fast against itx_xa_piece on generated alternates: names of the index, near misses, long and empty names; positions
 * with and without signs, leading zeros, hexadecimal, white space, too many digits; any number of commas.  Returns the number of
 * pieces on which verdict or malformed flag differ (0). */
uint64_t emu_xa_fuzz(emu_index *E, uint64_t seed, uint64_t n) {
    const itx_dev_index &D = E->D; const itx_index &ix = E->ix;
    uint64_t st = seed * 6364136223846793005ull + 1442695040888963407ull, bad = 0;
    auto rnd = [&](uint32_t m) { st = st * 6364136223846793005ull + 1442695040888963407ull; return (uint32_t)((st >> 33) % (m ? m : 1)); };
    alignas(16) static thread_local uint8_t pool[512 + 64];
    for (uint64_t it = 0; it < n; it++) {
        std::string p;
        /* name */
        switch (rnd(8)) {
        case 0: break;
        case 1: { const int L = 1 + (int)rnd(40); for (int i = 0; i < L; i++) p.push_back((char)('a' + rnd(26))); break; }
        case 2: { std::string nm = ix.chroms.n ? ix.chroms.names[rnd((uint32_t)ix.chroms.n)] : "chr1"; nm.push_back((char)('0' + rnd(10))); p += nm; break; }
        case 3: { std::string nm = ix.chroms.n ? ix.chroms.names[rnd((uint32_t)ix.chroms.n)] : "chr1"; if (!nm.empty()) nm.pop_back(); p += nm; break; }
        default: p += ix.chroms.n ? ix.chroms.names[rnd((uint32_t)ix.chroms.n)] : "chr1";
        }
        const uint32_t ncomma = rnd(10) < 7 ? 3u : rnd(6);
        for (uint32_t f = 1; f <= ncomma; f++) {
            p.push_back(',');
            if (f == 1 || f == 3 || f > 3) {                       /* a number */
                const uint32_t k = rnd(16);
                if (k == 0) continue;
                if (k == 1) p += " ";
                if (k == 2) p += "0x";
                if (k == 3) p += "0";
                if (f == 1 && rnd(4)) p.push_back(rnd(2) ? '+' : '-');
                if (k == 4) p.push_back('-');
                const uint32_t nd = f == 1 ? (k == 5 ? 9 + rnd(12) : 1 + rnd(9)) : (k == 5 ? 1 + rnd(6) : 1);
                for (uint32_t i = 0; i < nd; i++) p.push_back((char)('0' + ((i == 0 && k != 6) ? 1 + rnd(9) : rnd(10))));
                if (k == 7) p.push_back('x');
                if (k == 8) p += "  ";
            } else { const int L = (int)rnd(8); for (int i = 0; i < L; i++) p.push_back("0123456789MIDNS"[rnd(15)]); }
        }
        if (p.empty() || p.size() > 400) continue;
        const uint32_t off = 16u * rnd(4) + rnd(4);                /* every alignment of the piece inside its words */
        memset(pool, 0xA5, sizeof pool);
        memcpy(pool + off, p.data(), p.size());
        const itx_src_flat S{pool, 0ull};
        const int32_t nm = (int32_t)rnd(4), qlen = 30 + (int32_t)rnd(100), fold = (int32_t)rnd((uint32_t)(ix.subs.n ? ix.subs.n : 1));
        bool m1 = false, m2 = false;
        int64_t a1[5], a2[5];
        memset(g_xa_walk, 0, sizeof g_xa_walk);
        const bool h1 = itx_xa_piece_fast(D, S, off, off + (uint32_t)p.size(), nm, qlen, fold, &m1);
        memcpy(a1, g_xa_walk, sizeof a1); memset(g_xa_walk, 0, sizeof g_xa_walk);
        const bool h2 = itx_xa_piece(D, S, off, off + (uint32_t)p.size(), nm, qlen, fold, &m2);
        memcpy(a2, g_xa_walk, sizeof a2);
        /* the same verdict, the same malformed flag, and the same question to the table (chromosome, start, end) if one was asked */
        if (h1 != h2 || m1 != m2 || memcmp(a1, a2, sizeof a1) != 0) { if (bad < 5) fprintf(stderr, "xa fuzz: '%s' fast %d/%d general %d/%d\n", p.c_str(), (int)h1, (int)m1, (int)h2, (int)m2); bad++; }
    }
    return bad;
}
uint64_t emu_xa_mismatch(emu_index *E) { return E->xa_mismatch; }
uint64_t emu_ring_checked(emu_index *E) { return E->ring_checked; }
uint64_t emu_ring_mismatch(emu_index *E) { return E->ring_mismatch; }
uint64_t emu_tile_checked(emu_index *E) { return E->tile_checked; }
uint64_t emu_tile_mismatch(emu_index *E) { return E->tile_mismatch; }
uint64_t emu_tile_entry_miss(emu_index *E) { return E->tile_entry_miss; }

/* The two arithmetic shortcuts of itx_select_walk, checked against the float arithmetic they stand for (getCov,
 * generic.c:296-301, and the comparisons at generic.c:950-962):
 *   (1) for den < 2^23 and ra, rb <= den, (float)ra / (float)den > (float)rb / (float)den  <=>  ra > rb;
 *   (2) itx_cov_thr(r, den, thr) < thr  <=>  the float quotient < thr, for any thr.
 * Random cases plus the edges (overlaps around den / 4096, den around 2^23 and 2^24, thresholds next to 2^-13).
 * Returns the number of violations. */
static float exact_cov(uint32_t r, uint32_t den) {
    if (r != 0 && r == den) return 1.0f;
    volatile float d = (float)den, n = (float)(int32_t)r;      /* volatile: plain float division, no contraction */
    return d == 0.0f ? 0.0f : n / d;
}
uint64_t emu_check_cov_rules(uint64_t n, uint64_t seed) {
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + 1, bad = 0;
    auto rnd = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    const float thr_fixed[] = {1e-4f, ITX_COV_FLOOR, std::nextafterf(ITX_COV_FLOOR, 0.0f), std::nextafterf(ITX_COV_FLOOR, 1.0f), 0.0f, 0.00012f,
                               0.000244140625f, 0.5f, 1.0f, 2.0f, -1.0f, 1e-30f};
    for (uint64_t k = 0; k < n; k++) {
        uint32_t den;
        switch (rnd() % 6) {
            case 0: den = 1 + (uint32_t)(rnd() % 400); break;                        /* reads */
            case 1: den = 1 + (uint32_t)(rnd() % 100000); break;                     /* fragments */
            case 2: den = (1u << 23) - 1 - (uint32_t)(rnd() % 64); break;            /* just below the integer-comparison limit */
            case 3: den = (1u << 23) + (uint32_t)(rnd() % (1u << 24)); break;        /* above it: only rule (2) applies */
            case 4: den = 4096u * (1 + (uint32_t)(rnd() % 5000)) + (uint32_t)(rnd() % 3) - 1; break;   /* around multiples of 2^12 */
            default: den = 1 + (uint32_t)(rnd() % ((1u << 23) - 1)); break;
        }
        uint32_t ra, rb;
        switch (rnd() % 4) {
            case 0: ra = (uint32_t)(rnd() % ((uint64_t)den + 1)); rb = (uint32_t)(rnd() % ((uint64_t)den + 1)); break;
            case 1: ra = (uint32_t)(rnd() % ((uint64_t)den + 1)); rb = ra ? ra - 1 : 0; break;              /* neighbours */
            case 2: ra = den - (uint32_t)(rnd() % (den < 4 ? den : 4)); rb = den - (uint32_t)(rnd() % (den < 4 ? den : 4)); break;   /* near full coverage */
            default: ra = (den >> 12) + (uint32_t)(rnd() % 3); rb = (den >> 12) + (uint32_t)(rnd() % 3); if (ra > den) ra = den; if (rb > den) rb = den; break;   /* around den / 4096 */
        }
        if (den < (1u << 23)) {
            const bool fa = exact_cov(ra, den) > exact_cov(rb, den);
            if (fa != (ra > rb)) bad++;
        }
        for (float thr : thr_fixed) {
            if ((itx_cov_thr(ra, den, thr) < thr) != (exact_cov(ra, den) < thr)) bad++;
        }
        union { uint32_t u; float f; } t; t.u = (uint32_t)rnd() & 0x7fffffffu;               /* any non-negative float, NaN and inf included */
        if ((itx_cov_thr(ra, den, t.f) < t.f) != (exact_cov(ra, den) < t.f)) bad++;
        if (itx_cov(100u, 100u + den, 100 + (int32_t)(den - ra), 100 + (int32_t)den) != exact_cov(ra, den) && den < (1u << 30)) bad++;   /* itx_cov is getCov */
    }
    return bad;
}

int32_t emu_query(emu_index *E, const char *chrom, uint32_t start, uint32_t end, float min_cov, int32_t *n_hits) {
    int32_t c = itx_strtab_find(&E->ix.chroms, chrom); if (n_hits) *n_hits = 0;
    if (c < 0) return -1;
    int32_t nh; float tcov; itx_iv e; e.row = 0; long long sel = itx_find_select(E->D, c, start, end, min_cov, &nh, &tcov, &e);
    if (n_hits) *n_hits = nh;
    if (sel >= 0 && tcov < min_cov) sel = -1;
    return sel >= 0 ? (int32_t)e.row : -1;
}

/* CpG rows in file order (the kernel k_cpg, sequentially) */
int emu_scan_cpg(emu_index *E, const char *bedgraph, int filter, uint32_t *n_lines, uint32_t *n_in_repeat, char *err) {
    itx_index &ix = E->ix; itx_dev_index &D = E->D;
    FILE *f = fopen(bedgraph, "r"); if (!f) { snprintf(err, ITX_ERRLEN, "Couldn't open %s", bedgraph); return ITX_EIO; }
    char *line = NULL; size_t lc = 0; uint32_t lines = 0, inrep = 0;
    while (getline(&line, &lc, f) >= 0) {
        char *s = line; while (*s == ' ' || (*s >= 9 && *s <= 13)) s++;
        if (*s == 0 || *s == '#') continue;
        char *w[20]; int nw = 0; char *q = s;
        while (nw < 20) { while (*q == ' ' || (*q >= 9 && *q <= 13)) q++; if (!*q) break; w[nw++] = q; while (*q && !(*q == ' ' || (*q >= 9 && *q <= 13))) q++; if (!*q) break; *q++ = 0; }
        if (nw < 4) { snprintf(err, ITX_ERRLEN, "file %s doesn't appear to be in bedGraph format. At least 4 fields required, got %d", bedgraph, nw); free(line); fclose(f); return ITX_EFORMAT; }
        lines++;
        int32_t c = itx_strtab_find(&ix.chroms, w[0]);
        uint32_t st = (uint32_t)strtol(w[1], NULL, 0), en = (uint32_t)strtol(w[2], NULL, 0); double sc = strtod(w[3], NULL);
        if (c < 0) continue;
        itx_iv e; e.start = e.end = 0; e.pmax = 0; e.row = 0;
        long long sel = itx_find_head(D, c, st, en, &e);
        if (sel < 0) continue;
        inrep++;
        if (filter) { D.el_cpg[sel]++; D.el_cpg_score[sel] += sc; continue; }
        if (!D.stat_mode) continue;
        const itx_meta mt = D.meta[sel]; const itx_meta2 m2 = D.meta2[sel];
        const uint32_t gs = mt.sub, gf = (uint32_t)(D.n_sub + m2.fam), gc = (uint32_t)(D.n_sub + D.n_fam + m2.cla);
        D.grp_cpg[gs]++; D.grp_cpg_score[gs] += sc; D.grp_cpg[gf]++; D.grp_cpg_score[gf] += sc; D.grp_cpg[gc]++; D.grp_cpg_score[gc] += sc;
        const uint32_t L = D.sub_len[mt.sub]; uint32_t ja, jb;
        if (L && itx_cov_range(st, 2u, e.start, e.end, mt.cons_start, mt.cons_end, L, &ja, &jb)) {
            const unsigned long long off = D.sub_bp_off[mt.sub];
            for (uint32_t j = ja; j < jb; j++) D.bp_cpg[off + j] += sc;
        }
    }
    free(line); fclose(f);
    if (n_lines) *n_lines = lines;
    if (n_in_repeat) *n_in_repeat = inrep;
    return ITX_OK;
}

/* the device inflater (itx_inflate.cuh) on one raw-deflate stream, with plain arrays as its table stores */
struct emu_tab {
    uint16_t *cells, *luts;
    uint16_t operator()(uint32_t j) const { return cells[j]; }
    void set(uint32_t j, uint16_t v) const { cells[j] = v; }
    uint16_t lut(uint32_t j) const { return luts[j]; }
    void lut_set(uint32_t j, uint16_t v) const { luts[j] = v; }
};
/* defer = 0: matches copied in line.  defer = 1: the two-pass mode of the device -- matches listed by the decoder,
 * then resolved in batches of 32 list entries exactly as the lanes of k_lz_resolve do (an entry goes once its
 * source ends before the first unfinished entry's output; entries of one round never depend on each other).  defer = 2: the
 * pointer jumping of k_lz_jump.  defer = 3..8: itx_lzw_resolve's windows of 8192 / 2048 / 256 / 6144 / 3072 / 1536 bytes. */
int emu_inflate(const uint8_t *in, uint32_t in_len, uint8_t *out, uint32_t out_cap, uint32_t expect, uint32_t *produced, int defer) {
    uint16_t cells[ITX_T_CELLS], luts[ITX_LUT_CELLS]; memset(cells, 0, sizeof cells); memset(luts, 0, sizeof luts);
    /* the decoder reads whole aligned words, a few of them past the end: give the stream an odd alignment and slack */
    std::vector<uint8_t> padded(in_len + 64, 0);
    const uint32_t skew = in_len % 4;
    if (in_len) memcpy(padded.data() + 4 + skew, in, in_len);
    const uint32_t cap = 21848;
    std::vector<uint32_t> mpl(defer ? cap : 1); std::vector<uint16_t> md(defer ? cap : 1);
    itx_inflater<emu_tab> I;
    I.tab.cells = cells; I.tab.luts = luts; I.out = out; I.out_cap = out_cap; I.err = 0;
    I.m_cap = defer ? cap : 0; I.m_pl = mpl.data(); I.m_d = md.data();
    const uint32_t rc = I.run(padded.data() + 4 + skew, in_len, expect);
    if (produced) *produced = I.out_pos;
    if (I.state == ITX_ST_OVERFLOW) return 99;
    if (defer >= 3 && rc == ITX_INF_OK) {
        /* itx_lzw_resolve (k_inflate's own second pass), lane by lane: windows of W bytes, the same per-lane pieces as the device */
        /* defer 6..8: the windows k_inflate runs at 32 / 16 / 8 blocks per warp (ITX_LZW_W5 / W4 / W3) */
        static const uint32_t Ws[6] = {8192u, 2048u, 256u, 6144u, 3072u, 1536u};
        const uint32_t W = Ws[(defer - 3) % 6], n = I.n_match, isize = I.out_pos;       /* multiples of 256 (itx_lzw_init) */
        std::vector<uint16_t> src(W);
        uint32_t k0 = 0;
        for (uint32_t w0 = 0; w0 < isize && k0 < n; w0 += W) {
            const uint32_t w1 = w0 + W < isize ? w0 + W : isize, cnt = w1 - w0;
            if ((mpl[k0] & 0xffffu) >= w1) continue;
            for (uint32_t l = 0; l < 32; l++) itx_lzw_init(src.data(), w0, cnt, l);
            for (uint32_t k = k0;; k += 32) {
                uint32_t c = 0;
                for (int l = 31; l >= 0; l--) {                    /* any lane order: the matches of a list do not overlap */
                    const bool in = k + (uint32_t)l < n;
                    const uint32_t e = in ? mpl[k + l] : 0xffffu, pos = e & 0xffffu, len = e >> 16;
                    if (in && pos < w1) itx_lzw_scatter(src.data(), w0, w1, pos, len, md[k + l]);
                    if (in && pos + len <= w1) c++;
                }
                k0 = k + c;
                if (c < 32) break;
            }
            for (bool any = true; any;) { any = false; for (int l = 31; l >= 0; l--) if (itx_lzw_jump(src.data(), w0, cnt, (uint32_t)l)) any = true; }
            for (uint32_t i = 0; i < cnt; i++) if (src[i] != (uint16_t)(w0 + i)) out[w0 + i] = out[src[i]];
        }
    } else if (defer == 2 && rc == ITX_INF_OK) {
        /* k_lz_jump: src[i] = where byte i comes from, pointer jumping until every byte points at a literal, then one gather */
        const uint32_t n = I.n_match, isize = I.out_pos;
        std::vector<uint16_t> src(65536 + 2);
        for (uint32_t i = 0; i < isize; i++) src[i] = (uint16_t)i;
        for (uint32_t k = 0; k < n; k++) { const uint32_t pos = mpl[k] & 0xffffu, len = mpl[k] >> 16, d = md[k]; for (uint32_t j = 0; j < len; j++) src[pos + j] = (uint16_t)(pos + j - d); }
        for (bool changed = true; changed;) {
            changed = false;
            for (uint32_t i = isize; i-- > 0;) {               /* any order gives the same fixed point; backwards is the least favourable for an in-place sweep */
                const uint32_t sidx = src[i];
                if (sidx != i) { const uint32_t ss = src[sidx]; if (ss != sidx) { src[i] = (uint16_t)ss; changed = true; } }
            }
        }
        for (uint32_t i = 0; i < isize && i < out_cap; i++) if (src[i] != i) out[i] = out[src[i]];
    } else if (defer && rc == ITX_INF_OK) {
        const uint32_t n = I.n_match;
        for (uint32_t k0 = 0; k0 < n; k0 += 32) {
            uint32_t undone = 0;
            for (uint32_t l = 0; l < 32 && k0 + l < n; l++) undone |= 1u << l;
            while (undone) {
                const uint32_t m = (uint32_t)__builtin_ctz(undone);
                const uint32_t pm = mpl[k0 + m] & 0xffffu;
                uint32_t go = 0;
                for (uint32_t l = 0; l < 32; l++) if ((undone >> l) & 1u) {
                    const uint32_t e = mpl[k0 + l];
                    if (itx_lz_ready(e & 0xffffu, e >> 16, md[k0 + l] ? md[k0 + l] : 65536u, l == m, pm)) go |= 1u << l;
                }
                /* in reverse lane order: if two entries of a round depended on each other the result would be wrong */
                for (int l = 31; l >= 0; l--) if ((go >> l) & 1u) { const uint32_t e = mpl[k0 + l]; itx_lz_copy<false>(out + (e & 0xffffu), e >> 16, md[k0 + l]); }
                undone &= ~go;
            }
        }
    }
    return (int)rc;
}

/* itx_strtod_fast on a C string: returns the value, *exact = 0 where the device leaves the line to the host */
double emu_strtod(const char *str, int *exact) {
    const size_t n = strlen(str);
    std::vector<uint8_t> buf(n + 64, 0); memcpy(buf.data(), str, n);
    bool ex = false;
    const double v = itx_strtod_fast(itx_src_global{buf.data()}, 0, n, &ex);
    *exact = ex ? 1 : 0;
    return v;
}
}
