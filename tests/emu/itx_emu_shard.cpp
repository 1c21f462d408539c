/* itx_emu_shard.cpp -- TEST-ONLY: -R across ranks on the host emulation of the device logic (tests/emu/itx_emu.cpp, included
 * whole), for tests/test_emu_shard_rmdup.py, which builds it.  What itx_shard_dedup_keys / itx_shard_dedup_fetch / itx_dedup_admit
 * do on the device:
 *   phase 1: the part scanned with -R on a scratch index whose key state starts empty -- its key map then holds exactly the keys of
 *            the part's unique fragments, and its two minima say whether the part held a unique / some other fragment;
 *   admission: other parts' keys entered into a rank's key map with ONE freshly reserved ordinal, the flags lowering its minima.
 * Phase 2 is emu_scan_shard with -R on the rank's own index. */
#include "itx_emu.cpp"

extern "C" {

/* phase 1 of one part on the scratch index S (reset first): the chain report as emu_scan_shard gives it, the number of keys, the flags
 * (bit 0: a unique fragment, bit 1: some other fragment).  A part whose chain found no record start or ended in a cut record
 * (forced entry NONE / END) exports nothing. */
int emu_part_dedup_keys(emu_index *S, const uint8_t *hdr_bam, uint64_t hdr_bytes, const uint8_t *bam, uint64_t len, uint64_t own, uint64_t carry0,
                        const itx_scan_opts *so, uint32_t chunk, uint64_t *entry_rel, uint64_t *exit_rel, uint64_t *n_keys, uint32_t *flags, char *err) {
    emu_reset(S);
    itx_scan_opts o = *so; o.rmDup = 1;
    uint64_t cnt[13];
    const int rc = emu_scan_shard(S, hdr_bam, hdr_bytes, bam, len, own, carry0, &o, chunk, cnt, entry_rel, exit_rel, err);
    if (rc) return rc;
    if (carry0 != ~0ull && *entry_rel >= ITX_OFF_GUESS) { emu_reset(S); *n_keys = 0; *flags = 0; return ITX_OK; }
    *n_keys = S->dup_first.size();
    *flags = (S->dup_min_unique != ~0ull ? 1u : 0u) | (S->dup_min_other != ~0ull ? 2u : 0u);
    return ITX_OK;
}
/* the keys phase 1 left in S, as (lo, hi) pairs */
uint64_t emu_part_dedup_fetch(emu_index *S, unsigned long long *dst, uint64_t cap) {
    uint64_t n = 0;
    for (auto it = S->dup_first.begin(); it != S->dup_first.end() && n < cap; ++it, n++) { dst[2 * n] = it->first.first; dst[2 * n + 1] = it->first.second; }
    return n;
}
void emu_dedup_admit(emu_index *E, const unsigned long long *keys, uint64_t n, uint32_t flags) {
    const unsigned long long ord = E->dup_ord_base++;
    for (uint64_t i = 0; i < n; i++) {
        auto it = E->dup_first.insert(std::make_pair(std::make_pair(keys[2 * i], keys[2 * i + 1]), ord)).first;
        if (ord < it->second) it->second = ord;
    }
    if ((flags & 1u) && ord < E->dup_min_unique) E->dup_min_unique = ord;
    if ((flags & 2u) && ord < E->dup_min_other) E->dup_min_other = ord;
}

}
