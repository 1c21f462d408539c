"""The device logic (host emulation) against the oracle on generated inputs of the benchmark shapes,
scaled down: every counter, table and coverage vector bit-exact, and the per-record trace (fragment,
selected rmsk row, flags) identical record by record.  Also the oracle against the reference's stored outputs
for generated BAMs (tests/golden/synthetic/), and against the reference binary itself where it is built."""
import filecmp
import os

import numpy as np
import pytest

import emu_lib
import oracle_lib as O
import synth
import synthetic_golden as SG
from iteres_b200 import capi

CASES = [
    # name, shape, n_rmsk, mode, n_units, opts
    ("se50_chr1", 0, 20000, 0, 30000, {}),
    ("se50_hg19_E0", 1, 60000, 0, 40000, dict(extension=0)),
    ("se75_xa_hg19", 1, 60000, 1, 40000, {}),
    ("se75_xa_nodiff", 1, 60000, 1, 20000, dict(diffSubfam=0)),
    ("pe100_hg19", 1, 60000, 2, 20000, {}),
    ("pe100_treat", 1, 60000, 2, 20000, dict(treat=1)),
    ("pe100_D_I300", 1, 60000, 2, 20000, dict(discardWrongEnd=1, iSize=300)),
    ("se50_Q30_c05", 0, 20000, 0, 20000, dict(mapQ=30, minCoverage=0.5)),
    ("se50_chrM_R", 2, 3000, 0, 60000, dict(rmDup=1)),
    ("pe100_R", 1, 60000, 2, 20000, dict(rmDup=1)),
]


@pytest.fixture(scope="module")
def worlds(tmp_path_factory):
    made = {}

    def get(shape, n_rmsk):
        if (shape, n_rmsk) not in made:
            d = str(tmp_path_factory.mktemp("synth%d" % shape))
            s = synth.Synth(shape, n_rmsk, seed=7)
            made[(shape, n_rmsk)] = (s, s.write_tables(d), d)
        return made[(shape, n_rmsk)]
    yield get
    for s, _, _ in made.values():
        s.close()


def tables_equal(a, b):
    for which in range(3):
        assert a.table(which) == b.table(which)


def assert_group_tables_and_coverage(emu, ora):
    """subfamily / family / class rows (names in Kent hash order, read counts, unique counts, lengths, genome counts) and
    the per-base coverage vectors, all and unique"""
    import ctypes as C
    L = O.lib()
    c4 = (C.c_uint64 * 4)()
    for which, nfun in ((0, L.ora_n_subfam), (1, L.ora_n_fam), (2, L.ora_n_class)):
        got = emu.table(which)
        assert len(got) == nfun(ora.h)
        for i, row in enumerate(got):
            L.ora_counts(ora.h, which, i, c4)
            assert row == (L.ora_name(ora.h, which, i).decode(),) + tuple(c4)
    for i in range(L.ora_n_subfam(ora.h)):
        ln = L.ora_subfam_length(ora.h, i)
        if ln:
            for u in (0, 1):
                want = np.ctypeslib.as_array(L.ora_subfam_bp(ora.h, i, u), shape=(ln,))
                assert np.array_equal(emu.coverage(i, u), want)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_emu_matches_oracle(case, worlds):
    name, shape, n_rmsk, mode, n_units, kw = case
    s, (cs, rs, rm), _ = worlds(shape, n_rmsk)
    buf, n, nrec = s.stream(mode, n_units)
    raw = buf[:n].tobytes()
    ora = O.OracleIndex(cs, rs, rm)
    cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(**kw), trace=True)
    emu = emu_lib.EmuIndex(cs, rs, rm, chunk=4096)
    fast0 = emu.xa_fast()
    cnt_e, tr_e = emu.scan_stream(raw, capi.default_opts(**kw), trace=True)
    assert cnt_e == cnt_o
    assert cnt_o[0] + cnt_o[1] == nrec and cnt_o[9] > 0
    checked, mism = emu.ring_check()
    assert checked >= nrec and mism == 0          # ring addressing decodes every record identically
    tc, tm, te = emu.tile_check()
    assert tc > 0 and tm == 0 and te == emu.n_bad()   # the span kernels' chain (staged guess, run-predicted walk) == the sequential chain
    assert len(tr_e) == len(tr_o) == nrec
    for f in ("start", "end", "tid", "sel_row"):
        assert np.array_equal(tr_e[f], tr_o[f]), f
    mask = ~np.uint32(8 | 64)               # HAS_XA is reported by the oracle even where it is not evaluated; DUP is the product's own flag
    assert np.array_equal(tr_e["flags"] & mask, tr_o["flags"] & mask)
    if kw.get("diffSubfam", 1) and mode == 1:
        assert cnt_o[12] > 0
        f0, g0 = fast0
        checked, differed = emu.xa_check()              # the lane-per-alternate walk of k_scan against the one-lane walk
        assert checked > 0 and differed == 0
        f1, g1 = emu.xa_fast()                          # ... whose pieces k_xa reads in registers when they have the usual shape: these do
        assert f1 - f0 > 0 and f1 - f0 > 20 * (g1 - g0)
    assert_group_tables_and_coverage(emu, ora)
    ora.close()
    emu.close()


@pytest.mark.parametrize("chunk", [64, 448, 8192, 1 << 20])
def test_chunk_size_never_changes_the_answer(chunk, worlds):
    """Speculated chunk entries only cost time: any chunk size (even smaller than a record) gives the chain."""
    s, (cs, rs, rm), _ = worlds(1, 60000)
    buf, n, nrec = s.stream(1, 5000)
    raw = buf[:n].tobytes()
    ref = emu_lib.EmuIndex(cs, rs, rm, chunk=4096)
    want = ref.scan_stream(raw, capi.default_opts())
    emu = emu_lib.EmuIndex(cs, rs, rm, chunk=chunk)
    assert emu.scan_stream(raw, capi.default_opts()) == want
    # chunks smaller than a record: most spans hold no record start at all; the chain rule takes them as they stand
    # (itx_span_consistent: the chain runs over them), which is what keeps long-read BAMs off the repair path
    assert emu.table(0) == ref.table(0)
    ref.close()
    emu.close()


def test_truncated_stream_stops_like_the_reference(worlds):
    """bam_read1 fails on a cut record and the reference's loop ends silently (generic.c:745)."""
    s, (cs, rs, rm), _ = worlds(0, 20000)
    buf, n, nrec = s.stream(0, 3000)
    for cut in (n - 1, n - 40, n - 131, n // 2 + 3):
        raw = buf[:cut].tobytes()
        ora = O.OracleIndex(cs, rs, rm)
        emu = emu_lib.EmuIndex(cs, rs, rm, chunk=512)
        assert emu.scan_stream(raw, capi.default_opts()) == ora.scan_stream(raw, O.default_opts())
        ora.close()
        emu.close()


@pytest.mark.skipif(not os.path.exists(SG.MANIFEST), reason="no stored outputs of the reference under tests/golden/synthetic")
@pytest.mark.parametrize("mode,n_units,args", SG.STAT_CASES)
def test_reference_binary_matches_oracle_on_synthetic_bam(mode, n_units, args, worlds, tmp_path):
    """Pins the oracle (and with it everything compared to the oracle) to the UNMODIFIED reference on
    inputs far larger than the known-answer files: the oracle's files against the reference's as stored under
    tests/golden/synthetic/, and against the reference binary itself where it has been built."""
    s, tables, _ = worlds(*SG.STAT_WORLD[:2])
    bam = str(tmp_path / "reads.bam")
    SG.write_bam(s, bam, mode, n_units)
    rd, od = tmp_path / "ref", tmp_path / "ora"
    rd.mkdir(); od.mkdir()
    SG.oracle_stat(tables, bam, args, str(od))
    SG.check_stat(SG.stat_case(mode, n_units, args), str(od))
    if os.path.exists(O.REF_BIN):
        SG.reference_stat(tables, bam, args, str(rd))
        for fn in SG.STAT_TEXT + SG.STAT_WIG:
            assert filecmp.cmp(str(rd / fn), str(od / fn), shallow=False), fn


@pytest.mark.parametrize("chunk", [4096, 32768])
def test_records_of_every_size(chunk, tmp_path):
    """records from 60 bytes to 70 KB (longer than a chunk and than the decode ring): same counters and trace"""
    import mixed_records
    tabs = mixed_records.tables(str(tmp_path))
    raw, nrec = mixed_records.make()
    for kw in ({}, dict(extension=0, treat=1)):
        ora = O.OracleIndex(*tabs)
        cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(**kw), trace=True)
        emu = emu_lib.EmuIndex(*tabs, chunk=chunk)
        cnt_e, tr_e = emu.scan_stream(raw, capi.default_opts(**kw), trace=True)
        assert cnt_e == cnt_o and cnt_o[9] > 0 and cnt_o[0] + cnt_o[1] == nrec
        for f in ("start", "end", "tid", "sel_row"):
            assert np.array_equal(tr_e[f], tr_o[f]), f
        assert np.array_equal(tr_e["flags"] & ~np.uint32(8), tr_o["flags"] & ~np.uint32(8))
        assert emu.ring_check()[1] == 0
        tc, tm, te = emu.tile_check()
        assert tc > 0 and tm == 0                 # entry misses (te) are allowed here: records longer than a chunk
        ora.close()
        emu.close()


def _nested_world(d):
    """a hand-made chromosome: stacks of 2..7 nested / staggered elements (hit lists longer than the two kept in
    registers), elements that straddle 128 kb and 1 Mb bin edges, and long fragments that touch an element by a few bases"""
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chrN\t4000000\n")
    rng = np.random.default_rng(11)
    rows, subs = [], ["S%d" % i for i in range(12)]
    open(rs, "w").write("".join("%s\t%d\n" % (s, 3000) for s in subs))
    pos = 5000
    while pos < 3900000:
        depth = int(rng.integers(1, 8))
        a, b = pos, pos + int(rng.integers(200, 4000))
        for k in range(depth):
            rows.append((a, b))
            a += int(rng.integers(0, 60)); b -= int(rng.integers(-40, 60))
            if b <= a + 5:
                break
        pos = b + int(rng.integers(1, 30000))
    for k in range(1, 30):
        rows.append((k * 131072 - 40, k * 131072 + 70))
    rows.append((1048576 - 300, 1048576 + 300))
    rows.sort()
    with open(rm, "w") as f:
        for i, (a, b) in enumerate(rows):
            sub = subs[i % len(subs)]
            f.write("\t".join(["585", "1000", "0", "0", "0", "chrN", str(a), str(b), "-1", "+", sub, "CLS%d" % (i % 3), "FAM%d" % (i % 5),
                               "1", str(min(3000, b - a)), "0", str(i)]) + "\n")
    return cs, rs, rm, rows


def test_emu_query_matches_oracle_on_nested_table(tmp_path):
    """overlap + "last ascent" selection + minCoverage of the device logic against the oracle's binKeeper restatement:
    hit lists of every length (the long-list path included) and coverages on both sides of every threshold"""
    cs, rs, rm, rows = _nested_world(str(tmp_path))
    ora = O.OracleIndex(cs, rs, rm)
    emu = emu_lib.EmuIndex(cs, rs, rm)
    rng = np.random.default_rng(3)
    q = []
    for (a, b) in rows:
        for _ in range(6):
            st = max(0, a + int(rng.integers(-120, 120)))
            q.append((st, st + int(rng.integers(1, 300))))
        q.append((a, b)); q.append((a + 1, b - 1)); q.append((max(0, a - 1), b + 1))
        for ov in (1, 2, 3, 4, 5, 9):                 # a long fragment that touches the element by ov bases: coverage ov / length
            for length in (ov * 4095, ov * 4096, ov * 4097, ov * 8191, ov * 8192, ov * 8193, ov * 9999, ov * 10000, ov * 10001):
                st = b - ov
                q.append((st, st + length))
    for (a, b) in rows[-12:]:                         # fragments of 2^23 bases and more (float comparison of the coverages) over the last few stacks
        q += [(max(0, a - 3), a - 3 + 9000000), (a + 1, a + 1 + (1 << 23)), (b - 2, b - 2 + 20000000)]
    seen = set()
    for mc in (1e-4, 0.0, 2.0 ** -13, 0.00012, 0.5):
        for (st, en) in q:
            ws, hits = ora.find_select("chrN", st, en, mc)
            sel, nh = emu.query("chrN", st, en, mc)
            assert (sel, nh) == (ws, len(hits)), (st, en, mc)
            seen.add(min(nh, 5))
    assert seen >= {0, 1, 2, 3, 4, 5}
    ora.close()
    emu.close()


XA_ODD = [
    "chr1,+5101,36M,1;",                                  # plain: another subfamily at 5101 -> discarded
    "chr1,+5101,36M,1",                                   # no trailing separator
    "chr1,+5101,36M,2;",                                  # nm2 > NM: ignored
    "",                                                   # empty string: no pieces
    ";",                                                  # one empty piece
    ";;chr1,+5101,36M,1;;",                               # empty pieces around a real one
    "chr1,+5101,36M;",                                    # three fields: malformed, skipped
    "chr1,+5101;chr1,+5101,36M,1;",                       # malformed first, real second
    "chr1,+5101,36M,1,extra,more;",                       # the fourth field stops at the next comma
    "chr1,+5101,36M,;",                                   # empty fourth field: strtol("") = 0 <= NM
    "chr1,,36M,1;",                                       # empty position: 0
    ",+5101,36M,1;",                                      # empty chromosome name: unknown
    "chrQ,+5101,36M,1;chr1,-5101,36M,0;",                 # unknown chromosome, then a hit on the minus strand
    "chr1,0x13ed,36M,1;",                                 # strtol base 0: hexadecimal 5101
    "chr1,011755,36M,01;",                                # octal 5101, octal 1
    "chr1, +5101,36M, 1;",                                # leading white space is strtol's
    "chr1,+5101x,36M,1z;",                                # trailing garbage stops the parse
    "chr1,+1101,36M,0;",                                  # the same subfamily: kept
    "chr1,+99999999999,36M,1;",                           # overflow saturates, (int) keeps the low word
    "chr1,+5101,36M,1;" * 99 + "chr1,+1101,36M,0;",       # 100 pieces, the last one harmless... but an earlier one hits
    "chr1,+1101,36M,0;" * 100 + "chr1,+5101,36M,1;",      # the 101st piece is never looked at
    "chr1,+1101,36M,0;" * 99 + "chr1,+5101,36M,1;",       # the 100th is
]


def xa_odd_reads():
    """the reads of test_xa_strings_of_every_shape (shared with the device test of the same name)"""
    import kats
    reads = []
    for k, xa in enumerate(XA_ODD):
        for ty in ("Z", "H"):
            reads.append(kats.se("x%d%s" % (k, ty), 0, 1050, 0, aux=[("NM", "i", 1), ("XA", ty, xa)]))
    reads.append(kats.se("xi", 0, 1050, 0, aux=[("NM", "i", 1), ("XA", "i", 7)]))          # XA that is not a string
    reads.append(kats.se("xnm", 0, 1050, 0, aux=[("XA", "Z", "chr1,+5101,36M,0;")]))      # no NM: 0
    # k_xa parses the aux area out of a staged copy with 32-bit offsets: an aux area larger than its 6 KiB pool, byte arrays in front of
    # the tags, and an array count that leaves the aux area between XA and NM (NM is then not found: 0) take its fall-backs
    import struct
    big = b"C" + struct.pack("<i", 7000) + bytes(7000)          # (the reference copies the list into char[2000]: the LIST stays short)
    reads.append(kats.se("xbig_hit", 0, 1050, 0, aux=[("ZB", "B", big), ("NM", "i", 1), ("XA", "Z", "chr1,+1101,36M,0;chr1,+5101,36M,1;")]))
    reads.append(kats.se("xbig_keep", 0, 1050, 0, aux=[("NM", "i", 1), ("XA", "Z", "chr1,+1101,36M,0;"), ("ZB", "B", big)]))
    arr = b"C" + struct.pack("<i", 40) + bytes(range(40))
    reads.append(kats.se("xarr", 0, 1050, 0, aux=[("ZB", "B", arr), ("NM", "i", 1), ("ZC", "B", b"s" + struct.pack("<i", 3) + bytes(6)), ("XA", "Z", "chr1,+5101,36M,1;")]))
    reads.append(kats.se("xarr_bad", 0, 1050, 0, aux=[("XA", "Z", "chr1,+5101,36M,0;"), ("ZB", "B", b"I" + struct.pack("<I", 0x40000000)), ("NM", "i", 1)]))
    reads.append(kats.se("xarr_bad2", 0, 1050, 0, aux=[("XA", "Z", "chr1,+5101,36M,1;"), ("ZB", "B", b"I" + struct.pack("<I", 0x40000000)), ("NM", "i", 1)]))
    return reads


def test_xa_strings_of_every_shape(tmp_path):
    """mapped2diffSubfam (generic.c:303-341) on alternate lists that chopByChar / strtol treat in their own ways: the
    device logic's single pass over the string against the oracle, read by read"""
    import bamio
    import kats
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    open(rm, "w").write("\n".join(kats.ANNOT1) + "\n")
    reads = xa_odd_reads()
    # (here only: array counts that are negative or of an unknown subtype -- the tag walk then steps backwards or into the count's own
    # bytes, as bam_aux_get does; k_xa's 32-bit walk hands such a read to the 64-bit one)
    import struct
    reads.append(kats.se("neg_small", 0, 1050, 0, aux=[("XA", "Z", "chr1,+5101,36M,1;"), ("ZB", "B", b"C" + struct.pack("<i", -3) + b"NMC\x01xx"), ("NM", "i", 1)]))
    reads.append(kats.se("neg_back", 0, 1050, 0, aux=[("NM", "i", 1), ("ZB", "B", b"I" + struct.pack("<i", -4)), ("XA", "Z", "chr1,+5101,36M,1;")]))
    reads.append(kats.se("neg_back2", 0, 1050, 0, aux=[("XA", "Z", "chr1,+5101,36M,1;"), ("ZB", "B", b"I" + struct.pack("<i", -4)), ("NM", "i", 1)]))
    reads.append(kats.se("zero_sub", 0, 1050, 0, aux=[("ZB", "B", b"?" + struct.pack("<i", 7)), ("NM", "i", 1), ("XA", "Z", "chr1,+5101,36M,1;")]))
    raw = bamio.encode_header([("chr1", 1000000)]) + b"".join(bamio.encode_record(r) for r in reads)
    ora = O.OracleIndex(cs, rs, rm)
    cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(), trace=True)
    for chunk in (256, 4096):
        emu = emu_lib.EmuIndex(cs, rs, rm, chunk=chunk)
        cnt_e, tr_e = emu.scan_stream(raw, capi.default_opts(), trace=True)
        assert cnt_e == cnt_o
        mask = ~np.uint32(8 | 64)
        bad = np.nonzero((tr_e["flags"] & mask) != (tr_o["flags"] & mask))[0]
        assert len(bad) == 0, [reads[i]["qname"] for i in bad]
        # k_scan walks the alternates one LANE per alternate (itx_xa_count / itx_xa_kth / itx_xa_piece, first yes wins, malformed
        # ones before it counted): the same verdicts and the same malformed count as the one-lane walk, read by read
        checked, differed = emu.xa_check()
        assert checked > 0 and differed == 0
        fast, general = emu.xa_fast()
        assert fast > 0 and general > 0                 # the register path and the general parser both met these lists
        emu.close()
    assert 0 < cnt_o[12] < len(reads)
    ora.close()


def test_register_parser_of_an_alternate_agrees_with_the_general_one(tmp_path):
    """k_xa reads an alternate of the usual shape in registers (itx_xa_piece_fast) and hands anything else to the general parser
    (itx_xa_piece: strtol(.., 0, 0), chopByChar): on generated pieces -- names of the table, near misses, long and empty names,
    numbers with signs, leading zeros, hexadecimal, white space, too many digits, any number of commas, every alignment -- the two
    give the same verdict, the same malformed flag and ask the interval table the same question (chromosome, start, end), and both
    paths are taken"""
    d = str(tmp_path)
    s = synth.Synth(1, 20000, seed=11)
    cs, rs, rm = s.write_tables(d)
    emu = emu_lib.EmuIndex(cs, rs, rm, chunk=4096)
    f0, g0 = emu.xa_fast()
    for seed in range(1, 9):
        assert emu.xa_fuzz(seed, 250_000) == 0
    f1, g1 = emu.xa_fast()
    assert f1 - f0 > 200_000 and g1 - g0 > 200_000
    emu.close()
    s.close()


def test_coverage_shortcuts_are_the_float_arithmetic():
    """itx_select_walk compares overlaps as integers (fragments shorter than 2^23 bases) and forms the coverage quotient
    only when it can fall below the threshold: both rules against the float arithmetic of getCov, on two million cases
    that include the edges the proofs in itx_logic.cuh lean on"""
    assert emu_lib.lib().emu_check_cov_rules(2_000_000, 12345) == 0


def _adversarial_records(rng, n, n_ref):
    """records whose fields sit on the edges the fragment logic branches on (generic.c:748-905): positions at 0, at and
    past the chromosome end, negative; reference ids at and past n_ref; isize 0, +-iSize, +-(iSize+1), INT_MIN-ish;
    every flag combination; CIGARs with and without reference-consuming ops; no CIGAR; reads longer than the chromosome"""
    import kats
    recs = []
    sizes = {0: 1000000, 1: 16571}
    for i in range(n):
        tid = int(rng.choice([0, 0, 0, 1, 1, 2, n_ref, n_ref + 3, -1, -2]))
        size = sizes.get(tid, 5000)
        pos = int(rng.choice([0, 1, 35, 36, 1000, 1050, 1299, 1300, 5000, 5880, 5999, 6099, size - 37, size - 36, size - 1, size, size + 100,
                              -1, 2 ** 31 - 40, int(rng.integers(0, 7000))]))
        flag = int(rng.choice([0, 16, 4, 1, 1 | 64, 1 | 128, 1 | 64 | 8, 1 | 128 | 8, 99, 147, 83, 163, 73, 133, 69, 137, 1 | 2 | 64 | 16 | 32, 1024, 256 | 16, 2048,
                               int(rng.integers(0, 4096))]))
        L = int(rng.choice([1, 20, 36, 50, 100, 400]))
        cigar = str(rng.choice(["%dM" % L, "*", "5S%dM" % max(1, L - 5), "10M5D%dM" % max(1, L - 10), "10M200N%dM" % max(1, L - 10), "%d=" % L, "3I%dX" % max(1, L - 3),
                                "1M" * 0 + "%dM2D3N4M" % L, "20000M"]))
        isize = int(rng.choice([0, 1, -1, 36, 200, -200, 499, 500, 501, -499, -500, -501, 100000, -100000, 2 ** 31 - 1, -(2 ** 31)]))
        mpos = int(rng.choice([0, pos, max(0, pos - 300), pos + 300 if pos < 2 ** 31 - 400 else pos, size - 10, size + 50, -1]))
        mtid = int(rng.choice([tid, tid, 0, -1, 1]))
        aux = [("NM", "C", int(rng.integers(0, 3)))]
        if rng.random() < 0.3:
            aux.append(("XA", "Z", str(rng.choice(["chr1,+5101,36M,1;", "chr1,-1101,36M,0;", "chrM,+200,36M,2;chr1,+5950,36M,0;", "chr9,+5,36M,0;"]))))
        recs.append(dict(qname="a%d" % i, flag=flag, tid=tid, pos=pos, mapq=int(rng.choice([0, 9, 10, 11, 29, 30, 31, 60, 255])), cigar=cigar,
                         mtid=mtid, mpos=mpos, isize=isize, seq="A" * L, qual="I" * L, aux=aux))
    return recs


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_adversarial_records_match_oracle(seed, tmp_path):
    """fragment logic, bam_calend, clamping, strand / extension arithmetic with unsigned wrap-around, -C renaming, the unknown-
    chromosome path and the counters, on records built to sit on every branch -- the device logic against the oracle, record
    by record, under several option sets"""
    import bamio
    import kats
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\nchrM\t16571\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    rows = kats.ANNOT1 + [kats.rmsk_row("chrM", 100, 400, "+", "AluY", "SINE", "Alu", 1, 300, 0),
                          kats.rmsk_row("chr1", 999900, 1000000, "-", "L1PA2", "LINE", "L1", -100, 5900, 5800),
                          kats.rmsk_row("chr1", 0, 40, "+", "MIR", "SINE", "MIR", 1, 41, 0)]
    open(rm, "w").write("\n".join(rows) + "\n")
    rng = np.random.default_rng(seed)
    refs = [("chr1", 1000000), ("chrM", 16571), ("chrUn_x", 5000)]
    reads = _adversarial_records(rng, 1500, len(refs))
    import struct

    def enc(r):                                   # the bin field is not on the path: encode with a tame position, then put the real one in
        b = bytearray(bamio.encode_record(dict(r, pos=min(max(r["pos"], 0), 1 << 28))))
        b[8:12] = struct.pack("<i", r["pos"])
        return bytes(b)
    raw = bamio.encode_header(refs) + b"".join(enc(r) for r in reads)
    option_sets = [dict(), dict(extension=0), dict(extension=1000), dict(treat=1), dict(discardWrongEnd=1, iSize=200), dict(iSize=0),
                   dict(mapQ=30, minCoverage=0.5), dict(mapQ=0, minCoverage=0.0), dict(diffSubfam=0, extension=36), dict(filter=1), dict(addChr=1)]
    for kw in option_sets:
        ora = O.OracleIndex(cs, rs, rm)
        cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(**kw), trace=True)
        emu = emu_lib.EmuIndex(cs, rs, rm, chunk=4096)
        cnt_e, tr_e = emu.scan_stream(raw, capi.default_opts(**kw), trace=True)
        assert cnt_e == cnt_o, kw
        assert cnt_o[6] > 200 and cnt_o[9] > 20 and cnt_o[4] + cnt_o[5] < cnt_o[2] + cnt_o[3] < len(reads), cnt_o     # every stage of the funnel drops some
        assert len(tr_e) == len(tr_o) == len(reads)
        for f in ("start", "end", "tid", "sel_row"):
            bad = np.nonzero(tr_e[f] != tr_o[f])[0]
            assert len(bad) == 0, (kw, f, [reads[i] for i in bad[:3]])
        mask = ~np.uint32(8 | 64)
        bad = np.nonzero((tr_e["flags"] & mask) != (tr_o["flags"] & mask))[0]
        assert len(bad) == 0, (kw, [reads[i] for i in bad[:3]])
        if not kw.get("filter"):
            assert_group_tables_and_coverage(emu, ora)
        ora.close()
        emu.close()


def decoy_stream():
    """records that carry, inside a byte-array aux field, back-to-back copies of a perfectly valid record: a span that begins
    inside such a field GUESSES one of the copies as its first record (the copies pass every structural test, next record
    included), so the chain check must catch it and the span must be walked again from where the previous one really ended"""
    import struct
    import bamio
    import kats
    small = bamio.encode_record(kats.se("decoy", 0, 5100, 37))
    payload = small * 90                                   # ~ 9 KB: longer than two 4 KiB spans
    carrier_aux = [("NM", "C", 0), ("ZB", "B", b"C" + struct.pack("<i", len(payload)) + payload)]
    reads = []
    for k in range(12):
        reads.append(kats.se("carrier%d" % k, 0, 1050 + k, 37, aux=carrier_aux))
        for j in range(25):
            reads.append(kats.se("r%d_%d" % (k, j), 16 if j % 2 else 0, 1000 + 7 * j, 30 + j % 3, aux=[("NM", "C", 1)]))
    raw = bamio.encode_header([("chr1", 1000000)]) + b"".join(bamio.encode_record(r) for r in reads)
    return raw, len(reads)


def test_wrong_span_guesses_are_caught_and_repaired(tmp_path):
    import kats
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    open(rm, "w").write("\n".join(kats.ANNOT1) + "\n")
    raw, nrec = decoy_stream()
    ora = O.OracleIndex(cs, rs, rm)
    cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(), trace=True)
    assert cnt_o[0] == nrec and cnt_o[9] > 0
    for chunk in (4096, 8192):
        emu = emu_lib.EmuIndex(cs, rs, rm, chunk=chunk)
        cnt_e, tr_e = emu.scan_stream(raw, capi.default_opts(), trace=True)
        assert emu.n_bad() > 0                                  # decoys were taken for record starts ...
        assert cnt_e == cnt_o                                   # ... and it made no difference
        for f in ("start", "end", "tid", "sel_row"):
            assert np.array_equal(tr_e[f], tr_o[f]), f
        tc, tm, te = emu.tile_check()
        assert tc > 0 and tm == 0 and te > 0                    # the span kernels' guess falls for them too; their walks otherwise agree
        assert_group_tables_and_coverage(emu, ora)
        emu.close()
    ora.close()


def inconsistent_cigar_stream():
    """records whose n_cigar overstates what the record holds (a corrupt file -- or the garbage a wrongly guessed span walks): the
    CIGAR walk of bam_calend must stop at the record's own end.  The last record of the stream is one of them: an unclamped walk
    would read past the end of the buffer (the reference itself reads whatever follows in its malloc'ed block: undefined)."""
    import struct
    import bamio
    import kats
    good = [bamio.encode_record(kats.se("g%d" % j, 16 if j % 2 else 0, 1000 + 11 * j, 37, aux=[("NM", "C", 1)])) for j in range(40)]

    def broken(qname, flag, pos, n_cigar_claimed, n_cigar_present, l_seq=0):
        q = qname.encode() + b"\0"
        cig = b"".join(struct.pack("<I", (20 << 4) | 0) for _ in range(n_cigar_present))
        core = struct.pack("<iiIIiiii", 0, pos, (4680 << 16) | (37 << 8) | len(q), (flag << 16) | n_cigar_claimed, l_seq, -1, -1, 0)
        data = core + q + cig
        return struct.pack("<i", len(data)) + data
    recs = good[:20] + [broken("b1", 16, 1040, 9, 2), broken("b2", 0, 1060, 65535, 0), broken("b3", 16, 5100, 3, 3)] + good[20:] + [broken("last", 16, 1100, 60000, 1)]
    return bamio.encode_header([("chr1", 1000000)]) + b"".join(recs), len(recs)


def test_n_cigar_beyond_the_record_is_not_followed(tmp_path):
    import kats
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    open(rm, "w").write("\n".join(kats.ANNOT1) + "\n")
    raw, nrec = inconsistent_cigar_stream()
    for ext in (0, 150):                                        # -E 0: every read's end comes from the CIGAR; -E 150: only the minus strand's
        ora = O.OracleIndex(cs, rs, rm)
        cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(extension=ext), trace=True)
        assert cnt_o[0] == nrec and cnt_o[9] > 0
        emu = emu_lib.EmuIndex(cs, rs, rm, chunk=4096)
        cnt_e, tr_e = emu.scan_stream(raw, capi.default_opts(extension=ext), trace=True)
        assert cnt_e == cnt_o
        for f in ("start", "end", "tid", "sel_row"):
            assert np.array_equal(tr_e[f], tr_o[f]), f
        ora.close()
        emu.close()
