"""Parity of the CUDA path (through the C ABI of include/iteres_gpu.h) with the reference:
  * the reference's own outputs (tests/golden/, byte for byte) for every known-answer input,
  * the oracle on generated inputs of the benchmark shapes: all 13 counters, the subfamily / family /
    class tables, both coverage vectors and the per-record trace, bit-exact,
  * the bench's table density (5.5 M rows) and size-independent properties in tests/test_gpu_fullsize.py.
Integer results must be bit-exact; the only floating point on the path (CpG score sums, printed
%.4f) is compared at 1e-9 relative, the tolerance BASELINE.json states."""
import ctypes as C
import filecmp
import os

import numpy as np
import pytest

import kats
import oracle_lib as O
import runners
import synth
from iteres_b200 import capi

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = [(k, v) for k in kats.KATS for v in kats.KATS[k]["variants"]
         if not runners.needs_host_order(*kats.KATS[k]["variants"][v])]


@pytest.mark.parametrize("inflate", ["device", "host"])
@pytest.mark.parametrize("kat,variant", CASES)
def test_cuda_path_matches_reference_output(kat, variant, inflate, tmp_path, monkeypatch):
    """BGZF file -> inflate (k_inflate on the device, or zlib on host threads) -> device kernels -> tables,
    against what the reference printed."""
    monkeypatch.setenv("ITX_INFLATE", inflate)
    cmd, args = kats.KATS[kat]["variants"][variant]
    vdir = os.path.join(GOLD, kat, variant)
    scan = lambda ix, bam, opts: ix.scan_alignments(bam, opts)
    runners.run_itx(capi.Index, scan, os.path.join(GOLD, kat, "input"), cmd, args, str(tmp_path))
    for fn in runners.expected_files(vdir):
        got = os.path.join(str(tmp_path), fn)
        assert os.path.exists(got), fn
        assert same_output(cmd, got, os.path.join(vdir, fn)), "%s differs from the reference's" % fn


def same_output(cmd, got, want):
    """byte for byte, except the CpG tables: their f64 sums are accumulated in another order on the device, so the text
    is compared number by number at 1e-9 relative; the bigWig made from a CpG wiggle is held to the bytes whenever
    that wiggle came out identical"""
    if filecmp.cmp(got, want, shallow=False):
        return True
    if not cmd.startswith("cpg"):
        return False
    if got.endswith(".bigWig"):
        wg, ww = got[:-len(".bigWig")] + ".wig", want[:-len(".bigWig")] + ".wig"
        return os.path.exists(wg) and os.path.exists(ww) and not filecmp.cmp(wg, ww, shallow=False) and close_text(wg, ww)
    return close_text(got, want)


def close_text(a, b, rel=1e-9):
    """equal token by token; numeric tokens within rel (CpG f64 sums are accumulated in another order)"""
    la, lb = open(a).read().split("\n"), open(b).read().split("\n")
    if len(la) != len(lb):
        return False
    for x, y in zip(la, lb):
        tx, ty = x.split("\t"), y.split("\t")
        if len(tx) != len(ty):
            return False
        for p, q in zip(tx, ty):
            if p == q:
                continue
            try:
                fp, fq = float(p), float(q)
            except ValueError:
                return False
            if abs(fp - fq) > rel * max(abs(fp), abs(fq)) + 5.1e-5:   # + half a unit of the printed %.4f
                return False
    return True


SYN = [
    ("se50_chr1", 0, 20000, 0, 200000, {}),
    ("se50_hg19_E0", 1, 60000, 0, 200000, dict(extension=0)),
    ("se75_xa_hg19", 1, 60000, 1, 200000, {}),
    ("se75_xa_nodiff", 1, 60000, 1, 50000, dict(diffSubfam=0)),
    ("pe100_hg19", 1, 60000, 2, 100000, {}),
    ("pe100_treat", 1, 60000, 2, 50000, dict(treat=1)),
    ("pe100_D_I300", 1, 60000, 2, 50000, dict(discardWrongEnd=1, iSize=300)),
    ("se50_Q30_c05", 0, 20000, 0, 50000, dict(mapQ=30, minCoverage=0.5)),
    ("se50_addChr", 1, 60000, 0, 50000, dict(addChr=1)),
    ("se50_chrM_R", 2, 3000, 0, 200000, dict(rmDup=1)),
    ("pe100_R", 1, 60000, 2, 100000, dict(rmDup=1)),
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


def assert_same_tables(ix, ora):
    L = O.lib()
    c4 = (C.c_uint64 * 4)()
    for which, nfun in ((0, L.ora_n_subfam), (1, L.ora_n_fam), (2, L.ora_n_class)):
        got = ix.table(which)
        assert len(got) == nfun(ora.h)
        for i, row in enumerate(got):
            L.ora_counts(ora.h, which, i, c4)
            assert row == (L.ora_name(ora.h, which, i).decode(),) + tuple(c4)
    for i in range(L.ora_n_subfam(ora.h)):
        ln = L.ora_subfam_length(ora.h, i)
        if ln:
            for u in (0, 1):
                want = np.ctypeslib.as_array(L.ora_subfam_bp(ora.h, i, u), shape=(ln,))
                assert np.array_equal(ix.coverage(i, u), want), (i, u)


@pytest.mark.parametrize("chunk", [1024, 8192], ids=["thread_kernel", "tma_span_kernel"])
@pytest.mark.parametrize("case", SYN, ids=[c[0] for c in SYN])
def test_cuda_path_matches_oracle(case, chunk, worlds):
    """chunk 1024 runs k_decode (one thread per chunk); chunks that are whole 4 KiB stages run k_decode_span"""
    name, shape, n_rmsk, mode, n_units, kw = case
    s, (cs, rs, rm), _ = worlds(shape, n_rmsk)
    buf, n, nrec = s.stream(mode, n_units)
    raw = buf[:n].tobytes()
    ora = O.OracleIndex(cs, rs, rm)
    cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(**kw), trace=True)
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=chunk, window_bytes=1 << 20)         # many windows: the carry between windows is on the path
    cnt_g, tr_g = ix.scan_stream(raw, capi.default_opts(**kw), trace=True)
    assert cnt_g == cnt_o
    assert len(tr_g) == len(tr_o) == nrec
    for f in ("start", "end", "tid", "sel_row"):
        assert np.array_equal(tr_g[f], tr_o[f]), f
    mask = ~np.uint32(8 | 64)                                 # HAS_XA: the oracle reports it even where it is not evaluated; DUP is the product's own flag
    assert np.array_equal(tr_g["flags"] & mask, tr_o["flags"] & mask)
    assert_same_tables(ix, ora)
    ora.close()
    ix.close()


@pytest.mark.parametrize("chunk,window", [(256, 1 << 16), (448, 1 << 18), (4096, 1 << 16), (4096, 1 << 30), (32768, 1 << 20), (65536, 1 << 22), (1 << 20, 1 << 23)])
def test_chunk_and_window_size_never_change_the_answer(chunk, window, worlds):
    s, (cs, rs, rm), _ = worlds(1, 60000)
    buf, n, nrec = s.stream(1, 60000)
    raw = buf[:n].tobytes()
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_stream(raw, O.default_opts())
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=chunk, window_bytes=window)
    assert ix.scan_stream(raw, capi.default_opts()) == want
    assert_same_tables(ix, ora)
    if chunk == 256:
        assert ix.profile()["n_bad_chunks"] == 0 or True      # informative only: guesses may or may not miss
    ora.close()
    ix.close()


def test_truncated_stream_stops_like_the_reference(worlds):
    s, (cs, rs, rm), _ = worlds(0, 20000)
    buf, n, nrec = s.stream(0, 30000)
    for cut in (n - 1, n - 40, n - 131, n // 2 + 3):
        raw = buf[:cut].tobytes()
        ora = O.OracleIndex(cs, rs, rm)
        ix = capi.Index(cs, rs, rm)
        ix.tune(chunk_bytes=512, window_bytes=1 << 18)
        assert ix.scan_stream(raw, capi.default_opts()) == ora.scan_stream(raw, O.default_opts())
        ora.close()
        ix.close()


@pytest.mark.parametrize("level", [0, 1, 6])
def test_device_inflate_matches_host_inflate(level, worlds, tmp_path, monkeypatch):
    """every BGZF block through k_inflate (one thread per block) gives the stream zlib gives"""
    s, (cs, rs, rm), _ = worlds(1, 60000)
    bam = str(tmp_path / "reads.bam")
    s.write_bam(bam, 1, 80000, level=level, threads=4)
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_file(bam, O.default_opts())
    for mode in ("device", "host"):
        monkeypatch.setenv("ITX_INFLATE", mode)
        ix = capi.Index(cs, rs, rm)
        assert ix.scan_alignments(bam, capi.default_opts()) == want, mode
        assert_same_tables(ix, ora)
        ix.close()
    ora.close()


@pytest.mark.parametrize("lz", ["2", "0", "1"])
@pytest.mark.parametrize("block", [65536, 0xff00, 6144 + 1, 3072, 257, 40])
def test_bgzf_blocks_of_every_size_and_every_match_copy_pass(block, lz, worlds, tmp_path, monkeypatch):
    """BGZF blocks from the largest the format allows (ISIZE 65536: positions fill 16 bits) down to a few bytes, cut at the edges of
    the match-copy windows, through the three second passes (ITX_LZ=2 inside k_inflate, 0 k_lz_resolve, 1 k_lz_jump): the stream on
    the device is the stream that was compressed, byte for byte"""
    import bamio
    monkeypatch.delenv("ITX_INFLATE", raising=False)
    monkeypatch.setenv("ITX_LZ", lz)
    s, (cs, rs, rm), _ = worlds(1, 60000)
    buf, n, _ = s.stream(1, 6000 if block >= 3072 else 600)
    raw = buf[:n].tobytes()
    bam = str(tmp_path / "reads.bam")
    with open(bam, "wb") as f:
        for i in range(0, n, block):
            f.write(bamio.bgzf_block(raw[i:i + block], 6 if (i // block) % 3 else 1))
        f.write(bamio.EOF_BLOCK)
    ix = capi.Index(cs, rs, rm)
    want = ix.scan_bam_host(buf.ctypes.data, n, capi.default_opts())
    ix.reset()
    assert ix.scan_alignments(bam, capi.default_opts()) == want
    assert ix.stream_fetch(n + 100) == raw
    ix.close()


@pytest.mark.parametrize("mode,level", [(0, 1), (1, 6), (2, 9), (2, 0)])
def test_device_inflate_reproduces_the_stream_byte_for_byte(mode, level, worlds, tmp_path, monkeypatch):
    """k_inflate (decoding and match copies) against the bytes the generator compressed (file entry and memory-image entry)"""
    monkeypatch.delenv("ITX_INFLATE", raising=False)
    s, (cs, rs, rm), _ = worlds(1, 60000)
    bam = str(tmp_path / "reads.bam")
    n, nrec = s.write_bam(bam, mode, 50000, level=level, threads=4)
    buf, n2, _ = s.stream(mode, 50000)
    assert n2 == n
    ix = capi.Index(cs, rs, rm)
    want = ix.scan_bam_host(buf.ctypes.data, n, capi.default_opts())
    ix.reset()
    assert ix.scan_alignments(bam, capi.default_opts()) == want
    assert ix.stream_fetch(n + 100) == buf[:n].tobytes()
    ix.reset()
    img = np.fromfile(bam, dtype=np.uint8)
    assert ix.scan_bgzf_memory(img.ctypes.data, len(img), capi.default_opts()) == want
    assert ix.stream_fetch(n + 100) == buf[:n].tobytes()
    ix.close()


def test_bytes_after_the_eof_block_and_cut_files_end_the_stream_silently(worlds, tmp_path, monkeypatch):
    """bgzf_read stops at an empty block, a bad header or a short block; whatever came before still counts"""
    monkeypatch.delenv("ITX_INFLATE", raising=False)
    s, (cs, rs, rm), _ = worlds(1, 60000)
    bam = str(tmp_path / "reads.bam")
    s.write_bam(bam, 0, 40000, level=1, threads=4)
    raw = open(bam, "rb").read()
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_file(bam, O.default_opts())
    ora.close()
    junk = str(tmp_path / "junk.bam")
    open(junk, "wb").write(raw + b"not a gzip member at all" * 3)
    ix = capi.Index(cs, rs, rm)
    assert ix.scan_alignments(junk, capi.default_opts()) == want
    ix.close()
    # cut inside a block: the blocks before it are the stream
    cut = str(tmp_path / "cut.bam")
    open(cut, "wb").write(raw[: len(raw) * 2 // 3])
    for inflate in ("device", "host"):
        monkeypatch.setenv("ITX_INFLATE", inflate)
        ix = capi.Index(cs, rs, rm)
        got = ix.scan_alignments(cut, capi.default_opts())
        if inflate == "device":
            first = got
        else:
            assert got == first
        assert 0 < got[0] < want[0]
        ix.close()


def test_rmdup_keys_persist_across_the_files_of_a_run(worlds, tmp_path):
    """-R: the key hash lives for the whole run (generic.c:700-745), so every read of a second copy of the file is a
    duplicate; a reset starts a new run.  Small windows: the key table is grown and re-hashed on the way."""
    s, (cs, rs, rm), _ = worlds(2, 3000)
    bam = str(tmp_path / "reads.bam")
    s.write_bam(bam, 0, 150000, level=1, threads=4)
    ora = O.OracleIndex(cs, rs, rm)
    o1 = ora.scan_file(bam, O.default_opts(rmDup=1))
    o2 = ora.scan_file(bam, O.default_opts(rmDup=1))
    assert o2[11] == o1[11] and o2[6] == 2 * o1[6] and o1[11] < o1[7]
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=4096, window_bytes=1 << 20)
    assert ix.scan_alignments(bam + "," + bam, capi.default_opts(rmDup=1)) == o2
    assert_same_tables(ix, ora)
    ix.reset()
    assert ix.scan_alignments(bam, capi.default_opts(rmDup=1)) == o1
    ora.close()
    ix.close()


@pytest.mark.parametrize("mode", ["fused", "tuple_path", "fused_replayed"])
@pytest.mark.parametrize("case", [SYN[1], SYN[2], SYN[4], SYN[7]], ids=lambda c: c[0])
def test_fused_and_tuple_paths_count_the_same(case, mode, worlds, monkeypatch):
    """k_scan (one kernel per launch group), the tuple path it falls back to, and the replay of a scan whose chain
    check is declared failed (take everything back with sign -1, count again through the tuple path) all give
    the oracle's numbers"""
    name, shape, n_rmsk, rmode, n_units, kw = case
    if mode == "tuple_path":
        monkeypatch.setenv("ITX_FUSED", "0")
    if mode == "fused_replayed":
        monkeypatch.setenv("ITX_FUSED_TEST_REPLAY", "1")
    s, (cs, rs, rm), _ = worlds(shape, n_rmsk)
    buf, n, nrec = s.stream(rmode, n_units)
    raw = buf[:n].tobytes()
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_stream(raw, O.default_opts(**kw))
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=8192, window_bytes=1 << 20)           # several launch groups: the carry crosses them
    assert ix.scan_stream(raw, capi.default_opts(**kw)) == want
    pr = ix.profile()
    assert pr["fused"] == (0 if mode == "tuple_path" else 1)
    assert (pr["n_replayed_windows"] > 0) == (mode == "fused_replayed")
    assert_same_tables(ix, ora)
    ora.close()
    ix.close()


@pytest.mark.parametrize("flags", [0, 3, 4, 12, 15, 16, 16 + 256, 256, 511, 2 + 4 + 8 + 32 + 256, 2 + 4 + 8 + 16 + 32 + 64 + 256])
@pytest.mark.parametrize("case", [SYN[1], SYN[2], SYN[4]], ids=lambda c: c[0])
def test_scan_kernel_switches_never_change_the_counts(case, flags, worlds, monkeypatch):
    """k_scan's switches (L2 prefetch, dominant-size chain walk, table window, window look-ahead, early stage copy, evict-first hint,
    lane-per-alternate XA walk, margin carry) are performance choices only: every combination gives the oracle's numbers, on a resident stream taken as ONE launch
    group as well as through the host path"""
    name, shape, n_rmsk, rmode, n_units, kw = case
    monkeypatch.setenv("ITX_SCAN_FLAGS", str(flags))
    s, (cs, rs, rm), _ = worlds(shape, n_rmsk)
    buf, n, nrec = s.stream(rmode, n_units)
    raw = buf[:n].tobytes()
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_stream(raw, O.default_opts(**kw))
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=4096)                                  # many spans per warp, one launch group
    L = capi.lib()
    a = np.frombuffer(raw + b"\0" * 64, dtype=np.uint8)
    d = L.itx_dev_alloc(len(a))
    assert d and L.itx_dev_upload(d, a.ctypes.data, len(a)) == 0
    hdr = ix.header(a.ctypes.data, n)
    assert ix.scan_bam_device(hdr, d, n, capi.default_opts(**kw)) == want
    # one k_scan per launch group, plus k_xa (the reads with XA:Z alternates) when mapped2diffSubfam is on
    assert ix.profile()["fused"] == 1 and ix.profile()["n_launches"] == (2 if capi.default_opts(**kw).diffSubfam else 1)
    assert_same_tables(ix, ora)
    ix.reset()
    assert ix.scan_stream(raw, capi.default_opts(**kw)) == want
    assert_same_tables(ix, ora)
    L.itx_bam_header_free(hdr)
    L.itx_dev_free(d)
    ora.close()
    ix.close()


def test_damaged_bgzf_block_is_reported(worlds, tmp_path, monkeypatch):
    s, (cs, rs, rm), _ = worlds(1, 60000)
    bam = str(tmp_path / "reads.bam")
    s.write_bam(bam, 0, 30000, level=6, threads=4)
    raw = bytearray(open(bam, "rb").read())
    for k in range(40000, 40400):
        raw[k] ^= 0x5a
    open(bam, "wb").write(raw)
    for mode in ("device", "host"):
        monkeypatch.setenv("ITX_INFLATE", mode)
        ix = capi.Index(cs, rs, rm)
        with pytest.raises(capi.ItxError) as e:
            ix.scan_alignments(bam, capi.default_opts())
        assert e.value.code == -2 and "inflate failed" in str(e.value)
        ix.close()


def test_bgzf_file_host_stream_and_device_stream_agree(worlds, tmp_path):
    """the three entry points (file, host stream, device-resident stream) share one result; counters
    persist across calls until reset (multi-file runs, generic.c:700-745)"""
    s, (cs, rs, rm), _ = worlds(1, 60000)
    bam = str(tmp_path / "reads.bam")
    n, nrec = s.write_bam(bam, 2, 60000, level=1, threads=4)
    buf, n2, _ = s.stream(2, 60000)
    assert n2 == n
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_file(bam, O.default_opts())
    ix = capi.Index(cs, rs, rm)
    opts = capi.default_opts()
    assert ix.scan_alignments(bam, opts) == want
    assert_same_tables(ix, ora)
    ix.reset()
    assert ix.scan_bam_host(buf.ctypes.data, n, opts) == want
    ix.reset()
    L = capi.lib()
    d = L.itx_dev_alloc(n + 64)
    assert d and L.itx_dev_upload(d, buf.ctypes.data, n + 64) == 0
    hdr = ix.header(buf.ctypes.data, n)
    assert ix.scan_bam_device(hdr, d, n, opts) == want
    assert_same_tables(ix, ora)
    # a second file on the same index adds up (the reference's comma separated list)
    assert ix.scan_alignments(bam + "," + bam, opts) == [3 * v for v in want]
    L.itx_bam_header_free(hdr)
    L.itx_dev_free(d)
    ora.close()
    ix.close()


def test_overlap_kernel_property(worlds):
    """random queries (bin straddlers, nested and abutting elements, chromosome ends) against the oracle's
    binKeeper restatement: same selected rmsk row, same hit count"""
    s, (cs, rs, rm), _ = worlds(1, 60000)
    ora = O.OracleIndex(cs, rs, rm)
    ix = capi.Index(cs, rs, rm)
    rng = np.random.default_rng(5)
    rows = [l.split("\t") for l in open(rm)]
    for chrom in ("chr1", "chr7", "chrM", "chrX"):
        el = np.array([(int(r[6]), int(r[7])) for r in rows if r[5] == chrom], dtype=np.int64)
        size = dict(l.split() for l in open(cs))[chrom]
        size = int(size)
        q = []
        pick = el[rng.integers(0, len(el), 3000)] if len(el) else np.zeros((0, 2), dtype=np.int64)
        for (a, b) in pick:                      # around element edges
            st = max(0, a + int(rng.integers(-200, 200)))
            q.append((st, st + int(rng.integers(1, 400))))
        for k in range(1, 40):                   # across 128 kb / 1 Mb bin boundaries
            for w in (1, 36, 150, 2000):
                q.append((max(0, k * 131072 - w // 2), k * 131072 + w))
                q.append((max(0, k * 1048576 - w), k * 1048576 + 1))
        q += [(0, 1), (0, 150), (size - 150, size - 1), (size - 1, size), (size, size + 10), (5, 5), (10, 3), (2 ** 31 + 5, 2 ** 31 + 9)]
        st = np.array([x[0] for x in q], dtype=np.uint32)
        en = np.array([min(x[1], 2 ** 32 - 1) for x in q], dtype=np.uint32)
        for mc in (1e-4, 0.5):
            sel, nh = ix.query_select(chrom, st, en, mc)
            for i in range(len(q)):
                ws, hits = ora.find_select(chrom, int(st[i]), int(en[i]), mc)
                assert (sel[i], nh[i]) == (ws, len(hits)), (chrom, q[i], mc)
    ora.close()
    ix.close()


def test_overlap_kernel_on_nested_table(tmp_path):
    """hit lists of every length (the long-list path included) and coverages on both sides of every threshold: k_query
    against the oracle's binKeeper restatement"""
    from test_emu_synth import _nested_world
    cs, rs, rm, rows = _nested_world(str(tmp_path))
    ora = O.OracleIndex(cs, rs, rm)
    ix = capi.Index(cs, rs, rm)
    rng = np.random.default_rng(3)
    q = []
    for (a, b) in rows:
        for _ in range(6):
            st = max(0, a + int(rng.integers(-120, 120)))
            q.append((st, st + int(rng.integers(1, 300))))
        q += [(a, b), (a + 1, b - 1), (max(0, a - 1), b + 1)]
        for ov in (1, 2, 3, 5):
            for length in (ov * 4095, ov * 4096, ov * 4097, ov * 8191, ov * 8192, ov * 8193, ov * 9999, ov * 10000, ov * 10001):
                q.append((b - ov, b - ov + length))
    for (a, b) in rows[-12:]:                         # fragments of 2^23 bases and more (float comparison of the coverages) over the last few stacks
        q += [(max(0, a - 3), a - 3 + 9000000), (a + 1, a + 1 + (1 << 23)), (b - 2, b - 2 + 20000000)]
    st = np.array([x[0] for x in q], dtype=np.uint32)
    en = np.array([x[1] for x in q], dtype=np.uint32)
    for mc in (1e-4, 0.0, 2.0 ** -13, 0.00012, 0.5):
        sel, nh = ix.query_select("chrN", st, en, mc)
        for i in range(len(q)):
            ws, hits = ora.find_select("chrN", int(st[i]), int(en[i]), mc)
            assert (sel[i], nh[i]) == (ws, len(hits)), (q[i], mc)
    ora.close()
    ix.close()


@pytest.mark.parametrize("fused", [1, 0])
def test_xa_strings_of_every_shape(fused, tmp_path, monkeypatch):
    """mapped2diffSubfam on alternate lists that chopByChar / strtol treat in their own ways (empty and malformed pieces,
    more than 100 pieces, hexadecimal and octal numbers, XA of another type, aux areas larger than k_xa's pool, array counts that leave
    the aux area): k_scan + k_xa and the tuple path against the oracle"""
    import bamio
    from test_emu_synth import xa_odd_reads
    monkeypatch.setenv("ITX_FUSED", str(fused))
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    open(rm, "w").write("\n".join(kats.ANNOT1) + "\n")
    reads = xa_odd_reads()
    raw = bamio.encode_header([("chr1", 1000000)]) + b"".join(bamio.encode_record(r) for r in reads)
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_stream(raw, O.default_opts())
    assert 0 < want[12] < len(reads)
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=4096)
    assert ix.scan_stream(raw, capi.default_opts()) == want
    assert ix.profile()["fused"] == fused
    assert_same_tables(ix, ora)
    ora.close()
    ix.close()


@pytest.mark.parametrize("fused", [1, 0])
def test_adversarial_records_match_oracle(fused, tmp_path, monkeypatch):
    """records built to sit on every branch of the fragment logic (positions at and past chromosome ends, reference ids
    past n_ref, isize edges, every flag mix) under several option sets: k_scan and the tuple path against the oracle"""
    import struct
    import bamio
    from test_emu_synth import _adversarial_records
    monkeypatch.setenv("ITX_FUSED", str(fused))
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\nchrM\t16571\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    rows = kats.ANNOT1 + [kats.rmsk_row("chrM", 100, 400, "+", "AluY", "SINE", "Alu", 1, 300, 0),
                          kats.rmsk_row("chr1", 999900, 1000000, "-", "L1PA2", "LINE", "L1", -100, 5900, 5800),
                          kats.rmsk_row("chr1", 0, 40, "+", "MIR", "SINE", "MIR", 1, 41, 0)]
    open(rm, "w").write("\n".join(rows) + "\n")
    refs = [("chr1", 1000000), ("chrM", 16571), ("chrUn_x", 5000)]
    reads = _adversarial_records(np.random.default_rng(4), 3000, len(refs))

    def enc(r):
        b = bytearray(bamio.encode_record(dict(r, pos=min(max(r["pos"], 0), 1 << 28))))
        b[8:12] = struct.pack("<i", r["pos"])
        return bytes(b)
    raw = bamio.encode_header(refs) + b"".join(enc(r) for r in reads)
    for kw in (dict(), dict(extension=0), dict(extension=1000), dict(treat=1), dict(discardWrongEnd=1, iSize=200), dict(mapQ=30, minCoverage=0.5),
               dict(mapQ=0, minCoverage=0.0), dict(addChr=1)):
        ora = O.OracleIndex(cs, rs, rm)
        want = ora.scan_stream(raw, O.default_opts(**kw))
        ix = capi.Index(cs, rs, rm)
        ix.tune(chunk_bytes=4096)
        assert ix.scan_stream(raw, capi.default_opts(**kw)) == want, kw
        assert ix.profile()["fused"] == fused
        assert_same_tables(ix, ora)
        ora.close()
        ix.close()


@pytest.mark.parametrize("window", [0, 1 << 16])
@pytest.mark.parametrize("fused", [1, 0])
def test_wrong_span_guesses_are_caught_and_repaired(fused, window, tmp_path, monkeypatch):
    """valid-looking records inside byte-array aux fields are taken for record starts by the span guess: k_scan's chain
    check must notice, take back what it counted (sign -1) and count again through the tuple path, whose k_fixup repairs
    the guesses -- without the test hook, on wrong guesses the kernels really make"""
    from test_emu_synth import decoy_stream
    monkeypatch.setenv("ITX_FUSED", str(fused))
    d = str(tmp_path)
    cs, rs, rm = (os.path.join(d, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    open(cs, "w").write("chr1\t1000000\n")
    open(rs, "w").write("AluY\t300\nL1PA2\t6000\n")
    open(rm, "w").write("\n".join(kats.ANNOT1) + "\n")
    raw, nrec = decoy_stream()
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_stream(raw, O.default_opts())
    assert want[0] == nrec and want[9] > 0
    ix = capi.Index(cs, rs, rm)
    ix.tune(chunk_bytes=4096, window_bytes=window)              # one launch group, or several: the undo restarts from a logged carry
    assert ix.scan_stream(raw, capi.default_opts()) == want
    pr = ix.profile()
    assert pr["fused"] == fused
    assert pr["n_replayed_windows"] > 0 if fused else pr["n_bad_chunks"] > 0
    assert_same_tables(ix, ora)
    ora.close()
    ix.close()


def test_cpg_matches_oracle(worlds, tmp_path):
    s, (cs, rs, rm), _ = worlds(1, 60000)
    bg = str(tmp_path / "cpg.bedGraph")
    s.write_bedgraph(bg, 300000)
    for filt in (0, 1):
        ora = O.OracleIndex(cs, rs, rm)
        ix = capi.Index(cs, rs, rm)
        assert ix.scan_cpg(bg, filt) == ora.scan_cpg(bg, filt)
        a, b = str(tmp_path / ("g%d" % filt)), str(tmp_path / ("o%d" % filt))
        if filt == 0:
            ix.write_cpg_stat(a); ora.write_cpg_stat(b)
            names = [".CpG.subfamily.stat", ".CpGstat.wig", ".CpG.family.stat", ".CpG.class.stat"]
        else:
            ix.write_cpg_filter(a + ".loci", 1.0); ora.write_cpg_filter(b + ".loci", 1.0)
            names = [".loci"]
        for nme in names:
            assert close_text(a + nme, b + nme), nme
        ora.close()
        ix.close()


def test_filter_mode_counts_per_locus(worlds):
    s, (cs, rs, rm), _ = worlds(1, 60000)
    buf, n, nrec = s.stream(0, 100000)
    raw = buf[:n].tobytes()
    ora = O.OracleIndex(cs, rs, rm)
    cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(filter=1, diffSubfam=0), trace=True)
    ix = capi.Index(cs, rs, rm)
    assert ix.scan_stream(raw, capi.default_opts(filter=1, diffSubfam=0)) == cnt_o
    want = np.zeros(len(ix.elem_counts_by_row()), dtype=np.uint32)
    counted = (tr_o["flags"] & 32) != 0
    np.add.at(want, tr_o["sel_row"][counted], 1)
    assert np.array_equal(ix.elem_counts_by_row(), want)
    ora.close()
    ix.close()


@pytest.mark.parametrize("chunk,window", [(1024, 1 << 18), (4096, 1 << 18), (32768, 1 << 30), (65536, 1 << 20)])
def test_records_of_every_size(chunk, window, tmp_path):
    """records from 60 bytes to 70 KB: longer than a span (spans without any record start), than a stage and its
    margin (the global-memory fall-back of the staged source), of 64 KiB and more (stepped over one at a time by the
    chain walk) and straddling launch groups"""
    import mixed_records
    tabs = mixed_records.tables(str(tmp_path))
    raw, nrec = mixed_records.make()
    for kw in ({}, dict(extension=0, treat=1)):
        ora = O.OracleIndex(*tabs)
        cnt_o, tr_o = ora.scan_stream(raw, O.default_opts(**kw), trace=True)
        ix = capi.Index(*tabs)
        ix.tune(chunk_bytes=chunk, window_bytes=window)
        cnt_g, tr_g = ix.scan_stream(raw, capi.default_opts(**kw), trace=True)
        assert cnt_g == cnt_o and cnt_o[0] + cnt_o[1] == nrec
        for f in ("start", "end", "tid", "sel_row"):
            assert np.array_equal(tr_g[f], tr_o[f]), f
        assert np.array_equal(tr_g["flags"] & ~np.uint32(8), tr_o["flags"] & ~np.uint32(8))
        assert_same_tables(ix, ora)
        ora.close()
        ix.close()


def test_window_smaller_than_a_record_is_refused(tmp_path):
    import mixed_records
    tabs = mixed_records.tables(str(tmp_path))
    raw, nrec = mixed_records.make()
    ix = capi.Index(*tabs)
    ix.tune(chunk_bytes=4096, window_bytes=1 << 16)          # 64 KiB windows, 70 KB records
    with pytest.raises(capi.ItxError) as e:
        ix.scan_stream(raw, capi.default_opts())
    assert e.value.code == -6 and "longer than the staged window" in str(e.value)
    ix.close()


@pytest.mark.parametrize("kat,variant", [("kat1_basic", "default"), ("kat1_basic", "S"), ("kat4_paired_xa", "B"), ("kat4_paired_xa", "S_B"),
                                         ("kat4_paired_xa", "R"), ("kat1_basic", "filter_r"), ("kat5_cpg", "cpgstat"), ("kat5_cpg", "cpgfilter")])
def test_command_line_tool_is_a_drop_in(kat, variant, tmp_path):
    """the `iteres` binary with the reference's own command line: same files, same bytes (stderr is not compared)"""
    import subprocess
    cmd, args = kats.KATS[kat]["variants"][variant]
    inp = os.path.join(GOLD, kat, "input")
    data = "cpg.bedGraph" if cmd.startswith("cpg") else ("reads.sam" if "-S" in args else "reads.bam")
    cli = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "iteres_b200", "csrc", "iteres")
    p = subprocess.run([cli, cmd] + args + ["-o", "out"] + [os.path.join(inp, x) for x in ("chrom.sizes", "rep.sizes", "rmsk.txt", data)],
                       cwd=str(tmp_path), capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    vdir = os.path.join(GOLD, kat, variant)
    want = runners.expected_files(vdir)
    assert sorted(os.listdir(str(tmp_path))) == want
    for fn in want:
        assert same_output(cmd, os.path.join(str(tmp_path), fn), os.path.join(vdir, fn)), fn


@pytest.mark.parametrize("parse", ["device", "host"])
def test_bedgraph_text_oddities(parse, worlds, tmp_path, monkeypatch):
    """k_bedgraph parses the text itself: blank and comment lines, leading blanks, CRLF, extra columns, hexadecimal
    and octal coordinates, exponents, and scores that only the host's strtod can do (handed back by offset)"""
    if parse == "host":
        monkeypatch.setenv("ITX_CPG_PARSE", "host")
    s, (cs, rs, rm), d = worlds(1, 60000)
    src = str(tmp_path / "base.bedGraph")
    s.write_bedgraph(src, 3000)
    rows = [l.split() for l in open(src)]
    rnd = np.random.RandomState(5)
    out = ["# a comment", "", "   ", "track type=bedGraph"[0:0]]
    for i, (c, a, b, v) in enumerate(rows):
        k = i % 9
        if k == 0: out.append("  %s\t%s\t%s\t%s" % (c, a, b, v))
        elif k == 1: out.append("%s %s %s %s extra columns here" % (c, a, b, v))
        elif k == 2: out.append("%s\t0x%x\t%s\t%s\r" % (c, int(a), b, v))
        elif k == 3: out.append("%s\t%s\t%s\t%se0" % (c, a, b, v))
        elif k == 4: out.append("%s\t%s\t%s\t%s" % (c, a, b, "0.1234567890123456789012"))      # more digits than 64 bits hold: host
        elif k == 5: out.append("%s\t%s\t%s\t%s" % (c, a, b, "1e-30"))                          # power of ten beyond the exact range: host
        elif k == 6: out.append("#%s\t%s\t%s\t%s" % (c, a, b, v))
        elif k == 7: out.append("%s\t%s\t%s\t%.3e" % (c, a, b, float(v)))
        else: out.append("%s\t%s\t%s\t%s" % (c, a, b, v))
    odd = str(tmp_path / "odd.bedGraph")
    open(odd, "w").write("\n".join(out))                       # no newline after the last line
    ora = O.OracleIndex(cs, rs, rm)
    want = ora.scan_cpg(odd, 0)
    ix = capi.Index(cs, rs, rm)
    assert ix.scan_cpg(odd, 0) == want
    a, b = str(tmp_path / "g"), str(tmp_path / "o")
    ix.write_cpg_stat(a); ora.write_cpg_stat(b)
    for nme in (".CpG.subfamily.stat", ".CpGstat.wig", ".CpG.family.stat", ".CpG.class.stat"):
        assert close_text(a + nme, b + nme), nme
    assert want[0] == sum(1 for i in range(len(rows)) if i % 9 != 6) and want[1] > 0
    ora.close()
    ix.close()
    bad = str(tmp_path / "bad.bedGraph")
    open(bad, "w").write("\n".join(out[:50] + ["chr1\t5\t7"] + out[50:]) + "\n")
    ix = capi.Index(cs, rs, rm)
    with pytest.raises(capi.ItxError) as e:
        ix.scan_cpg(bad, 0)
    assert "At least 4 fields required, got 3" in str(e.value)
    ix.close()


def test_two_indexes_of_different_sizes_in_one_process(worlds):
    """the scan kernels' shared-memory attribute belongs to the function, not to an index: an index with a larger histogram must
    still launch after a smaller one has been used (a process that holds several indexes: the bench, a multi-device caller)"""
    s_big, tabs_big, _ = worlds(1, 60000)          # 1395 subfamilies
    s_small, tabs_small, _ = worlds(0, 20000)      # 1200 subfamilies
    buf, n, nrec = s_big.stream(0, 30000)
    raw_big = buf[:n].tobytes()
    buf, n, nrec = s_small.stream(0, 30000)
    raw_small = buf[:n].tobytes()
    a, b = capi.Index(*tabs_big), capi.Index(*tabs_small)
    want_a = a.scan_stream(raw_big, capi.default_opts())
    want_b = b.scan_stream(raw_small, capi.default_opts())
    a.reset(); b.reset()
    assert a.scan_stream(raw_big, capi.default_opts()) == want_a
    assert b.scan_stream(raw_small, capi.default_opts()) == want_b
    a.reset()
    assert a.scan_stream(raw_big, capi.default_opts()) == want_a
    a.close(); b.close()
