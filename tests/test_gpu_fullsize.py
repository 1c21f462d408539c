"""The CUDA path at the bench's table density (5.5 M rmsk rows, BASELINE.json configs[1]) against the oracle on a bounded number of
reads, and -- at the full 50 M reads, where the CPU oracle would need minutes -- through properties that do not depend on the size:
the fused kernel, the tuple path and the BGZF file path are three different routes to the same sums, and a stream cut at a record
boundary adds up (every output is a sum over reads)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
import synth
from iteres_b200 import capi
from test_gpu_parity import assert_same_tables

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dense(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("dense"))
    s = synth.Synth(1, 5_500_000, seed=1)
    tabs = s.write_tables(d)
    yield s, tabs, d
    s.close()


def test_bench_density_against_the_oracle(dense):
    """2 M SE-50 reads, 1 M SE-75 reads with XA lists and 0.5 M PE-100 pairs vs 5.5 M rows: all 13 counters, the three tables, both
    coverage vectors; then the per-locus counts of filter mode"""
    s, tabs, d = dense
    ora = O.OracleIndex(*tabs)
    ix = capi.Index(*tabs)
    for mode, units in ((0, 2_000_000), (1, 1_000_000), (2, 500_000)):
        bam = os.path.join(d, "m%d.bam" % mode)
        s.write_bam(bam, mode, units, level=1, threads=8)
        ora.reset()
        want = ora.scan_file(bam, O.default_opts())
        ix.reset()
        assert ix.scan_alignments(bam, capi.default_opts()) == want and want[9] > 0
        if mode == 1:
            assert want[12] > 0                                  # mapped2diffSubfam did discard reads
        assert_same_tables(ix, ora)
    # filter mode on the XA file: per-locus counts summed per subfamily are the stat-mode counts without -x ...
    bam = os.path.join(d, "m1.bam")
    ora.reset()
    ix.reset()
    want = ora.scan_file(bam, O.default_opts(filter=1, diffSubfam=0))
    assert ix.scan_alignments(bam, capi.default_opts(filter=1, diffSubfam=0)) == want
    got = ix.elem_counts_by_row(0)
    assert int(got.astype(np.uint64).sum()) == want[9] and int(ix.elem_counts_by_row(1).astype(np.uint64).sum()) == want[10]
    ix.close()
    ora.close()


def test_full_size_routes_agree(dense, monkeypatch):
    """50 M SE-50 reads (6.5 GB) resident in HBM: k_scan (one launch), the tuple path (k_decode_span / k_verify / k_fixup / k_overlap)
    and the two halves of the stream scanned one after the other give the same counters, tables and coverage vectors"""
    s, tabs, d = dense
    L = capi.lib()
    ix = capi.Index(*tabs)
    n_units = 50_000_000
    hdr = s.header()
    sz, nrec = s.records_size(0, n_units, 0, None, 16)
    n = len(hdr) + sz
    hbuf = L.itx_host_alloc_pinned(n + 64)
    assert hbuf
    C.memmove(hbuf, hdr.ctypes.data, len(hdr))
    assert s.records_into(hbuf + len(hdr), 0, n_units, 0, None, 16) == sz
    C.memset(hbuf + n, 0, 64)
    dbuf = L.itx_dev_alloc(n + 64)
    assert dbuf and L.itx_dev_upload(dbuf, hbuf, n + 64) == 0
    h = ix.header(hbuf, n)
    opts = capi.default_opts()
    fused = ix.scan_bam_device(h, dbuf, n, opts)
    assert ix.profile()["fused"] == 1 and ix.profile()["n_replayed_windows"] == 0
    assert fused[0] + fused[1] == nrec
    t_fused = [ix.table(w) for w in range(3)]
    cov_fused = [ix.coverage(i, u) for i in range(0, ix.n(0), 11) for u in (0, 1)]
    monkeypatch.setenv("ITX_FUSED", "0")
    ix.reset()
    assert ix.scan_bam_device(h, dbuf, n, opts) == fused and ix.profile()["fused"] == 0
    assert [ix.table(w) for w in range(3)] == t_fused
    monkeypatch.delenv("ITX_FUSED")
    # two halves: generator chunks [0, k) and [k, end) are whole records; the second half is a stream of its own behind a copy of the header
    nch = s.n_chunks(n_units)
    k = nch // 2
    sz_a, nrec_a = s.records_size(0, n_units, 0, k, 16)
    cut = len(hdr) + sz_a
    ix.reset()
    first = ix.scan_bam_device(h, dbuf, cut, opts)
    assert first[0] + first[1] == nrec_a
    # second half in place: the header bytes are written over the tail of the first half (device copy of the host image)
    hl = len(hdr)
    C.memmove(hbuf + cut - hl, hdr.ctypes.data, hl)
    assert L.itx_dev_upload(dbuf + cut - hl, hbuf + cut - hl, hl) == 0
    both = ix.scan_bam_device(h, dbuf + cut - hl, n - cut + hl, opts) if (cut - hl) % 16 == 0 else None
    if both is None:                                            # the device path wants a 16-byte aligned stream: go through the host entry point
        both = ix.scan_bam_host(hbuf + cut - hl, n - cut + hl, opts)
    assert both == fused                                        # counters accumulate across scans until the next reset
    assert [ix.table(w) for w in range(3)] == t_fused
    assert all(np.array_equal(a, b) for a, b in zip(cov_fused, [ix.coverage(i, u) for i in range(0, ix.n(0), 11) for u in (0, 1)]))
    L.itx_bam_header_free(h)
    L.itx_dev_free(dbuf)
    L.itx_host_free_pinned(hbuf)
    ix.close()
