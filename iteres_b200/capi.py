"""ctypes binding of libiteres_gpu.so -- one Python method per C-ABI entry point of
include/iteres_gpu.h (which cites the reference function each one replaces)."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
ERRLEN = 256


def lib_path():
    # ITX_LIB: another build of the same library (A/B measurements of compile-time variants)
    return os.environ.get("ITX_LIB") or os.path.join(HERE, "csrc", "libiteres_gpu.so")


class ItxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("[%d] %s" % (code, msg))
        self.code = code


class ScanOpts(C.Structure):
    """itx_scan_opts == the scalar arguments of samFiles2nodupRepbedFileNew (generic.c:700)."""
    _fields_ = [("mapQ", C.c_uint32), ("filter", C.c_int32), ("rmDup", C.c_int32), ("addChr", C.c_int32),
                ("discardWrongEnd", C.c_int32), ("iSize", C.c_uint32), ("extension", C.c_uint32),
                ("minCoverage", C.c_float), ("treat", C.c_int32), ("diffSubfam", C.c_int32),
                ("readNames", C.c_int32), ("isSam", C.c_int32), ("outbed", C.c_char_p), ("outbed_unique", C.c_char_p)]


class ShardReport(C.Structure):
    """itx_shard_report: how the record chain entered and left one rank's part of a file"""
    _fields_ = [("entry_rel", C.c_uint64), ("exit_rel", C.c_uint64), ("own_bytes", C.c_uint64)]


SHARD_GUESS, SHARD_END, SHARD_NONE = 0xfffffffffffffffd, 0xfffffffffffffffe, 0xffffffffffffffff


def shard_chain_check(reports, L=None):
    """itx_shard_chain_check on a list of (entry_rel, exit_rel, own_bytes): (first rank that must scan again or -1, its entry)"""
    L = L or lib()
    arr = (ShardReport * len(reports))(*[ShardReport(*r) for r in reports])
    forced = C.c_uint64(0)
    L.itx_shard_chain_check.argtypes = [C.c_int, C.POINTER(ShardReport), C.POINTER(C.c_uint64)]
    bad = L.itx_shard_chain_check(len(reports), arr, C.byref(forced))
    return bad, forced.value


class Trace(C.Structure):
    _fields_ = [("start", C.c_uint32), ("end", C.c_uint32), ("tid", C.c_int32), ("sel_row", C.c_int32),
                ("flags", C.c_uint32)]


class Profile(C.Structure):
    _fields_ = [("decode_ms", C.c_double), ("overlap_ms", C.c_double), ("finalize_ms", C.c_double),
                ("total_ms", C.c_double), ("h2d_ms", C.c_double), ("inflate_ms", C.c_double),
                ("n_records", C.c_uint64), ("n_fragments", C.c_uint64), ("stream_bytes", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("n_launches", C.c_uint64),
                ("n_bad_chunks", C.c_uint64), ("inflate_threads", C.c_int32), ("fused", C.c_int32), ("n_replayed_windows", C.c_uint64),
                ("cpg_kernel_ms", C.c_double), ("rmdup_keys_ms", C.c_double), ("rmdup_exchange_ms", C.c_double),
                ("rmdup_count_ms", C.c_double), ("rmdup_bcast_bytes", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def default_opts(**kw):
    o = ScanOpts(10, 0, 0, 0, 0, 500, 150, 1e-4, 0, 1, 0, 0, None, None)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


# every symbol include/iteres_gpu.h declares (tests/test_abi.py checks the library exports them all)
SYMBOLS = """itx_scan_opts_default itx_device_count itx_set_device itx_version itx_index_build itx_index_free
itx_index_reset_counts itx_scan_alignments itx_scan_alignment_file itx_scan_bgzf_memory itx_scan_bam_host itx_bam_header_parse
itx_bam_header_len itx_bam_header_free itx_scan_bam_device itx_scan_cpg itx_sync_counts itx_write_stat
itx_write_report itx_write_filter itx_write_cpg_stat itx_write_cpg_filter itx_n_subfam itx_n_fam itx_n_class
itx_n_elem itx_n_repeats_parsed itx_n_chrom itx_name itx_counts itx_subfam_length itx_subfam_bp itx_n_rows itx_elem_counts_by_row
itx_trace_enable itx_trace_fetch itx_query_select itx_last_profile itx_mark itx_elapsed_ms itx_tune itx_comm_unique_id itx_comm_init
itx_comm_allreduce_counts itx_get_counters itx_comm_destroy itx_scan_shard_file itx_shard_chain_check
itx_scan_alignments_shard itx_scan_cpg_shard itx_get_cpg_totals itx_comm_rank itx_index_build_on itx_dev_alloc itx_dev_free itx_dev_upload itx_host_alloc_pinned
itx_host_free_pinned itx_dev_flush_l2 itx_dev_sync itx_stream_fetch itx_wig_to_bigwig itx_sam_to_bam itx_free
itx_shard_dedup_keys itx_shard_dedup_fetch itx_dedup_admit itx_scan_shard_file_rmdup""".split()

_lib = None


def bind(L):
    """argtypes/restypes shared by the product library and the test-only emulator (host-side symbols)."""
    vp, cp, u64 = C.c_void_p, C.c_char_p, C.c_uint64
    L.itx_write_stat.argtypes = [vp] + [cp] * 5 + [u64, u64]
    L.itx_write_report.argtypes = [cp, C.POINTER(u64), C.c_uint32, cp]
    L.itx_write_filter.argtypes = [vp, cp, C.c_int, C.c_int, u64]
    L.itx_write_cpg_stat.argtypes = [vp] + [cp] * 4
    L.itx_write_cpg_filter.argtypes = [vp, cp, C.c_double]
    for f in ("itx_n_subfam", "itx_n_fam", "itx_n_class", "itx_n_chrom"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = C.c_int32
    for f in ("itx_n_elem", "itx_n_rows", "itx_n_repeats_parsed"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = C.c_int64
    L.itx_name.restype = cp
    L.itx_name.argtypes = [vp, C.c_int, C.c_int32]
    L.itx_counts.argtypes = [vp, C.c_int, C.c_int32, C.POINTER(u64)]
    L.itx_subfam_length.restype = C.c_uint32
    L.itx_subfam_length.argtypes = [vp, C.c_int32]
    L.itx_subfam_bp.restype = C.POINTER(C.c_uint32)
    L.itx_subfam_bp.argtypes = [vp, C.c_int32, C.c_int]
    L.itx_elem_counts_by_row.restype = C.POINTER(C.c_uint32)
    L.itx_elem_counts_by_row.argtypes = [vp, C.c_int]
    return L


def lib():
    """Load the CUDA library; fails loudly when it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise ItxError(-3, "libiteres_gpu.so is not built (run __graft_entry__.build()); there is no CPU path")
        L = bind(C.CDLL(p))
        vp, cp, u64 = C.c_void_p, C.c_char_p, C.c_uint64
        L.itx_version.restype = cp
        L.itx_index_build.restype = vp
        L.itx_index_build.argtypes = [cp, cp, cp, C.c_int, cp, cp]
        L.itx_index_free.argtypes = [vp]
        L.itx_index_reset_counts.argtypes = [vp]
        L.itx_scan_alignments.argtypes = [vp, cp, C.POINTER(ScanOpts), C.POINTER(u64), cp]
        L.itx_scan_bgzf_memory.argtypes = [vp, vp, u64, C.POINTER(ScanOpts), C.POINTER(u64), cp]
        L.itx_scan_alignment_file.argtypes = [vp, cp, C.POINTER(ScanOpts), C.POINTER(u64), cp]
        L.itx_scan_shard_file.argtypes = [vp, cp, C.POINTER(ScanOpts), C.c_int, C.c_int, u64, C.POINTER(ShardReport), C.POINTER(u64), cp]
        L.itx_shard_chain_check.argtypes = [C.c_int, C.POINTER(ShardReport), C.POINTER(u64)]
        L.itx_shard_dedup_keys.argtypes = [vp, cp, C.POINTER(ScanOpts), C.c_int, C.c_int, u64, C.POINTER(ShardReport), C.POINTER(u64), C.POINTER(C.c_uint32), cp]
        L.itx_shard_dedup_fetch.restype = u64
        L.itx_shard_dedup_fetch.argtypes = [vp, vp, u64]
        L.itx_dedup_admit.argtypes = [vp, vp, u64, C.c_uint32, cp]
        L.itx_scan_shard_file_rmdup.argtypes = [vp, cp, C.POINTER(ScanOpts), C.c_int, C.c_int, u64, C.POINTER(ShardReport), C.POINTER(u64), cp]
        L.itx_scan_alignments_shard.argtypes = [vp, cp, C.POINTER(ScanOpts), C.POINTER(u64), cp]
        L.itx_scan_cpg_shard.argtypes = [vp, cp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), cp]
        L.itx_get_cpg_totals.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
        L.itx_comm_rank.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.itx_index_build_on.restype = vp
        L.itx_index_build_on.argtypes = [C.c_int, cp, cp, cp, C.c_int, cp, cp]
        L.itx_scan_bam_host.argtypes = [vp, vp, u64, C.POINTER(ScanOpts), C.POINTER(u64), cp]
        L.itx_bam_header_parse.restype = vp
        L.itx_bam_header_parse.argtypes = [vp, vp, u64, C.c_int, cp]
        L.itx_bam_header_len.restype = u64
        L.itx_bam_header_len.argtypes = [vp]
        L.itx_bam_header_free.argtypes = [vp]
        L.itx_scan_bam_device.argtypes = [vp, vp, vp, u64, C.POINTER(ScanOpts), C.POINTER(u64), cp]
        L.itx_scan_cpg.argtypes = [vp, cp, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), cp]
        L.itx_sync_counts.argtypes = [vp, cp]
        L.itx_trace_enable.argtypes = [vp, u64]
        L.itx_trace_fetch.restype = u64
        L.itx_trace_fetch.argtypes = [vp, vp, u64]
        L.itx_query_select.argtypes = [vp, cp, vp, vp, C.c_int64, C.c_float, vp, vp, cp]
        L.itx_last_profile.argtypes = [vp, C.POINTER(Profile)]
        L.itx_tune.argtypes = [vp, C.c_uint32, u64, C.c_int32]
        L.itx_mark.argtypes = [vp, C.c_int]
        L.itx_elapsed_ms.restype = C.c_double
        L.itx_elapsed_ms.argtypes = [vp, C.c_int, C.c_int]
        L.itx_comm_unique_id.argtypes = [vp, cp]
        L.itx_comm_init.argtypes = [vp, vp, C.c_int, C.c_int, cp]
        L.itx_comm_allreduce_counts.argtypes = [vp, cp]
        L.itx_get_counters.argtypes = [vp, C.POINTER(u64)]
        L.itx_comm_destroy.argtypes = [vp]
        L.itx_dev_alloc.restype = vp
        L.itx_dev_alloc.argtypes = [u64]
        L.itx_dev_free.argtypes = [vp]
        L.itx_dev_upload.argtypes = [vp, vp, u64]
        L.itx_host_alloc_pinned.restype = vp
        L.itx_host_alloc_pinned.argtypes = [u64]
        L.itx_host_free_pinned.argtypes = [vp]
        L.itx_dev_flush_l2.argtypes = [vp]
        L.itx_wig_to_bigwig.argtypes = [cp, cp, cp, cp]
        L.itx_sam_to_bam.argtypes = [cp, C.POINTER(C.c_void_p), C.POINTER(u64), cp]
        L.itx_free.argtypes = [C.c_void_p]
        L.itx_free.restype = None
        L.itx_stream_fetch.restype = u64
        L.itx_stream_fetch.argtypes = [vp, vp, u64]
        _lib = L
    return _lib


class IndexBase:
    """Accessors and writers shared by the device index and the test emulator (same host structures)."""
    L = None
    h = None

    def sync(self):
        pass

    def write_stat(self, prefix, nindex=9, nindex2=10):
        self.sync()
        f = lambda s: (prefix + s).encode()
        rc = self.L.itx_write_stat(self.h, f(".iteres.subfamily.stat"), f(".iteres.wig"), f(".iteres.family.stat"),
                                   f(".iteres.class.stat"), f(".iteres.unique.wig"), self.cnt[nindex], self.cnt[nindex2])
        if rc:
            raise ItxError(rc, "itx_write_stat")

    def write_report(self, path, mapQ=10, subfam="ALL"):
        rc = self.L.itx_write_report(path.encode(), self.cnt, mapQ, subfam.encode())
        if rc:
            raise ItxError(rc, "itx_write_report")

    def write_filter(self, path, readlist=0, threshold=1, nindex=7):
        self.sync()
        rc = self.L.itx_write_filter(self.h, path.encode(), readlist, threshold, self.cnt[nindex])
        if rc:
            raise ItxError(rc, "itx_write_filter")

    def write_cpg_stat(self, prefix):
        self.sync()
        f = lambda s: (prefix + s).encode()
        rc = self.L.itx_write_cpg_stat(self.h, f(".CpG.subfamily.stat"), f(".CpGstat.wig"), f(".CpG.family.stat"), f(".CpG.class.stat"))
        if rc:
            raise ItxError(rc, "itx_write_cpg_stat")

    def write_cpg_filter(self, path, thr=0.0):
        self.sync()
        rc = self.L.itx_write_cpg_filter(self.h, path.encode(), thr)
        if rc:
            raise ItxError(rc, "itx_write_cpg_filter")

    def n(self, which):
        return [self.L.itx_n_subfam, self.L.itx_n_fam, self.L.itx_n_class][which](self.h)

    def table(self, which):
        """[(name, read_count, unique, total_length, genome_count)] in output-row order."""
        self.sync()
        out = []
        c = (C.c_uint64 * 4)()
        for i in range(self.n(which)):
            self.L.itx_counts(self.h, which, i, c)
            out.append((self.L.itx_name(self.h, which, i).decode(),) + tuple(c))
        return out

    def coverage(self, i, unique=0):
        import numpy as np
        self.sync()
        n = self.L.itx_subfam_length(self.h, i)
        if n == 0:
            return np.zeros(0, dtype=np.uint32)
        return np.ctypeslib.as_array(self.L.itx_subfam_bp(self.h, i, unique), shape=(n,)).copy()

    def elem_counts_by_row(self, unique=0):
        import numpy as np
        self.sync()
        n = self.L.itx_n_rows(self.h)
        p = self.L.itx_elem_counts_by_row(self.h, unique)
        return np.ctypeslib.as_array(p, shape=(n,)).copy() if n else np.zeros(0, dtype=np.uint32)


class Index(IndexBase):
    """itx_index: built from the three text tables, lives on one CUDA device."""

    def __init__(self, chrom_sizes, rep_sizes, rmsk, filter_field=0, filter_name="ALL", device=None):
        self.L = lib()
        err = C.create_string_buffer(ERRLEN)
        if device is not None:
            self.L.itx_set_device(device)      # the process-wide default too: itx_dev_alloc / itx_host_alloc_pinned follow it
            self.h = self.L.itx_index_build_on(device, chrom_sizes.encode(), rep_sizes.encode(), rmsk.encode(), filter_field,
                                               filter_name.encode(), err)
        else:
            self.h = self.L.itx_index_build(chrom_sizes.encode(), rep_sizes.encode(), rmsk.encode(), filter_field,
                                            filter_name.encode(), err)
        if not self.h:
            raise ItxError(-1, err.value.decode())
        self.cnt = (C.c_uint64 * 13)()
        self._dirty = True

    def close(self):
        if self.h:
            self.L.itx_index_free(self.h)
            self.h = None

    def _ck(self, rc, err):
        self._dirty = True
        if rc:
            raise ItxError(rc, err.value.decode())

    def reset(self):
        self.L.itx_index_reset_counts(self.h)
        self._dirty = True

    def tune(self, chunk_bytes=0, window_bytes=0, inflate_threads=0):
        rc = self.L.itx_tune(self.h, chunk_bytes, window_bytes, inflate_threads)
        if rc:
            raise ItxError(rc, "itx_tune: bad value")

    def scan_alignments(self, bam_list, opts):
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_alignments(self.h, bam_list.encode(), C.byref(opts), self.cnt, err), err)
        return list(self.cnt)

    def scan_alignment_file(self, path, opts):
        """the single-file twin (what `iteres filter` calls): the path is not split at commas"""
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_alignment_file(self.h, path.encode(), C.byref(opts), self.cnt, err), err)
        return list(self.cnt)

    def scan_shard_file(self, path, opts, rank, nranks, entry=SHARD_GUESS):
        """rank `rank` of `nranks` scans its block range of ONE file -> (counters so far, (entry_rel, exit_rel, own_bytes))"""
        err = C.create_string_buffer(ERRLEN)
        rep = ShardReport()
        self._ck(self.L.itx_scan_shard_file(self.h, path.encode(), C.byref(opts), rank, nranks, entry, C.byref(rep), self.cnt, err), err)
        return list(self.cnt), (rep.entry_rel, rep.exit_rel, rep.own_bytes)

    def shard_dedup_keys(self, path, opts, rank, nranks, entry=SHARD_GUESS):
        """-R across ranks, phase 1: settle the part and collect its unique fragments' keys, counting nothing
        -> ((entry_rel, exit_rel, own_bytes), n_keys, flags)"""
        err = C.create_string_buffer(ERRLEN)
        rep, n, fl = ShardReport(), C.c_uint64(0), C.c_uint32(0)
        self._ck(self.L.itx_shard_dedup_keys(self.h, path.encode(), C.byref(opts), rank, nranks, entry, C.byref(rep), C.byref(n), C.byref(fl), err), err)
        return (rep.entry_rel, rep.exit_rel, rep.own_bytes), n.value, fl.value

    def shard_dedup_fetch(self, n_keys):
        """the keys phase 1 collected, as an (n, 2) uint64 array (lo, hi), in no particular order"""
        import numpy as np
        a = np.empty((max(int(n_keys), 1), 2), dtype=np.uint64)
        got = self.L.itx_shard_dedup_fetch(self.h, a.ctypes.data, int(n_keys))
        return a[:got].copy()

    def dedup_admit(self, keys, flags):
        """enter other parts' keys ((n, 2) uint64) and flags into this index's -R table with one freshly reserved ordinal"""
        import numpy as np
        k = np.ascontiguousarray(keys, dtype=np.uint64).reshape(-1, 2)
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_dedup_admit(self.h, k.ctypes.data if len(k) else None, len(k), flags, err), err)

    def scan_shard_file_rmdup(self, path, opts, rank, nranks, entry):
        """-R across ranks, phase 2: count the part phase 1 settled (entry: its settled entry_rel) -> (counters so far, report)"""
        err = C.create_string_buffer(ERRLEN)
        rep = ShardReport()
        self._ck(self.L.itx_scan_shard_file_rmdup(self.h, path.encode(), C.byref(opts), rank, nranks, entry, C.byref(rep), self.cnt, err), err)
        return list(self.cnt), (rep.entry_rel, rep.exit_rel, rep.own_bytes)

    def scan_alignments_shard(self, bam_list, opts):
        """the whole protocol (scan, NCCL all-gather of the reports, re-scan where the chain check says so); rank / size from comm_init"""
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_alignments_shard(self.h, bam_list.encode(), C.byref(opts), self.cnt, err), err)
        return list(self.cnt)

    def scan_cpg_shard(self, path, rank, nranks, filter=0):
        a, b = C.c_uint32(0), C.c_uint32(0)
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_cpg_shard(self.h, path.encode(), filter, rank, nranks, C.byref(a), C.byref(b), err), err)
        return a.value, b.value

    def cpg_totals(self):
        a, b = C.c_uint64(0), C.c_uint64(0)
        self.L.itx_get_cpg_totals(self.h, C.byref(a), C.byref(b))
        return a.value, b.value

    def scan_bgzf_memory(self, ptr, nbytes, opts):
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_bgzf_memory(self.h, ptr, nbytes, C.byref(opts), self.cnt, err), err)
        return list(self.cnt)

    def scan_bam_host(self, ptr, nbytes, opts):
        """ptr: address of the uncompressed BAM stream in host memory (>= nbytes readable)."""
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_bam_host(self.h, ptr, nbytes, C.byref(opts), self.cnt, err), err)
        return list(self.cnt)

    def scan_stream(self, buf, opts, trace=False):
        """buf: bytes-like uncompressed BAM; mirrors OracleIndex.scan_stream."""
        import numpy as np
        a = np.frombuffer(buf, dtype=np.uint8)
        cap = max(1, len(a) // 36)
        self.L.itx_trace_enable(self.h, cap if trace else 0)
        cnt = self.scan_bam_host(a.ctypes.data, len(a), opts)
        if trace:
            t = (Trace * cap)()
            n = self.L.itx_trace_fetch(self.h, C.cast(t, C.c_void_p), cap)
            self.L.itx_trace_enable(self.h, 0)
            return cnt, np.ctypeslib.as_array(t)[:n].copy() if n else np.zeros(0, dtype=np.dtype(Trace))
        return cnt

    def header(self, host_ptr, nbytes, addChr=0):
        err = C.create_string_buffer(ERRLEN)
        h = self.L.itx_bam_header_parse(self.h, host_ptr, nbytes, addChr, err)
        if not h:
            raise ItxError(-2, err.value.decode())
        return h

    def scan_bam_device(self, hdr, dev_ptr, nbytes, opts):
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_bam_device(self.h, hdr, dev_ptr, nbytes, C.byref(opts), self.cnt, err), err)
        return list(self.cnt)

    def scan_cpg(self, path, filter=0):
        a, b = C.c_uint32(0), C.c_uint32(0)
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_scan_cpg(self.h, path.encode(), filter, C.byref(a), C.byref(b), err), err)
        return a.value, b.value

    def sync(self):
        if self._dirty:
            err = C.create_string_buffer(ERRLEN)
            rc = self.L.itx_sync_counts(self.h, err)
            if rc:
                raise ItxError(rc, err.value.decode())
            self._dirty = False

    def mark(self, slot):
        self.L.itx_mark(self.h, slot)

    def elapsed_ms(self, a, b):
        return self.L.itx_elapsed_ms(self.h, a, b)

    def stream_fetch(self, nbytes):
        """test hook: the uncompressed stream the last BGZF / host scan left on the device, as bytes"""
        import numpy as np
        a = np.empty(max(int(nbytes), 1), dtype=np.uint8)
        n = self.L.itx_stream_fetch(self.h, a.ctypes.data, int(nbytes))
        return a[:n].tobytes()

    def profile(self):
        p = Profile()
        self.L.itx_last_profile(self.h, C.byref(p))
        return p.as_dict()

    def query_select(self, chrom, starts, ends, min_cov=1e-4):
        import numpy as np
        s = np.ascontiguousarray(starts, dtype=np.uint32)
        e = np.ascontiguousarray(ends, dtype=np.uint32)
        sel = np.empty(len(s), dtype=np.int32)
        nh = np.empty(len(s), dtype=np.int32)
        err = C.create_string_buffer(ERRLEN)
        rc = self.L.itx_query_select(self.h, chrom.encode(), s.ctypes.data, e.ctypes.data, len(s), min_cov,
                                     sel.ctypes.data, nh.ctypes.data, err)
        if rc:
            raise ItxError(rc, err.value.decode())
        return sel, nh

    # multi-GPU
    def comm_unique_id(self):
        buf = (C.c_uint8 * 128)()
        err = C.create_string_buffer(ERRLEN)
        rc = self.L.itx_comm_unique_id(buf, err)
        if rc:
            raise ItxError(rc, err.value.decode())
        return bytes(buf)

    def comm_init(self, uid, rank, nranks):
        buf = (C.c_uint8 * 128).from_buffer_copy(uid)
        err = C.create_string_buffer(ERRLEN)
        rc = self.L.itx_comm_init(self.h, buf, rank, nranks, err)
        if rc:
            raise ItxError(rc, err.value.decode())

    def allreduce_counts(self):
        err = C.create_string_buffer(ERRLEN)
        self._ck(self.L.itx_comm_allreduce_counts(self.h, err), err)
        self.L.itx_get_counters(self.h, self.cnt)
        return list(self.cnt)
