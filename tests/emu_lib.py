"""ctypes binding of the TEST-ONLY host emulation of the device logic (tests/emu/libitx_emu.so):
iteres_b200/csrc/itx_logic.cuh compiled by g++ and driven sequentially.  Lets the non-GPU suite
check the per-record logic, the chunked boundary discovery and the writers against the oracle."""
import ctypes as C
import os

import numpy as np

from iteres_b200 import capi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "emu", "libitx_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        L = capi.bind(C.CDLL(LIB_PATH))
        vp, cp, u64 = C.c_void_p, C.c_char_p, C.c_uint64
        L.emu_build.restype = vp
        L.emu_build.argtypes = [cp, cp, cp, C.c_int, cp, cp]
        L.emu_free.argtypes = [vp]
        L.emu_reset.argtypes = [vp]
        L.emu_host_index.restype = vp
        L.emu_host_index.argtypes = [vp]
        L.emu_scan_stream.argtypes = [vp, vp, u64, C.POINTER(capi.ScanOpts), C.c_uint32, C.c_int, C.POINTER(u64), cp]
        L.emu_sync.argtypes = [vp]
        L.emu_trace.restype = u64
        L.emu_trace.argtypes = [vp, vp, u64]
        L.emu_n_bad.restype = u64
        L.emu_n_bad.argtypes = [vp]
        L.emu_scan_shard.argtypes = [vp, vp, u64, vp, u64, u64, u64, C.POINTER(capi.ScanOpts), C.c_uint32, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), cp]
        for f in ("emu_ring_checked", "emu_ring_mismatch", "emu_tile_checked", "emu_tile_mismatch", "emu_tile_entry_miss", "emu_xa_checked", "emu_xa_mismatch"):
            getattr(L, f).restype = u64
            getattr(L, f).argtypes = [vp]
        L.emu_xa_fast.restype = u64
        L.emu_xa_fast.argtypes = [C.c_int]
        L.emu_xa_fuzz.restype = u64
        L.emu_xa_fuzz.argtypes = [vp, u64, u64]
        L.emu_check_cov_rules.restype = C.c_uint64
        L.emu_check_cov_rules.argtypes = [C.c_uint64, C.c_uint64]
        L.emu_query.restype = C.c_int32
        L.emu_query.argtypes = [vp, cp, C.c_uint32, C.c_uint32, C.c_float, C.POINTER(C.c_int32)]
        L.emu_inflate.argtypes = [vp, C.c_uint32, vp, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.c_int]
        L.emu_strtod.restype = C.c_double
        L.emu_strtod.argtypes = [cp, C.POINTER(C.c_int)]
        L.emu_scan_cpg.argtypes = [vp, cp, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), cp]
        _lib = L
    return _lib


class EmuIndex(capi.IndexBase):
    def __init__(self, chrom_sizes, rep_sizes, rmsk, filter_field=0, filter_name="ALL", chunk=4096):
        self.L = lib()
        err = C.create_string_buffer(256)
        self.e = self.L.emu_build(chrom_sizes.encode(), rep_sizes.encode(), rmsk.encode(), filter_field, filter_name.encode(), err)
        if not self.e:
            raise capi.ItxError(-1, err.value.decode())
        self.h = self.L.emu_host_index(self.e)
        self.cnt = (C.c_uint64 * 13)()
        self.chunk = chunk
        self._dirty = True

    def close(self):
        if self.e:
            self.L.emu_free(self.e)
            self.e = None

    def reset(self):
        self.L.emu_reset(self.e)
        self._dirty = True

    def sync(self):
        if self._dirty:
            self.L.emu_sync(self.e)
            self._dirty = False

    def scan_stream(self, buf, opts, trace=False):
        a = np.frombuffer(bytes(buf) + b"\0" * 64, dtype=np.uint8)       # the device buffers carry 64 B of slack too
        n = len(a) - 64
        err = C.create_string_buffer(256)
        self._dirty = True
        rc = self.L.emu_scan_stream(self.e, a.ctypes.data, n, C.byref(opts), self.chunk, 1 if trace else 0, self.cnt, err)
        if rc:
            raise capi.ItxError(rc, err.value.decode())
        if trace:
            cap = max(1, n // 36)
            t = (capi.Trace * cap)()
            k = self.L.emu_trace(self.e, C.cast(t, C.c_void_p), cap)
            return list(self.cnt), (np.ctypeslib.as_array(t)[:k].copy() if k else np.zeros(0, dtype=np.dtype(capi.Trace)))
        return list(self.cnt)

    def scan_shard(self, header_buf, part, own, carry0, opts):
        """one rank's part of a stream: `part` = the rank's own bytes [0, own) followed by its margin; header_buf = the start of the
        whole stream (for the BAM header); carry0 = GUESS or a forced entry.  Returns (counters, entry_rel, exit_rel)."""
        hb = np.frombuffer(bytes(header_buf) + b"\0" * 64, dtype=np.uint8)
        a = np.frombuffer(bytes(part) + b"\0" * 64, dtype=np.uint8)
        err = C.create_string_buffer(256)
        en, ex = C.c_uint64(0), C.c_uint64(0)
        self._dirty = True
        rc = self.L.emu_scan_shard(self.e, hb.ctypes.data, len(hb) - 64, a.ctypes.data, len(a) - 64, own, carry0, C.byref(opts), self.chunk, self.cnt,
                                   C.byref(en), C.byref(ex), err)
        if rc:
            raise capi.ItxError(rc, err.value.decode())
        return list(self.cnt), en.value, ex.value

    def xa_check(self):
        """(reads with XA put through k_scan's lane-per-alternate decomposition, verdicts that differed from the one-lane walk)"""
        return self.L.emu_xa_checked(self.e), self.L.emu_xa_mismatch(self.e)

    def xa_fast(self):
        """(pieces of XA lists that took itx_xa_piece_fast's register path, pieces it handed to the general parser) -- process-wide"""
        return self.L.emu_xa_fast(0), self.L.emu_xa_fast(1)

    def xa_fuzz(self, seed, n):
        """itx_xa_piece_fast against itx_xa_piece on n generated alternates: the number of pieces they disagree on"""
        return self.L.emu_xa_fuzz(self.e, seed, n)

    def n_bad(self):
        return self.L.emu_n_bad(self.e)

    def ring_check(self):
        """(records re-decoded out of the shared-memory ring layout, mismatches against the global-memory decode)"""
        return self.L.emu_ring_checked(self.e), self.L.emu_ring_mismatch(self.e)

    def tile_check(self):
        """(chunks put through the warp kernel's lane-parallel chain, chunks whose record list differed from the
        sequential chain although the entry was right, chunks whose entry guess was wrong)"""
        return self.L.emu_tile_checked(self.e), self.L.emu_tile_mismatch(self.e), self.L.emu_tile_entry_miss(self.e)

    def scan_cpg(self, path, filter=0):
        a, b = C.c_uint32(0), C.c_uint32(0)
        err = C.create_string_buffer(256)
        self._dirty = True
        rc = self.L.emu_scan_cpg(self.e, path.encode(), filter, C.byref(a), C.byref(b), err)
        if rc:
            raise capi.ItxError(rc, err.value.decode())
        return a.value, b.value

    def query(self, chrom, start, end, min_cov=1e-4):
        n = C.c_int32(0)
        sel = self.L.emu_query(self.e, chrom.encode(), start, end, min_cov, C.byref(n))
        return sel, n.value


def inflate(raw_deflate, expect_len, cap=None, defer=1):
    """one raw-deflate stream through the device inflater (host build) -> (status, bytes).  defer=1 is the
    two-pass mode the device runs (matches listed, then resolved in warp-sized batches), defer=0 copies in line, defer=2 resolves
    by pointer jumping, defer=3..8 in the windows of itx_lzw_resolve (8192, 2048, 256, and the device's 6144, 3072, 1536 bytes)."""
    cap = expect_len if cap is None else cap
    src = np.frombuffer(bytes(raw_deflate), dtype=np.uint8)
    dst = np.zeros(max(cap, 1), dtype=np.uint8)
    got = C.c_uint32(0)
    rc = lib().emu_inflate(src.ctypes.data if len(src) else None, len(src), dst.ctypes.data, cap, expect_len, C.byref(got), defer)
    return rc, dst[: min(got.value, cap)].tobytes()


def strtod_fast(text):
    """the device's score parser (host build) -> (value, exact)"""
    ex = C.c_int(0)
    v = lib().emu_strtod(text.encode(), C.byref(ex))
    return v, bool(ex.value)
