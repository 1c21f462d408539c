"""-R across ranks on the CPU: the host emulation of the device logic runs the protocol of itx_scan_alignments_shard with -R over
byte ranges of ONE record stream (cut at arbitrary positions, as tests/test_shards_gloo.py cuts them), the ranks taken in turn in
one process.  Phase 1 settles every part and collects its unique fragments' keys, the keys and flags of the parts before a rank are
admitted with one ordinal below all of its own, the part is counted with -R, the keys of the parts after it are admitted -- and the
summed counters, tables and coverage are those of the single-pass -R scan of the whole stream.  This checks the ordinal and flag
arithmetic without a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import emu_lib
import synth
from iteres_b200 import capi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """the emulator with key export and admission (tests/emu/itx_emu_shard.cpp), built as tests/emu/Makefile builds the emulator"""
    d = str(tmp_path_factory.mktemp("emu_shard"))
    host, emu, so = (os.path.join(d, n) for n in ("itx_host_emu.o", "itx_emu_shard.o", "libitx_emu_shard.so"))
    subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-c", "-o", host, os.path.join(ROOT, "iteres_b200", "csrc", "itx_host.c")], check=True)
    subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-Wno-unknown-pragmas", "-fPIC", "-x", "c++", "-c", "-o", emu,
                    os.path.join(HERE, "emu", "itx_emu_shard.cpp")], check=True)
    subprocess.run([os.environ.get("CXX", "g++"), "-shared", "-o", so, emu, host], check=True)
    lib = capi.bind(C.CDLL(so))
    vp, cp, u64 = C.c_void_p, C.c_char_p, C.c_uint64
    lib.emu_build.restype = vp
    lib.emu_build.argtypes = [cp, cp, cp, C.c_int, cp, cp]
    lib.emu_free.argtypes = [vp]
    lib.emu_reset.argtypes = [vp]
    lib.emu_host_index.restype = vp
    lib.emu_host_index.argtypes = [vp]
    lib.emu_sync.argtypes = [vp]
    lib.emu_scan_stream.argtypes = [vp, vp, u64, C.POINTER(capi.ScanOpts), C.c_uint32, C.c_int, C.POINTER(u64), cp]
    lib.emu_scan_shard.argtypes = [vp, vp, u64, vp, u64, u64, u64, C.POINTER(capi.ScanOpts), C.c_uint32, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), cp]
    lib.emu_part_dedup_keys.argtypes = [vp, vp, u64, vp, u64, u64, u64, C.POINTER(capi.ScanOpts), C.c_uint32,
                                        C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_uint32), cp]
    lib.emu_part_dedup_fetch.restype = u64
    lib.emu_part_dedup_fetch.argtypes = [vp, vp, u64]
    lib.emu_dedup_admit.argtypes = [vp, vp, u64, C.c_uint32]
    return lib


class Emu(emu_lib.EmuIndex):
    """an emulator index of the library above (the accessors and scans of EmuIndex, on that library)"""

    def __init__(self, L, tabs, chunk=4096):
        self.L = L
        err = C.create_string_buffer(256)
        self.e = L.emu_build(*(t.encode() for t in tabs), 0, b"ALL", err)
        if not self.e:
            raise capi.ItxError(-1, err.value.decode())
        self.h = L.emu_host_index(self.e)
        self.cnt = (C.c_uint64 * 13)()
        self.chunk = chunk
        self._dirty = True


def _buf(b):
    return np.frombuffer(bytes(b) + b"\0" * 64, dtype=np.uint8)


def dedup_keys(scratch, header_buf, part, own, carry0, opts):
    """phase 1 of one part, on the scratch index -> (entry_rel, exit_rel, keys as an (n, 2) uint64 array, flags)"""
    L = scratch.L
    hb, a = _buf(header_buf), _buf(part)
    en, ex, n, fl = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)
    err = C.create_string_buffer(256)
    rc = L.emu_part_dedup_keys(scratch.e, hb.ctypes.data, len(hb) - 64, a.ctypes.data, len(a) - 64, own, carry0, C.byref(opts), scratch.chunk,
                               C.byref(en), C.byref(ex), C.byref(n), C.byref(fl), err)
    if rc:
        raise capi.ItxError(rc, err.value.decode())
    keys = np.zeros((max(n.value, 1), 2), dtype=np.uint64)
    got = L.emu_part_dedup_fetch(scratch.e, keys.ctypes.data, n.value)
    assert got == n.value
    return en.value, ex.value, keys[:got].copy(), fl.value


def admit(ix, keys, flags):
    k = np.ascontiguousarray(keys, dtype=np.uint64).reshape(-1, 2)
    ix.L.emu_dedup_admit(ix.e, k.ctypes.data if len(k) else None, len(k), flags)
    ix._dirty = True


def run_file(ixs, scratch, raw, hdr_len, cuts, opts, exchange=True):
    """one file of a run across len(ixs) ranks: phase 1 (on `scratch`) with the chain check, the exchange, phase 2.  -> the exported keys
    per part"""
    world, n = len(ixs), len(raw)
    parts = [raw[cuts[r]:min(n, cuts[r + 1] + 4096)] for r in range(world)]
    owns = [cuts[r + 1] - cuts[r] for r in range(world)]
    carry = [hdr_len] + [capi.SHARD_GUESS] * (world - 1)
    p1 = [dedup_keys(scratch, raw[:hdr_len + 64], parts[r], owns[r], carry[r], opts) for r in range(world)]
    for _ in range(world + 2):
        bad, forced = capi.shard_chain_check([(p[0], p[1], owns[r]) for r, p in enumerate(p1)], scratch.L)
        if bad < 0:
            break
        carry[bad] = forced
        p1[bad] = dedup_keys(scratch, raw[:hdr_len + 64], parts[bad], owns[bad], forced, opts)
    else:
        raise AssertionError("the parts do not chain")
    keys = [p[2] for p in p1]
    for r in range(world):
        before = [k for k in keys[:r] if len(k)]
        after = [k for k in keys[r + 1:] if len(k)]
        if exchange:
            admit(ixs[r], np.concatenate(before) if before else np.zeros((0, 2), np.uint64), int(np.bitwise_or.reduce([p[3] for p in p1[:r]] + [0])))
        entry = hdr_len if r == 0 else p1[r][0]
        if r == 0 or entry < capi.SHARD_GUESS:
            ixs[r].scan_shard(raw[:hdr_len + 64], parts[r], owns[r], entry, opts)
        if exchange:
            admit(ixs[r], np.concatenate(after) if after else np.zeros((0, 2), np.uint64), int(np.bitwise_or.reduce([p[3] for p in p1[r + 1:]] + [0])))
    return keys


def summed(ixs):
    cnt = [sum(int(ix.cnt[k]) for ix in ixs) for k in range(13)]
    tabs = [[(rows[0][i][0],) + tuple(sum(r[i][k] for r in rows) for k in (1, 2)) for i in range(len(rows[0]))]
            for rows in ([ix.table(w) for ix in ixs] for w in range(3))]
    cov = [sum(ix.coverage(i, u).astype(np.uint64) for ix in ixs) & 0xffffffff for i in range(ixs[0].n(0)) for u in (0, 1)]
    return cnt, tabs, cov


def whole(ref):
    return list(ref.cnt), [[row[:3] for row in ref.table(w)] for w in range(3)], [ref.coverage(i, u) for i in range(ref.n(0)) for u in (0, 1)]


def assert_same(got, want):
    assert got[0] == want[0]
    assert got[1] == want[1]
    assert all(np.array_equal(a.astype(np.uint32), b) for a, b in zip(got[2], want[2]))


@pytest.mark.parametrize("world", [2, 3, 5])
@pytest.mark.parametrize("shape,mode,n_rmsk,n_units", [(2, 0, 3000, 12000), (1, 2, 30000, 12000)], ids=["chrM_se50", "pe100"])
def test_rmdup_parts_equal_the_whole_stream(L, shape, mode, n_rmsk, n_units, world, tmp_path):
    d = str(tmp_path)
    s = synth.Synth(shape, n_rmsk, seed=31)
    tabs = s.write_tables(d)
    buf, n, nrec = s.stream(mode, n_units)
    hdr_len = len(s.header())
    raw = buf[:n].tobytes()
    raw += raw[hdr_len:]                  # the reads twice over: every key has copies far apart, in other parts than its first
    n = len(raw)
    opts = capi.default_opts(rmDup=1)
    ref = Emu(L, tabs)
    ref.scan_stream(raw, opts)
    want = whole(ref)
    scratch = Emu(L, tabs)
    plain = Emu(L, tabs)
    assert plain.scan_stream(raw, capi.default_opts())[11] > want[0][11] > 0          # -R drops reads in this stream
    for cut_seed in range(3):
        rng = np.random.RandomState(200 + cut_seed)
        cuts = [0] + sorted(int(x) for x in rng.randint(hdr_len + 1, n, size=world - 1)) + [n]
        ixs = [Emu(L, tabs) for _ in range(world)]
        keys = run_file(ixs, scratch, raw, hdr_len, cuts, opts)
        assert_same(summed(ixs), want)
        # the exchange matters: keys occur in more than one part, and without it the parts keep more reads
        allk = np.concatenate([k for k in keys if len(k)])
        assert len(np.unique(allk, axis=0)) < len(allk)
        alone = [Emu(L, tabs) for _ in range(world)]
        run_file(alone, scratch, raw, hdr_len, cuts, opts, exchange=False)
        assert summed(alone)[0][11] > want[0][11]
        for ix in ixs + alone:
            ix.close()
    ref.close(); plain.close(); scratch.close()


def test_rmdup_keys_persist_across_the_files_of_a_run(L, tmp_path):
    """a list of two files (the same stream twice, then two different ones) on 3 ranks: the second file's parts find every key of
    the first in their tables"""
    d = str(tmp_path)
    s = synth.Synth(2, 3000, seed=32)
    tabs = s.write_tables(d)
    hdr_len = len(s.header())
    a, n_a, _ = s.stream(0, 8000)
    raw_a = a[:n_a].tobytes()
    b, n_b, _ = synth.Synth(2, 3000, seed=33).stream(0, 6000)
    raw_b = raw_a[:hdr_len] + b[hdr_len:n_b].tobytes()        # the same header (the same references), other reads
    opts = capi.default_opts(rmDup=1)
    scratch = Emu(L, tabs)
    for second in (raw_a, raw_b):
        ref = Emu(L, tabs)
        ref.scan_stream(raw_a, opts)
        ref.scan_stream(second, opts)
        want = whole(ref)
        ixs = [Emu(L, tabs) for _ in range(3)]
        for raw in (raw_a, second):
            rng = np.random.RandomState(len(raw))
            cuts = [0] + sorted(int(x) for x in rng.randint(hdr_len + 1, len(raw), size=2)) + [len(raw)]
            run_file(ixs, scratch, raw, hdr_len, cuts, opts)
        assert_same(summed(ixs), want)
        if second is raw_a:                    # the repeated file keeps none of its unique reads
            once = Emu(L, tabs)
            assert once.scan_stream(raw_a, opts)[11] == want[0][11] > 0
            once.close()
        for ix in ixs + [ref]:
            ix.close()
    scratch.close()
