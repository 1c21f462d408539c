#!/usr/bin/env python
"""A/B driver for one B200 (round 2): everything is built once (index, streams, BGZF file), then the library's
run-time switches are flipped in-process.  Prints one line per variant; counters must never move.
  python tools/ab_r2.py scan     k_scan flag variants on SE-50 / PE-100 / SE-75+XA, device-resident
  python tools/ab_r2.py e2e      BGZF -> tables: pinned image (itx_scan_bgzf_memory) and file (itx_scan_alignments), inflate variants
  python tools/ab_r2.py ncu      one launch per k_scan variant (to run under ncu --metrics ...)
"""
import ctypes as C
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import iteres_b200 as itx   # noqa: E402
import synth as S           # noqa: E402

what = sys.argv[1] if len(sys.argv) > 1 else "scan"
reads = int(os.environ.get("AB_READS", "50000000"))
L = itx.lib()
ncpu = os.cpu_count() or 8
t0 = time.perf_counter()
world = S.Synth(1, 5_500_000, seed=1)
wd = "/dev/shm/itx_ab"
os.makedirs(wd, exist_ok=True)
tables = world.write_tables(os.path.join(wd, "tables"))
ix = itx.Index(*tables, device=0)
print("index built %.1f s" % (time.perf_counter() - t0), flush=True)
opts = itx.default_opts()


def make_stream(mode, n_units):
    hdr = world.header()
    sz, nrec = world.records_size(mode, n_units, 0, None, ncpu)
    n = len(hdr) + sz
    hbuf = L.itx_host_alloc_pinned(n + 64)
    C.memmove(hbuf, hdr.ctypes.data, len(hdr))
    assert world.records_into(hbuf + len(hdr), mode, n_units, 0, None, ncpu) == sz
    C.memset(hbuf + n, 0, 64)
    return hbuf, n, nrec, len(hdr)


def resident(hbuf, n):
    dbuf = L.itx_dev_alloc(n + 64)
    assert dbuf and L.itx_dev_upload(dbuf, hbuf, n + 64) == 0
    return dbuf, ix.header(hbuf, n)


def time_scan(h, dbuf, n, steps=20, warm=3):
    for _ in range(warm):
        ix.reset(); cnt = ix.scan_bam_device(h, dbuf, n, opts)
    dec = 0.0
    ix.mark(0)
    for _ in range(steps):
        ix.reset(); cnt = ix.scan_bam_device(h, dbuf, n, opts)
        dec += ix.profile()["decode_ms"]
    ix.mark(1)
    L.itx_dev_sync()
    return dec / steps, ix.elapsed_ms(0, 1) / steps, cnt, ix.profile()["n_replayed_windows"]


def scan_variants(name, mode, n_units, variants, steps=20):
    hbuf, n, nrec, _ = make_stream(mode, n_units)
    dbuf, h = resident(hbuf, n)
    L.itx_host_free_pinned(hbuf)
    base = None
    for tag, env in variants:
        for k in ("ITX_SCAN_FLAGS", "ITX_L2_PERSIST"):
            os.environ.pop(k, None)
        os.environ.update(env)
        k_ms, step_ms, cnt, rep = time_scan(h, dbuf, n, steps)
        if base is None:
            base = cnt
        F, H, HU = cnt[6], cnt[9] + cnt[12], cnt[10]
        b_alg = n + 16 * F + 28 * H + 8 * HU
        print("%-10s %-22s k_scan %.3f ms  step %.3f ms  frac(8d) %.3f  frac(stream) %.3f  replays %d  same_counts %s  diffsub %d" % (
            name, tag, k_ms, step_ms, b_alg / k_ms / 1e6 / 6552.3, n / k_ms / 1e6 / 6552.3, rep, cnt == base, cnt[12]), flush=True)
    L.itx_bam_header_free(h)
    L.itx_dev_free(dbuf)


V_SCAN = [("r1 (15)", {"ITX_SCAN_FLAGS": "15"}), ("early (31)", {"ITX_SCAN_FLAGS": "31"}), ("default (95)", {}),
          ("evict (127)", {"ITX_SCAN_FLAGS": "127"}), ("evict+pf (255)", {"ITX_SCAN_FLAGS": "255"}),
          ("default+persist", {"ITX_L2_PERSIST": "1"}), ("evict+persist", {"ITX_SCAN_FLAGS": "127", "ITX_L2_PERSIST": "1"})]

if what == "scan":
    scan_variants("SE-50", 0, reads, V_SCAN)
    scan_variants("PE-100", 2, reads // 2, [V_SCAN[0], V_SCAN[2], V_SCAN[3], V_SCAN[6]])
    scan_variants("SE-75+XA", 1, reads * 3 // 5, [("r1 (15)", {"ITX_SCAN_FLAGS": "15"}), ("early,serial XA (31)", {"ITX_SCAN_FLAGS": "31"}), ("default (95)", {})], steps=5)
elif what == "xa":
    # the SE-75 + XA:Z stream (cfg 3's shape) through the product kernels: k_scan + k_xa per step
    scan_variants("SE-75+XA", 1, reads * 3 // 5, [("product", {})], steps=10)
elif what == "three":
    # the product kernels on the three record shapes (ITX_LIB selects a variant library)
    V = [("product", {})]
    scan_variants("SE-50", 0, reads, V, steps=20)
    scan_variants("PE-100", 2, reads // 2, V, steps=10)
    scan_variants("SE-75+XA", 1, reads * 3 // 5, V, steps=6)
elif what == "ncu1":
    # ONE launch of k_scan (after two warm-up launches) on the stream AB_MODE / AB_READS name, with the environment as it is
    mode = int(os.environ.get("AB_MODE", "0"))
    hbuf, n, nrec, _ = make_stream(mode, reads)
    dbuf, h = resident(hbuf, n)
    for _ in range(3):
        ix.reset(); cnt = ix.scan_bam_device(h, dbuf, n, opts)
    print("mode", mode, "records", nrec, "bytes", n, "counters", cnt, flush=True)
elif what == "ncu":
    hbuf, n, nrec, _ = make_stream(0, reads)
    dbuf, h = resident(hbuf, n)
    V_NCU = [("all switches (127)", {"ITX_SCAN_FLAGS": "127"}), ("no L2 prefetch (126)", {"ITX_SCAN_FLAGS": "126"}), ("no evict-first hint (95)", {"ITX_SCAN_FLAGS": "95"}),
             ("no early copy (111)", {"ITX_SCAN_FLAGS": "111"}), ("no table window (115)", {"ITX_SCAN_FLAGS": "115"}), ("evict hint on the prefetch too (255)", {"ITX_SCAN_FLAGS": "255"}),
             ("persisting window on the coverage arrays", {"ITX_SCAN_FLAGS": "127", "ITX_L2_PERSIST": "1"})]
    for tag, env in V_NCU:
        for k in ("ITX_SCAN_FLAGS", "ITX_L2_PERSIST"):
            os.environ.pop(k, None)
        os.environ.update(env)
        ix.reset(); ix.scan_bam_device(h, dbuf, n, opts)
        print("launched", tag, flush=True)
elif what == "tuple":
    # the tuple path (ITX_FUSED=0) at several sizes: decode / overlap device time per scan
    os.environ["ITX_FUSED"] = "0"
    for nr in ((reads,) if os.environ.get("AB_TUPLE_ONE") else (10_000_000, 20_000_000, 50_000_000)):
        hbuf, n, nrec, _ = make_stream(0, nr)
        dbuf, h = resident(hbuf, n)
        L.itx_host_free_pinned(hbuf)
        for _ in range(2):
            ix.reset(); ix.scan_bam_device(h, dbuf, n, opts)
        d = o = 0.0
        for _ in range(5):
            ix.reset(); cnt = ix.scan_bam_device(h, dbuf, n, opts)
            pr = ix.profile(); d += pr["decode_ms"] / 5; o += pr["overlap_ms"] / 5
        print("tuple path %d M reads: decode %.3f ms overlap %.3f ms launches %d" % (nr // 1_000_000, d, o, pr["n_launches"]), flush=True)
        L.itx_bam_header_free(h); L.itx_dev_free(dbuf)
elif what == "e2e1":
    # ONE BGZF scan from a pinned image (for ncu on k_inflate / k_lz_resolve); AB_READS sizes the file
    hbuf, n, nrec, hl = make_stream(0, reads)
    bam = os.path.join(wd, "reads1.bam")
    assert S.lib().synth_write_bam(bam.encode(), hbuf, hl, hbuf + hl, n - hl, 1, ncpu) == 0
    L.itx_host_free_pinned(hbuf)
    fsz = os.path.getsize(bam)
    pin = L.itx_host_alloc_pinned(fsz + 64)
    with open(bam, "rb") as f:
        assert f.readinto((C.c_char * fsz).from_address(pin)) == fsz
    for i in range(2):
        t = time.perf_counter()
        ix.reset(); got = ix.scan_bgzf_memory(pin, fsz, opts)
        print("scan %d: %.1f ms, %d records" % (i, 1e3 * (time.perf_counter() - t), got[0] + got[1]), flush=True)
elif what == "e2e":
    hbuf, n, nrec, hl = make_stream(0, reads)
    bam = os.path.join(wd, "reads.bam")
    assert S.lib().synth_write_bam(bam.encode(), hbuf, hl, hbuf + hl, n - hl, 1, ncpu) == 0
    dbuf, h = resident(hbuf, n)
    ix.reset(); want = ix.scan_bam_device(h, dbuf, n, opts)
    L.itx_dev_free(dbuf); L.itx_host_free_pinned(hbuf)
    fsz = os.path.getsize(bam)
    pin = L.itx_host_alloc_pinned(fsz + 64)
    with open(bam, "rb") as f:
        mv = (C.c_char * fsz).from_address(pin)
        assert f.readinto(mv) == fsz
    print("BGZF %.2f GB written and pinned" % (fsz / 1e9), flush=True)
    variants = [("in-warp windows (2)", {}), ("k_lz_resolve (0)", {"ITX_LZ": "0"}), ("windows, tail 4096x8", {"ITX_INF_TAIL_GROUP": "4096"}),
                ("windows, 16 lanes", {"ITX_INF_LANES": "16"}), ("windows, g8192", {"ITX_INF_GROUP": "8192"}), ("windows, g8192 tail 2048", {"ITX_INF_GROUP": "8192", "ITX_INF_TAIL_GROUP": "2048"})]
    if os.environ.get("AB_E2E_VARIANTS"):
        variants = [(v, dict(kv.split("=") for kv in v.split(",") if kv)) for v in os.environ["AB_E2E_VARIANTS"].split(";")]
    for tag, env in variants:
        for k in ("ITX_INF_LANES", "ITX_INF_TAIL_LANES", "ITX_INF_GROUP", "ITX_INF_TAIL_GROUP", "ITX_TIMING", "ITX_LZ"):
            os.environ.pop(k, None)
        os.environ.update(env)
        for api in (("pinned", "file") if tag == variants[0][0] or os.environ.get("AB_E2E_FILE") else ("pinned",)):
            ts = []
            for i in range(4):
                if i == 3 and api == "pinned":
                    os.environ["ITX_TIMING"] = "1"
                t = time.perf_counter()
                ix.reset()
                got = ix.scan_bgzf_memory(pin, fsz, opts) if api == "pinned" else ix.scan_alignments(bam, opts)
                ix._dirty = True
                ix.sync()
                ts.append(time.perf_counter() - t)
                os.environ.pop("ITX_TIMING", None)
            pr = ix.profile()
            print("e2e %-22s %-6s %s ms  inflate_ms %.1f  same_counts %s  -> %.0f M reads/s" % (
                tag, api, " ".join("%.1f" % (1e3 * x) for x in ts), pr["inflate_ms"], got == want, nrec / min(ts[1:]) / 1e6), flush=True)
ix.close()
