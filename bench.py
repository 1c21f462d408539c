#!/usr/bin/env python
"""bench.py -- the iteres hot path on B200: aligned reads/sec for `iteres stat` (rmsk overlap count).

One step = one complete pass of the hot path over the workload: reset counters -> k_scan (record boundaries, decode,
overlap, selection, accumulation in one kernel) (-> one NCCL allreduce of the counter block when N > 1) -> the 13 global
counters back on the host.

  value        reads/s with the uncompressed BAM stream already resident in HBM (kernels only)
  e2e          the same metric through the C-ABI call a caller makes with HOST buffers: itx_scan_bgzf_memory() on the BGZF
               .bam image in pinned host memory -> cudaMemcpyAsync windows -> k_inflate (BGZF blocks inflated
               on the device) -> k_scan -> counter tables back on the host (itx_sync_counts), all inside the timed region
  e2e_file     the same from a FILE through itx_scan_alignments() (what the `iteres` command line does): a reader thread
               pread()s the file into a ring of pinned slots first.  The file lives on tmpfs / in the page cache (/dev/shm)
  roofline     k_scan against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline the UNMODIFIED reference binary (oracle/_ref/iteres stat) on the box's host cores, on a bounded sample of
               the same workload (the reference is single threaded: P independent copies side by side, P = cores used)
  parity       the gate: the CUDA path's tables for the cpu_baseline sample BAMs are compared BYTE FOR BYTE with the tables
               the reference binary wrote for them; any difference -> exit status 3, no JSON line
  extra_configs  BASELINE.json's other configs, each with its own value, kernel time, roofline fraction and parity check on
               a bounded prefix: cfg 1 (1 M SE reads, chr1, 200 k rows), cfg 3 (SE-75 + XA: stat AND filter / per-locus
               tables), cfg 4 (cpgstat), cfg 5 (PE-100)

N = 1 workload: BASELINE.json configs[1] (50 M SE-50 reads, hg19-shaped, vs a 5.5 M row rmsk table).
N > 1: the headline stays weak scaling (every rank scans its own 50 M read genomic-coordinate shard, one allreduce per step);
beside it `strong_scaling` scans ONE coordinate-sorted PE-100 BGZF file of fixed size, split by BGZF block ranges inside the
product (itx_scan_alignments_shard: guessed first records, cross-rank chain check), and `parity_multi_gpu` compares the
N-rank tables of one small file with the reference binary's.
Data is synthetic (tools/itx_synth.c), generated on the box; nothing is read from /root/reference.
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "aligned reads/sec for iteres stat (rmsk overlap count); HBM GB/s vs peak"
UNIT = "reads/s"
DTYPE = "u32/u64 integer (f32 coverage ratio)"


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: NVML polled every few milliseconds from a thread
    (nvidia-smi -lms as the fallback), so that even a 50 ms region holds several samples."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.p, self.nvml, self.stop_flag, self.th = gpu, [], None, None, False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.p = None

    def _poll(self):
        n = self.nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                try:
                    r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), sm, self.max_sm, [k for k, b in bits.items() if r & b]))
            except Exception:
                pass
            time.sleep(0.004)

    def _pump(self):
        for line in self.p.stdout:
            r = [x.strip() for x in line.split(",")]
            if len(r) >= 9 and r[1].replace(".", "").isdigit():
                reasons = [nm for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]) if v.lower().startswith("active")]
                self.rows.append((time.perf_counter(), int(float(r[1])), int(float(r[2])), reasons))

    def wait_first(self, timeout=4.0):
        t0 = time.perf_counter()
        while not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def window(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=2)
        if self.p:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                pass
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", 1e30)
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        rows = inside or [r for r in self.rows if t0 - 0.15 <= r[0] <= t1 + 0.15] or self.rows
        sm = sorted(r[1] for r in rows)
        reasons = sorted({x for r in rows for x in r[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[2] for r in rows), default=None), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


def workdir():
    base = None
    for cand in ("/dev/shm", tempfile.gettempdir()):
        try:
            if shutil.disk_usage(cand).free > (40 << 30):
                base = cand
                break
        except Exception:
            pass
    base = base or tempfile.gettempdir()
    d = os.path.join(base, "itx_bench_%s" % os.environ.get("MASTER_PORT", str(os.getpid())))
    os.makedirs(d, exist_ok=True)
    return d


# ------------------------------------------------------------------------------------------ the checker (reference binary, else the oracle port)
class Checker:
    """Runs the reference's own command on an input, in the background, into `outdir`: the unmodified reference binary
    (oracle/_ref/iteres) when it has been built, else the C oracle port through tests/runners.py."""

    def __init__(self, cmd, args, tables, data, outdir):
        import oracle_lib as O
        self.cmd, self.args, self.outdir = cmd, list(args), outdir
        os.makedirs(outdir, exist_ok=True)
        self.kind = "reference" if os.path.exists(O.REF_BIN) else "port"
        self.err = None
        self.t0 = time.perf_counter()
        if self.kind == "reference":
            self.p = subprocess.Popen([O.REF_BIN, cmd, "-o", "out"] + self.args + list(tables) + [data], cwd=outdir, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            self.th = None
        else:
            inp = os.path.join(outdir, "inp")
            os.makedirs(inp, exist_ok=True)
            for src, name in zip(list(tables) + [data], ("chrom.sizes", "rep.sizes", "rmsk.txt", "cpg.bedGraph" if cmd.startswith("cpg") else "reads.bam")):
                dst = os.path.join(inp, name)
                if os.path.lexists(dst):
                    os.unlink(dst)
                os.symlink(src, dst)
            self.p = None
            self.th = threading.Thread(target=self._port, args=(inp,), daemon=True)
            self.th.start()

    def _port(self, inp):
        try:
            import runners
            runners.run_oracle(inp, self.cmd, self.args, self.outdir)
        except Exception as ex:      # noqa: BLE001
            self.err = ex

    def wait(self):
        if self.p is not None:
            rc = self.p.wait()
            if rc:
                raise SystemExit("bench.py: the reference binary failed (%s %s): exit %d" % (self.cmd, " ".join(self.args), rc))
        else:
            self.th.join()
            if self.err:
                raise SystemExit("bench.py: the oracle port failed: %s" % self.err)
        self.seconds = time.perf_counter() - self.t0
        return self.outdir


FILES = {"stat": ["out.iteres.subfamily.stat", "out.iteres.family.stat", "out.iteres.class.stat", "out.iteres.report"],
         "filter": ["out_ALL.iteres.loci", "out_ALL.iteres.reportloci"],
         "cpgstat": ["out.CpG.subfamily.stat", "out.CpG.family.stat", "out.CpG.class.stat"]}


def gpu_tables(ix, cmd, outdir, opts):
    """the product's writers for the counters `ix` holds now -> the same file names the reference uses"""
    os.makedirs(outdir, exist_ok=True)
    p = os.path.join(outdir, "out")
    if cmd == "stat":
        ix.write_stat(p, 9, 10)
        ix.write_report(p + ".iteres.report", opts.mapQ, "ALL")
    elif cmd == "filter":
        ix.write_filter(p + "_ALL.iteres.loci", 0, 1, 7)
        ix.write_report(p + "_ALL.iteres.reportloci", opts.mapQ, "ALL")
    elif cmd == "cpgstat":
        ix.write_cpg_stat(p)


def same_numbers(a, b, rtol):
    """text tables equal field by field: integers and names exactly, floating-point fields within rtol"""
    la, lb = a.decode().split("\n"), b.decode().split("\n")
    if len(la) != len(lb):
        return False
    for x, y in zip(la, lb):
        if x == y:
            continue
        fx, fy = x.split("\t"), y.split("\t")
        if len(fx) != len(fy):
            return False
        for u, v in zip(fx, fy):
            if u == v:
                continue
            try:
                fu, fv = float(u), float(v)
            except ValueError:
                return False
            if "." not in u and "e" not in u.lower() and "." not in v and "e" not in v.lower():
                return False                       # integers must be identical
            if abs(fu - fv) > rtol * max(abs(fu), abs(fv)) + 5.1e-5:       # + half a unit of the printed %.4f
                return False
    return True


def compare_tables(cmd, got_dir, want_dir, what, rtol=0.0):
    """byte for byte (rtol == 0) or, for the CpG score sums -- the one floating-point sum whose order differs -- within rtol"""
    for fn in FILES[cmd]:
        with open(os.path.join(got_dir, fn), "rb") as f:
            a = f.read()
        with open(os.path.join(want_dir, fn), "rb") as f:
            b = f.read()
        if a == b:
            continue
        if rtol and same_numbers(a, b, rtol):
            continue
        sys.stderr.write("[bench] PARITY FAILURE in %s: %s differs from the checker's\n" % (what, fn))
        la, lb = a.split(b"\n"), b.split(b"\n")
        for i, (x, y) in enumerate(zip(la, lb)):
            if x != y:
                sys.stderr.write("  line %d\n   ours: %r\n   ref : %r\n" % (i + 1, x[:200], y[:200]))
                break
        raise SystemExit(3)
    return len(FILES[cmd])


# ------------------------------------------------------------------------------------------ reference arm
def reference_baseline(wd, tables, synth_world, sample_reads, mode, procs, keep_outputs=False):
    """Time the unmodified reference (oracle/_ref/iteres stat) on `procs` host cores: each process scans its own sample
    BAM of sample_reads reads (same generator, same rmsk).  The fixed cost (rmsk parse, wig/bigWig writing) is measured
    with header-only BAMs and subtracted, so the figure is the read loop."""
    import oracle_lib as O
    import synth as S
    cs, rs, rm = tables
    kind = "reference" if os.path.exists(O.REF_BIN) else "port"
    hdr = synth_world.header()
    empty = os.path.join(wd, "empty.bam")
    S.lib().synth_write_bam(empty.encode(), hdr.ctypes.data, len(hdr), hdr.ctypes.data, 0, 1, 1)
    bams = sample_bams(wd, synth_world, sample_reads, mode, procs)

    def run_all(paths, tag):
        t0 = time.perf_counter()
        ps = []
        for i, b in enumerate(paths):
            od = os.path.join(wd, "ref_%s_%d" % (tag, i))
            os.makedirs(od, exist_ok=True)
            if kind == "reference":
                ps.append(subprocess.Popen([O.REF_BIN, "stat", "-o", "out", cs, rs, rm, b], cwd=od, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
            else:
                code = ("import sys; sys.path[:0]=[%r,%r]; import oracle_lib as O; ix=O.OracleIndex(%r,%r,%r); cnt=ix.scan_file(%r,O.default_opts()); ix.write_stat('out'); ix.write_report('out.iteres.report', 10, 'ALL')"
                        % (ROOT, os.path.join(ROOT, "tests"), cs, rs, rm, b))
                ps.append(subprocess.Popen([sys.executable, "-c", code], cwd=od, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
        rcs = [p.wait() for p in ps]
        dt = time.perf_counter() - t0
        if any(rcs):
            raise RuntimeError("reference run failed: %r" % rcs)
        return dt

    fixed = run_all([empty] * procs, "fixed")
    t_full = run_all(bams, "full")
    loop = max(t_full - fixed, 1e-6)
    return {"kind": kind, "cores": procs, "sample_reads": sample_reads * procs, "fixed_s": fixed, "wall_s": t_full, "loop_s": loop, "bams": bams,
            "out_dirs": [os.path.join(wd, "ref_full_%d" % i) for i in range(procs)],
            "sample": "%d x %d reads (same generator and rmsk table as the GPU arm, %s), one single-threaded `iteres stat` per core; "
                      "fixed cost (rmsk parse + wig/bigWig, header-only BAM) of %.1f s subtracted" % (procs, sample_reads, MODE_NAME[mode] + " hg19-shaped", fixed)}


def sample_bams(wd, synth_world, sample_reads, mode, procs):
    ncpu = os.cpu_count() or 8
    bams = []
    for i in range(procs):
        b = os.path.join(wd, "sample_m%d_%d.bam" % (mode, i))
        if not os.path.exists(b):
            keep = synth_world.seed
            synth_world.seed = 1000 + i          # same tables (built from the construction seed), different reads per process
            synth_world.write_bam(b, mode, sample_reads, level=1, threads=max(1, ncpu // 2))
            synth_world.seed = keep
        bams.append(b)
    return bams


MODE_NAME = {0: "SE-50", 1: "SE-75+XA", 2: "PE-100"}
_REAL_STDOUT = None


def emit(obj):
    """the ONE JSON line of the contract, on the process's original stdout"""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


class Resident:
    """a generated uncompressed stream: in pinned host memory, and (optionally) uploaded to the device"""

    def __init__(self, L, ix, world, mode, n_units, c0=0, c1=None, threads=8, upload=True):
        hdr = world.header()
        c1 = world.n_chunks(n_units) if c1 is None else c1
        sz, self.nrec = world.records_size(mode, n_units, c0, c1, threads)
        self.L, self.n, self.hl = L, len(hdr) + sz, len(hdr)
        self.hbuf = L.itx_host_alloc_pinned(self.n + 64)
        if not self.hbuf:
            raise SystemExit("pinned allocation of %d bytes failed" % (self.n + 64))
        C.memmove(self.hbuf, hdr.ctypes.data, len(hdr))
        got = world.records_into(self.hbuf + len(hdr), mode, n_units, c0, c1, threads)
        assert got == sz
        C.memset(self.hbuf + self.n, 0, 64)
        self.dbuf = None
        self.h = ix.header(self.hbuf, self.n)
        if upload:
            self.dbuf = L.itx_dev_alloc(self.n + 64)
            assert self.dbuf and L.itx_dev_upload(self.dbuf, self.hbuf, self.n + 64) == 0

    def write_bgzf(self, path, threads):
        import synth as S
        rc = S.lib().synth_write_bam(path.encode(), self.hbuf, self.hl, self.hbuf + self.hl, self.n - self.hl, 1, threads)
        assert rc == 0
        return os.path.getsize(path)

    def free_host(self):
        if self.hbuf:
            self.L.itx_host_free_pinned(self.hbuf)
            self.hbuf = None

    def free(self):
        self.free_host()
        if self.dbuf:
            self.L.itx_dev_free(self.dbuf)
            self.dbuf = None
        if self.h:
            self.L.itx_bam_header_free(self.h)
            self.h = None


def kscan_bytes(n, cnt):
    """SURVEY 8(d) bytes of one k_scan launch: the stream + 16 B per fragment (its probe) + 28 B per read that reaches the
    accumulation (16 B hit + 4 + 8 B of counters) + 8 B per unique one"""
    F, H, HU = cnt[6], cnt[9] + cnt[12], cnt[10]
    return n + 16 * F + 28 * H + 8 * HU


def timed_resident(ix, R, opts, steps, warmup, after=None):
    """(k_scan ms per step from the library's CUDA events, whole step ms between two marks on the scan stream, counters, launches)"""
    for _ in range(warmup):
        ix.reset(); cnt = ix.scan_bam_device(R.h, R.dbuf, R.n, opts)
        if after:
            after()
    ix.L.itx_dev_sync()
    dec = 0.0
    launches = 0
    ix.mark(2)
    for _ in range(steps):
        ix.reset(); cnt = ix.scan_bam_device(R.h, R.dbuf, R.n, opts)
        if after:
            after()
        pr = ix.profile()
        dec += pr["decode_ms"] + pr["overlap_ms"]; launches += pr["n_launches"]
    ix.mark(3)
    ix.L.itx_dev_sync()
    return dec / steps, ix.elapsed_ms(2, 3) / steps, cnt, launches


def dump_outputs(ix, cnt, outdir, budget=48 << 20):
    """What the last headline step handed its caller, as float64 .npy files (every value is an exact integer there): the 13
    counters, the subfamily / family / class tables (read count, unique, total length, genome count per row), the per-subfamily
    sums of both coverage vectors, and both coverage vectors at a fixed, seeded sample of positions of their concatenation
    (4.4 M bases each at the bench's table shape), so that the arrays stay under `budget` bytes."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    ix._dirty = True
    ix.sync()
    out = {"counters": np.array(cnt, dtype=np.float64)}
    for which, name in enumerate(("subfamily", "family", "class")):
        out[name + "_table"] = np.array([row[1:] for row in ix.table(which)], dtype=np.float64).reshape(-1, 4)
    cov = [[ix.coverage(i, u) for i in range(ix.n(0))] for u in (0, 1)]
    out["coverage_sums"] = np.array([[int(c.sum(dtype=np.uint64)) for c in cov[u]] for u in (0, 1)], dtype=np.float64).T
    cov = [np.concatenate(c) for c in cov]
    n_sample = min(len(cov[0]), (budget - sum(a.nbytes for a in out.values())) // 24)
    idx = np.sort(np.random.default_rng(20240501).choice(len(cov[0]), n_sample, replace=False))
    out["coverage_sample_index"] = idx.astype(np.float64)
    out["coverage_all_sample"] = cov[0][idx].astype(np.float64)
    out["coverage_unique_sample"] = cov[1][idx].astype(np.float64)
    for name, arr in out.items():
        np.save(os.path.join(outdir, name + ".npy"), arr)
    log("outputs of the last timed step: %s (%.1f MB)" % (outdir, sum(a.nbytes for a in out.values()) / 1e6))


def main():
    # libraries (NCCL prints its version banner with some NCCL_DEBUG settings) must not add lines to stdout: everything
    # written to fd 1 during the run goes to stderr; the JSON line is written to a duplicate of the original stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=50_000_000, help="reads per GPU (BASELINE configs[1])")
    ap.add_argument("--rmsk", type=int, default=5_500_000)
    ap.add_argument("--mode", type=int, default=0, help="0 SE-50 (configs[1]), 1 SE-75 + XA, 2 PE-100")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-sample", type=int, default=2_000_000, help="reads per reference process in the CPU baseline")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra_configs / strong scaling (A/B runs)")
    ap.add_argument("--strong-pairs", type=int, default=40_000_000, help="PE-100 pairs in the ONE file of the strong-scaling pass (N > 1)")
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--window", type=int, default=0)
    ap.add_argument("--keep", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float64, about 50 MB in all)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; --impl reference does not run it")
    rank, world, lrank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if a.warmup < 3 and a.impl == "ours":
        log("note: fewer than 3 warm-up steps requested")
    ncpu = os.cpu_count() or 8
    import synth as S
    wd = workdir()
    shape = 1
    workload = "iteres stat, %d M %s reads per GPU, hg19-shaped, vs %.1f M-interval synthetic rmsk" % (a.reads // 1_000_000, MODE_NAME[a.mode], a.rmsk / 1e6)

    # ---------------------------------------------------------------- reference arm
    if a.impl == "reference":
        if rank != 0:
            return 0
        world_s = S.Synth(shape, a.rmsk, seed=1)
        tables = world_s.write_tables(os.path.join(wd, "tables"))
        procs = a.cpu_procs or min(ncpu, 8)
        vals = []
        res = None
        for i in range(a.warmup + a.steps):
            res = reference_baseline(wd, tables, world_s, a.cpu_sample, a.mode, procs)
            if i >= a.warmup:
                vals.append(res["sample_reads"] / res["loop_s"])
        v = sum(vals) / len(vals)
        ms = 1e3 * res["sample_reads"] / v
        emit(({"metric": METRIC, "value": v, "unit": UNIT, "impl": "reference", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
               "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
               "data": "synthetic", "config": {"workload": workload, "step": "bounded sample: " + res["sample"]},
               "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": res["kind"], "sample": res["sample"]},
               "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        if not a.keep:
            shutil.rmtree(wd, ignore_errors=True)
        return 0

    # ---------------------------------------------------------------- our arm
    import iteres_b200 as itx
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
    L = itx.lib()
    if L.itx_device_count() <= lrank:
        raise SystemExit("bench.py: no CUDA device %d (the product has no CPU path)" % lrank)

    def barrier():
        if dist:
            dist.barrier()

    def max_over_ranks(x):
        if not dist:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def sum_over_ranks(x):
        if not dist:
            return x
        import torch
        t = torch.tensor([float(x)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    t_setup = time.perf_counter()
    world_s = S.Synth(shape, a.rmsk, seed=1)
    tdir = os.path.join(wd, "tables")
    if rank == 0:
        tables = world_s.write_tables(tdir)
    barrier()
    tables = tuple(os.path.join(tdir, n) for n in ("chrom.sizes", "rep.sizes", "rmsk.txt"))
    opts = itx.default_opts()
    gth = max(1, ncpu // world)

    # the pre-flight half of the parity gate starts now, in the background: the checker on ONE small file (N = 1: the first
    # cpu_baseline sample; N > 1: a PE-100 file every rank will scan a block range of)
    pre = None
    pre_bam = os.path.join(wd, "preflight.bam")
    pre_mode = a.mode if world == 1 else 2
    if rank == 0:
        keep = world_s.seed
        world_s.seed = 777
        world_s.write_bam(pre_bam, pre_mode, 1_000_000 if world > 1 else a.cpu_sample, level=1, threads=max(1, ncpu // 2))
        world_s.seed = keep
        pre = Checker("stat", [], tables, pre_bam, os.path.join(wd, "pre_ref"))
    ix = itx.Index(*tables, device=lrank)
    if a.chunk or a.window:
        ix.tune(chunk_bytes=a.chunk, window_bytes=a.window)
    if world > 1:
        ix.tune(inflate_threads=max(2, ncpu // world))      # the ranks of a box share its host cores
    log("index: %d intervals, %d subfamilies (%.1f s)" % (L.itx_n_elem(ix.h), ix.n(0), time.perf_counter() - t_setup))
    if world > 1:
        uid = [ix.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ix.comm_init(uid[0], rank, world)
    barrier()

    # ---------------------------------------------------------------- parity gate, pre-flight: before anything is timed
    parity = {"status": "ok", "gate": "tables byte for byte (subfamily / family / class .stat + .report)", "checks": []}
    ix.reset()
    if world == 1:
        ix.scan_alignments(pre_bam, opts)
    else:
        ix.scan_alignments_shard(pre_bam, opts)
        ix.allreduce_counts()
    if rank == 0:
        ix.sync()
        gpu_tables(ix, "stat", os.path.join(wd, "pre_gpu"), opts)
        pre.wait()
        nf = compare_tables("stat", os.path.join(wd, "pre_gpu"), pre.outdir, "pre-flight (%s)" % os.path.basename(pre_bam))
        parity["checks"].append({"what": "pre-flight: `iteres stat` on a %s file of %d records, %s" % (
            MODE_NAME[pre_mode], int(ix.cnt[0] + ix.cnt[1]), "ONE file split by BGZF block ranges over %d ranks + allreduce" % world if world > 1 else "itx_scan_alignments"),
            "against": pre.kind, "files": nf, "status": "ok"})
        log("parity pre-flight ok (%s, %d files, checker %.1f s)" % (pre.kind, nf, pre.seconds))
    barrier()

    # ---------------------------------------------------------------- headline: this rank's shard of the coordinate-sorted stream, generator chunks [c0, c1)
    n_units = a.reads * world
    nch = world_s.n_chunks(n_units)
    c0, c1 = rank * nch // world, (rank + 1) * nch // world
    R = Resident(L, ix, world_s, a.mode, n_units, c0, c1, gth)
    n, nrec = R.n, R.nrec
    log("shard: %d records, %.2f GB uncompressed, generated+uploaded (%.1f s since start)" % (nrec, n / 1e9, time.perf_counter() - t_setup))

    def step():
        ix.reset()
        cnt = ix.scan_bam_device(R.h, R.dbuf, n, opts)     # this rank's counters
        if world > 1:
            step.global_cnt = ix.allreduce_counts()    # the job's counters after the one allreduce
        return cnt
    step.global_cnt = None

    for _ in range(a.warmup):
        step()
    L.itx_dev_sync()
    barrier()
    sampler = ClockSampler(lrank)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    barrier()
    for _ in range(2):              # every rank: keep the devices busy until the sampler is running (untimed)
        step()
    L.itx_dev_sync()
    barrier()
    dec = 0.0
    launches = 0
    t_w0 = time.perf_counter()
    ix.mark(0)
    for _ in range(a.steps):
        cnt = step()
        pr = ix.profile()
        dec += pr["decode_ms"] + pr["overlap_ms"]; launches += pr["n_launches"]
    ix.mark(1)
    L.itx_dev_sync()
    el_ms = ix.elapsed_ms(0, 1)
    sampler.window(t_w0, time.perf_counter())
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    assert cnt[0] + cnt[1] == nrec, (cnt, nrec)
    el_ms = max_over_ranks(el_ms)
    total_rec = int(sum_over_ranks(nrec))
    if dist:
        assert step.global_cnt[0] + step.global_cnt[1] == total_rec, (step.global_cnt, total_rec)   # the allreduce summed every shard
    value = total_rec * a.steps / (el_ms * 1e-3)
    pr = ix.profile()
    bad = pr["n_bad_chunks"]
    if a.dump_outputs and rank == 0:
        dump_outputs(ix, step.global_cnt if dist else cnt, a.dump_outputs)

    # roofline of the dominant kernel (per step, this rank)
    peak, peak_src = peaks()
    fused = bool(pr.get("fused"))
    ks_ms = dec / a.steps
    ks_bytes = kscan_bytes(n, cnt)
    all_k = {"k_scan": {"ms": ks_ms, "bytes": ks_bytes, "GBps": ks_bytes / max(ks_ms, 1e-9) / 1e6, "frac": ks_bytes / max(ks_ms, 1e-9) / 1e6 / peak}}
    if fused and not a.no_extra:
        # the tuple path (what -R and the ordered outputs run), timed outside the timed region for comparison
        R_, F_, H_, HU_ = cnt[0] + cnt[1], cnt[6], cnt[9] + cnt[12], cnt[10]
        k1_bytes = n + 16 * R_
        k2_bytes = 16 * R_ + 16 * F_ + 28 * H_ + 8 * HU_
        os.environ["ITX_FUSED"] = "0"
        d2 = o2 = 0.0
        ix.reset(); ix.scan_bam_device(R.h, R.dbuf, n, opts)        # untimed: the first launch of these kernels loads them
        for _ in range(5):
            ix.reset(); ix.scan_bam_device(R.h, R.dbuf, n, opts)
            p2 = ix.profile()
            d2 += p2["decode_ms"] / 5; o2 += p2["overlap_ms"] / 5
        del os.environ["ITX_FUSED"]
        all_k["tuple_path"] = {"k_decode_span": {"ms": d2, "bytes": k1_bytes, "GBps": k1_bytes / max(d2, 1e-9) / 1e6, "frac": k1_bytes / max(d2, 1e-9) / 1e6 / peak},
                               "k_overlap": {"ms": o2, "bytes": k2_bytes, "GBps": k2_bytes / max(o2, 1e-9) / 1e6, "frac": k2_bytes / max(o2, 1e-9) / 1e6 / peak}}
    ach = ks_bytes / (ks_ms * 1e-3) / 1e9 if ks_ms > 0 else 0.0
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("reads_per_gpu") == a.reads and tj.get("mode") == a.mode:
            traffic, traffic_src = tj.get("k_scan"), tj.get("source")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k_scan (K1+K2+K3 fused: record boundaries, decode, overlap, selection, accumulation)" if fused else "tuple path",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
                "frac_stream_bytes_only": n / (ks_ms * 1e-3) / 1e9 / peak if ks_ms > 0 else 0.0,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": ks_bytes, "stream_bytes_per_launch": n, "kernel_ms_per_step": ks_ms,
                "replayed_windows": int(pr.get("n_replayed_windows", 0)), "all_kernels": all_k}

    # ---------------------------------------------------------------- e2e: BGZF -> tables through the C ABI, host buffers, copies inside the timed region
    e2e = e2e_file = None
    if not a.no_e2e:
        bam = os.path.join(wd, "shard%d.bam" % rank)
        t0 = time.perf_counter()
        fsz = R.write_bgzf(bam, gth)
        log("BGZF shard written: %.2f GB (%.1f s)" % (fsz / 1e9, time.perf_counter() - t0))
        R.free_host()
        pin = L.itx_host_alloc_pinned(fsz + 64)
        if not pin:
            raise SystemExit("pinned allocation of %d bytes failed" % (fsz + 64))
        with open(bam, "rb") as f:
            assert f.readinto((C.c_char * fsz).from_address(pin)) == fsz

        def run_e2e(call, tag):
            times = []
            for i in range(1 + a.e2e_steps):
                barrier()
                t0 = time.perf_counter()
                ix.reset()
                c2 = call()
                if world > 1:
                    ix.allreduce_counts()
                ix._dirty = True
                ix.sync()                                   # counter tables + coverage vectors back on the host
                dt = max_over_ranks(time.perf_counter() - t0)
                if i:
                    times.append(dt)
                assert c2 == cnt, (tag, c2, cnt)           # the same counters as the device-resident scan of the same records
            pe = ix.profile()
            t = sum(times) / len(times)
            log("e2e %s: %s ms" % (tag, " ".join("%.1f" % (1e3 * x) for x in times)))
            return {"value": total_rec / t, "unit": UNIT, "h2d_bytes_per_step": int(pe["h2d_bytes"]), "d2h_bytes_per_step": int(pe["d2h_bytes"]),
                    "s_per_step": t, "steps": len(times), "inflate_ms": pe["inflate_ms"], "bam_bytes": fsz,
                    "inflate": "device: k_inflate (one thread per BGZF block decodes literals and lists matches, 16 blocks per warp; the warp then copies the matches of its blocks in shared-memory windows), launch groups on 8 streams"}
        e2e = run_e2e(lambda: ix.scan_bgzf_memory(pin, fsz, opts), "pinned image")
        e2e["api"] = "itx_scan_bgzf_memory(BGZF image in pinned host memory, deflate level 1) + itx_sync_counts"
        e2e_file = run_e2e(lambda: ix.scan_alignments(bam, opts), "file")
        e2e_file["api"] = "itx_scan_alignments(BGZF .bam file) + itx_sync_counts"
        e2e_file["file"] = "on tmpfs / page-cache resident (%s): no storage device is read inside the timed region" % os.path.dirname(bam)
        L.itx_host_free_pinned(pin)
    R.free()

    # ---------------------------------------------------------------- CPU baseline (rank 0, N = 1 only) + the gate's second half
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        procs = a.cpu_procs or min(ncpu, 8)
        try:
            r = reference_baseline(wd, tables, world_s, a.cpu_sample, a.mode, procs)
        except Exception as ex:   # the baseline is reported, never load-bearing
            r = None
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": "failed: %s" % ex}
        if r:
            cpu = {"value": r["sample_reads"] / r["loop_s"], "unit": UNIT, "cores": procs, "kind": r["kind"], "sample": r["sample"],
                   "wall_s": r["wall_s"], "fixed_s": r["fixed_s"], "host_cpus": ncpu}
            # every sample BAM the reference just wrote tables for goes through the CUDA path: byte for byte, at the bench's table density
            nf = 0
            for b, od in zip(r["bams"], r["out_dirs"]):
                ix.reset()
                ix.scan_alignments(b, opts)
                ix._dirty = True
                ix.sync()
                gd = od + "_gpu"
                gpu_tables(ix, "stat", gd, opts)
                nf += compare_tables("stat", gd, od, "cpu_baseline sample %s" % os.path.basename(b))
            parity["checks"].append({"what": "`iteres stat` on the %d cpu_baseline sample BAMs (%d reads each, 5.5 M-row table), itx_scan_alignments + itx_write_stat" % (len(r["bams"]), a.cpu_sample),
                                     "against": r["kind"], "files": nf, "status": "ok"})
            log("parity gate ok on %d sample BAMs (%d files)" % (len(r["bams"]), nf))

    # ---------------------------------------------------------------- the other BASELINE configs (N = 1), strong scaling (N > 1)
    extra = None
    strong = None
    if not a.no_extra and world == 1:
        extra = extra_configs(a, L, ix, world_s, tables, wd, opts, peak, ncpu, parity)
    if not a.no_extra:
        strong = strong_scaling(a, L, ix, world_s, tables, wd, opts, rank, world, barrier, max_over_ranks, ncpu, sum_over_ranks)

    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
               "ms_per_step": el_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": DTYPE, "data": "synthetic",
               "config": {"workload": workload, "records_per_gpu": nrec, "stream_bytes_per_gpu": n, "l2": "inputs (%.1f GB per GPU) are larger than the 126 MB L2; no flush needed" % (n / 1e9),
                          "chunk_bytes": a.chunk or 65536, "parallelism": "genome-coordinate shards x%d, one allreduce of the counter block per step" % world if world > 1 else "single GPU",
                          "repaired_chunk_entries": int(bad)},
               "clocks": clocks, "e2e": e2e, "e2e_file": e2e_file, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
               "counters": {"records": int(cnt[0] + cnt[1]), "fragments": int(cnt[6]), "in_repeats": int(cnt[9]), "unique_in_repeats": int(cnt[10])}}
        if extra is not None:
            out["extra_configs"] = extra
        if strong is not None:
            out["strong_scaling"] = strong
        emit(out)
    ix.close()
    barrier()
    if rank == 0 and not a.keep:
        shutil.rmtree(wd, ignore_errors=True)
    if dist:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------ BASELINE.json configs 1, 3, 4, 5 on one GPU
def extra_configs(a, L, ix, world_s, tables, wd, opts, peak, ncpu, parity):
    import iteres_b200 as itx
    import synth as S
    out = {}
    steps, warm = 10, 3
    checks = []          # (name, cmd, Checker, gpu dir, rtol) settled at the end, so that the checkers run while the GPU is timed

    def small_file(name, mode, units, seed, world=world_s):
        p = os.path.join(wd, name)
        keep = world.seed
        world.seed = seed
        world.write_bam(p, mode, units, level=1, threads=max(1, ncpu // 2))
        world.seed = keep
        return p

    def gpu_side(index, cmd, path, o, tag):
        index.reset()
        if cmd == "cpgstat":
            index.scan_cpg(path)
        else:
            index.scan_alignments(path, o)
        index._dirty = True
        index.sync()
        gd = os.path.join(wd, "x_%s_gpu" % tag)
        gpu_tables(index, cmd, gd, o)
        return gd

    # ---- cfg 3: SE-75 with XA:Z multi-reads; stat (per-subfamily tables, -x on) and filter (per-locus table)
    t0 = time.perf_counter()
    n3 = min(a.reads * 3 // 5, 30_000_000)
    p3 = small_file("cfg3_prefix.bam", 1, 1_000_000, 4243)
    o_f = itx.default_opts(filter=1, diffSubfam=0)
    checks.append(("cfg3 stat", "stat", Checker("stat", [], tables, p3, os.path.join(wd, "x_cfg3s_ref")), gpu_side(ix, "stat", p3, opts, "cfg3s"), 0.0))
    checks.append(("cfg3 filter", "filter", Checker("filter", [], tables, p3, os.path.join(wd, "x_cfg3f_ref")), gpu_side(ix, "filter", p3, o_f, "cfg3f"), 0.0))
    R3 = Resident(L, ix, world_s, 1, n3, threads=ncpu)
    ks, stp, c3, _ = timed_resident(ix, R3, opts, steps, warm)
    b3 = kscan_bytes(R3.n, c3)
    ksf, stpf, c3f, _ = timed_resident(ix, R3, o_f, steps, warm)
    b3f = R3.n + 16 * c3f[6] + 24 * c3f[9] + 4 * c3f[10]        # per-locus mode: 16 B hit + one 4 B counter (+ 4 B unique)
    out["cfg3_se75_xa"] = {"workload": "SE-75, 30 %% of the reads MAPQ 0 with NM + XA:Z (1-5 alternates), %d M reads (BASELINE names 100 M; bounded for the bench's time budget), 5.5 M-row table" % (n3 // 1_000_000),
                           "stat": {"value": R3.nrec / (stp * 1e-3), "unit": UNIT, "kernel_ms": ks, "ms_per_step": stp,
                                    "roofline": {"bound": "hbm", "achieved": b3 / ks / 1e6, "peak": peak, "unit": "GB/s", "frac": b3 / ks / 1e6 / peak, "frac_stream_bytes_only": R3.n / ks / 1e6 / peak},
                                    "reads_with_alternates_in_other_subfamilies": int(c3[12]), "in_repeats": int(c3[9])},
                           "filter": {"value": R3.nrec / (stpf * 1e-3), "unit": UNIT, "kernel_ms": ksf, "ms_per_step": stpf,
                                      "roofline": {"bound": "hbm", "achieved": b3f / ksf / 1e6, "peak": peak, "unit": "GB/s", "frac": b3f / ksf / 1e6 / peak, "frac_stream_bytes_only": R3.n / ksf / 1e6 / peak},
                                      "table": "per-locus counts (iteres filter / nameStat), %d loci hit" % int(c3f[9])}}
    R3.free()
    log("cfg3: stat k_scan %.2f ms, filter %.2f ms per %d M reads (%.1f s)" % (ks, ksf, n3 // 1_000_000, time.perf_counter() - t0))

    # ---- cfg 5: PE-100, proper pairs + discordant + one-end-mapped
    t0 = time.perf_counter()
    n5 = a.reads // 2
    p5 = small_file("cfg5_prefix.bam", 2, 1_000_000, 4245)
    checks.append(("cfg5 stat", "stat", Checker("stat", [], tables, p5, os.path.join(wd, "x_cfg5_ref")), gpu_side(ix, "stat", p5, opts, "cfg5"), 0.0))
    R5 = Resident(L, ix, world_s, 2, n5, threads=ncpu)
    ks, stp, c5, _ = timed_resident(ix, R5, opts, steps, warm)
    b5 = kscan_bytes(R5.n, c5)
    out["cfg5_pe100"] = {"workload": "PE-100, %d M pairs (%d M records) on ONE GPU, 5.5 M-row table; the 1/2/4/8-GPU split of one file is the strong_scaling block of the --gpus N lines" % (n5 // 1_000_000, R5.nrec // 1_000_000),
                         "value": R5.nrec / (stp * 1e-3), "unit": "read ends/s", "kernel_ms": ks, "ms_per_step": stp,
                         "roofline": {"bound": "hbm", "achieved": b5 / ks / 1e6, "peak": peak, "unit": "GB/s", "frac": b5 / ks / 1e6 / peak, "frac_stream_bytes_only": R5.n / ks / 1e6 / peak}}
    R5.free()
    log("cfg5: k_scan %.2f ms per %d M pairs (%.1f s)" % (ks, n5 // 1_000_000, time.perf_counter() - t0))

    # ---- cfg 4: cpgstat, 28 M-row bedGraph
    t0 = time.perf_counter()
    bg_small, bg = os.path.join(wd, "cpg_prefix.bedGraph"), os.path.join(wd, "cpg.bedGraph")
    world_s.write_bedgraph(bg_small, 1_000_000)
    checks.append(("cfg4 cpgstat", "cpgstat", Checker("cpgstat", [], tables, bg_small, os.path.join(wd, "x_cfg4_ref")), gpu_side(ix, "cpgstat", bg_small, opts, "cfg4"), 1e-9))
    n4 = max(1_000_000, 28_000_000 * a.reads // 50_000_000)       # 28 M rows at the bench's full size
    world_s.write_bedgraph(bg, n4)
    times = []
    for i in range(4):
        t1 = time.perf_counter()
        ix.reset()
        lines, inrep = ix.scan_cpg(bg)
        ix._dirty = True
        ix.sync()
        if i:
            times.append(time.perf_counter() - t1)
    pr = ix.profile()
    t4 = sum(times) / len(times)
    kms = pr.get("cpg_kernel_ms", 0.0)
    fsz = os.path.getsize(bg)
    b4 = fsz + 16 * lines + 16 * inrep
    out["cfg4_cpgstat"] = {"workload": "iteres cpgstat, %d M-row CpG bedGraph (%.0f MB of text, parsed on the device) vs the 5.5 M-row table" % (n4 // 1_000_000, fsz / 1e6),
                           "value": lines / t4, "unit": "CpG rows/s", "s_per_step": t4, "rows": int(lines), "rows_in_repeats": int(inrep),
                           "api": "itx_scan_cpg(file on tmpfs) + itx_sync_counts: pread -> pinned -> cudaMemcpyAsync -> k_bedgraph, all inside the timed region",
                           "kernel_ms": kms,
                           "roofline": {"bound": "hbm", "kernel": "k_bedgraph", "achieved": (b4 / kms / 1e6) if kms else None, "peak": peak, "unit": "GB/s",
                                        "frac": (b4 / kms / 1e6 / peak) if kms else None, "bytes": "text + 16 B probe per row + 16 B per hit"}}
    log("cfg4: %.1f M rows/s end to end, k_bedgraph %.2f ms (%.1f s)" % (lines / t4 / 1e6, kms, time.perf_counter() - t0))

    # ---- cfg 1: chr1 only, 1 M SE reads vs a 200 k-row table: the reference's own CPU-runnable case, whole, through the file path
    t0 = time.perf_counter()
    w1 = S.Synth(0, 200_000, seed=1)
    t1dir = os.path.join(wd, "tables_cfg1")
    tab1 = w1.write_tables(t1dir)
    p1 = small_file("cfg1.bam", 0, 1_000_000, 4241, world=w1)
    ix1 = itx.Index(*tab1, device=0)
    ck1 = Checker("stat", [], tab1, p1, os.path.join(wd, "x_cfg1_ref"))
    times = []
    for i in range(6):
        t1 = time.perf_counter()
        ix1.reset()
        c1 = ix1.scan_alignments(p1, opts)
        ix1._dirty = True
        ix1.sync()
        if i:
            times.append(time.perf_counter() - t1)
    gd1 = os.path.join(wd, "x_cfg1_gpu")
    gpu_tables(ix1, "stat", gd1, opts)
    w1.seed = 4241                                             # the reads of cfg1.bam
    R1 = Resident(L, ix1, w1, 0, 1_000_000, threads=ncpu)
    ks, stp, c1r, _ = timed_resident(ix1, R1, opts, 20, 3)
    assert c1r == c1
    ck1.wait()
    nf = compare_tables("stat", gd1, ck1.outdir, "cfg1 (whole config)")
    parity["checks"].append({"what": "cfg 1 whole: `iteres stat`, 1 M SE-50 reads (chr1) vs 200 k rows", "against": ck1.kind, "files": nf, "status": "ok"})
    b1 = kscan_bytes(R1.n, c1r)
    out["cfg1_1m_chr1"] = {"workload": "iteres stat, 1 M SE-50 reads (chr1 only) vs a 200 k-row rmsk: the whole config, as the reference runs it on a CPU",
                           "value": R1.nrec / (stp * 1e-3), "unit": UNIT, "kernel_ms": ks, "ms_per_step": stp,
                           "e2e_file": {"value": R1.nrec / (sum(times) / len(times)), "unit": UNIT, "s_per_step": sum(times) / len(times)},
                           "reference_wall_s": ck1.seconds, "reference_kind": ck1.kind,
                           "roofline": {"bound": "hbm", "achieved": b1 / ks / 1e6, "peak": peak, "unit": "GB/s", "frac": b1 / ks / 1e6 / peak,
                                        "note": "a 130 MB stream: one wave of spans, launch latency and the tail dominate"}}
    R1.free(); ix1.close(); w1.close()
    log("cfg1: k_scan %.3f ms, file path %.1f ms, reference %.1f s (%.1f s)" % (ks, 1e3 * sum(times) / len(times), ck1.seconds, time.perf_counter() - t0))

    # ---- settle the prefix checks
    for name, cmd, ck, gd, rtol in checks:
        ck.wait()
        nf = compare_tables(cmd, gd, ck.outdir, name, rtol)
        parity["checks"].append({"what": "%s: 1 M-unit prefix, %s" % (name, "CpG score sums within 1e-9 relative, counts exact" if rtol else "byte for byte"),
                                 "against": ck.kind, "files": nf, "status": "ok"})
        out[{"cfg3 stat": "cfg3_se75_xa", "cfg3 filter": "cfg3_se75_xa", "cfg5 stat": "cfg5_pe100", "cfg4 cpgstat": "cfg4_cpgstat"}[name]].setdefault("parity", []).append(
            {"check": name, "against": ck.kind, "status": "ok"})
    return out


# ------------------------------------------------------------------------------------------ ONE PE-100 file over N GPUs
def strong_scaling(a, L, ix, world_s, tables, wd, opts, rank, world, barrier, max_over_ranks, ncpu, sum_over_ranks):
    import synth as S
    bam = os.path.join(wd, "strong_pe100.bam")
    t0 = time.perf_counter()
    # ONE coordinate-sorted file, written once: every rank generates and compresses its slice of the generator's chunks (the header goes
    # into the first part only; BGZF parts concatenate once the empty end-of-file block of all but the last is dropped), rank 0 joins them
    import numpy as np
    hdr = world_s.header()
    nch = world_s.n_chunks(a.strong_pairs)
    c0, c1 = rank * nch // world, (rank + 1) * nch // world
    gth = max(1, ncpu // world)
    part = "%s.part%d" % (bam, rank)
    my_rec = 0
    with open(part, "wb") as fpart:
        per = max(1, (c1 - c0 + 3) // 4)                   # in a few slices, so that no rank holds more than a couple of GB at a time
        tmp = part + ".tmp"
        for k0 in range(c0, c1, per):
            k1 = min(c1, k0 + per)
            sz, nrec = world_s.records_size(2, a.strong_pairs, k0, k1, gth)
            buf = np.zeros(sz + 64, dtype=np.uint8)
            assert world_s.records_into(buf.ctypes.data, 2, a.strong_pairs, k0, k1, gth) == sz
            rc = S.lib().synth_write_bam(tmp.encode(), hdr.ctypes.data, len(hdr) if k0 == 0 else 0, buf.ctypes.data, sz, 1, gth)
            assert rc == 0
            with open(tmp, "rb") as f:
                data = f.read()
            if k1 < nch and data.endswith(BGZF_EOF):
                data = data[:-len(BGZF_EOF)]
            fpart.write(data)
            my_rec += nrec
        if os.path.exists(tmp):
            os.unlink(tmp)
    barrier()
    if rank == 0:
        with open(bam, "wb") as out:
            for r in range(world):
                with open("%s.part%d" % (bam, r), "rb") as f:
                    shutil.copyfileobj(f, out, 64 << 20)
                os.unlink("%s.part%d" % (bam, r))
        log("strong scaling: ONE PE-100 file, %d M pairs, %.2f GB BGZF (%.1f s)" % (a.strong_pairs // 1_000_000, os.path.getsize(bam) / 1e9, time.perf_counter() - t0))
    total_rec = int(sum_over_ranks(my_rec))
    barrier()
    times = []
    got = None
    for i in range(3):
        barrier()
        t1 = time.perf_counter()
        ix.reset()
        if world > 1:
            ix.scan_alignments_shard(bam, opts)
            got = ix.allreduce_counts()
        else:
            got = ix.scan_alignments(bam, opts)              # the 1-GPU point of the same curve: the whole file, one device
        ix._dirty = True
        ix.sync()
        dt = max_over_ranks(time.perf_counter() - t1)
        if i:
            times.append(dt)
    pr = ix.profile()
    dev_ms = max_over_ranks(pr["total_ms"])                 # device side of the slowest rank: first to last scan launch on its stream
    inf_ms = max_over_ranks(pr["inflate_ms"])
    if rank != 0:
        return None
    assert got[0] + got[1] == total_rec, (got, total_rec)
    t = sum(times) / len(times)
    return {"workload": "iteres stat on ONE coordinate-sorted PE-100 BGZF file, %d M pairs (%d M records, %.2f GB; BASELINE names 500 M: bounded by the bench's time budget), the same file at every N" % (
                a.strong_pairs // 1_000_000, total_rec // 1_000_000, os.path.getsize(bam) / 1e9),
            "scaling": "strong", "n_gpus": world, "value": total_rec / t, "unit": "read ends/s", "s_per_step": t, "steps": len(times),
            "api": ("itx_scan_alignments_shard (BGZF block ranges, guessed first records, NCCL all-gather chain check) + itx_comm_allreduce_counts + itx_sync_counts"
                    if world > 1 else "itx_scan_alignments + itx_sync_counts (one device: the whole file)"),
            "file": "on tmpfs / page-cache resident: every rank pread()s its block range into pinned slots with %d host threads (the box's %d cores are shared by the ranks)" % (max(2, ncpu // world), ncpu),
            "device_ms_slowest_rank": {"inflate_first_launch_to_last_end": inf_ms, "scan_stream_first_to_last_launch": dev_ms},
            "ranks_rescanned_after_chain_check": int(pr["n_bad_chunks"]),
            "counters": {"records": int(got[0] + got[1]), "fragments": int(got[6]), "in_repeats": int(got[9])}}


BGZF_EOF = bytes([0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0, 0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0])


if __name__ == "__main__":
    sys.exit(main())
