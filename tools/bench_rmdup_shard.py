#!/usr/bin/env python3
"""-R across devices: `iteres stat -R` on ONE coordinate-sorted PE-100 BGZF file of the strong-scaling shape of bench.py
(synthetic shape 1, 5.5 M-row rmsk table), through itx_scan_alignments_shard on 1, 2 and 8 devices (counts above the devices
present are skipped).  One process, one host thread and one index per device, as `ITERES_GPUS=N iteres` runs.  Reports per
device count: wall time per rank, the time in phase 1 (parts settled, keys collected), in the exchange (all-gathers, key export,
ncclBroadcast) and in phase 2 (admissions and the counting scan) of every rank, the bytes of keys broadcast, and whether the
counters and tables equal those of the single-device -R scan of the whole file.

usage: tools/bench_rmdup_shard.py [--pairs 40000000] [--gpus 1,2,8] [--steps 2] [--out FILE]
The file and the tables are written to a temporary directory, removed at the end."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from iteres_b200 import capi  # noqa: E402
import synth  # noqa: E402


def tables_of(ix):
    ix._dirty = True
    return [ix.table(w) for w in range(3)]


def run_ranks(n, fn):
    out, errs = [None] * n, []

    def one(r):
        try:
            out[r] = fn(r)
        except Exception as e:            # noqa: BLE001
            errs.append((r, repr(e)))
    th = [threading.Thread(target=one, args=(r,)) for r in range(n)]
    [t.start() for t in th]
    [t.join() for t in th]
    if errs:
        raise RuntimeError(errs)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=40_000_000)
    ap.add_argument("--rmsk", type=int, default=5_500_000)
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--steps", type=int, default=2, help="timed runs per device count (after one untimed run)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = capi.lib()
    ndev = L.itx_device_count()
    if ndev < 1:
        sys.exit("no CUDA device: this measurement runs on the GPU only")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    wd = tempfile.mkdtemp(prefix="itx_rmdup_bench_")
    try:
        s = synth.Synth(1, a.rmsk, seed=1)
        tabs = s.write_tables(os.path.join(wd, "tables"))
        bam = os.path.join(wd, "strong_pe100.bam")
        t0 = time.perf_counter()
        nbytes, nrec = s.write_bam(bam, 2, a.pairs, level=1, threads=os.cpu_count() or 8)
        s.close()
        res = {"workload": "iteres stat -R on ONE coordinate-sorted PE-100 BGZF file: %d M pairs, %d M records, %.2f GB BGZF, %.2f GB uncompressed; %d M-row rmsk table"
                           % (a.pairs // 1_000_000, nrec // 1_000_000, os.path.getsize(bam) / 1e9, nbytes / 1e9, a.rmsk // 1_000_000),
               "gpus_present": ndev, "gpu": gpu, "file_written_s": round(time.perf_counter() - t0, 1), "runs": []}
        opts = capi.default_opts(rmDup=1)
        ref = None
        for n in [int(x) for x in a.gpus.split(",")]:
            if n > ndev:
                res["runs"].append({"n_gpus": n, "skipped": "only %d device(s) present" % ndev})
                continue
            ixs = run_ranks(n, lambda r: capi.Index(*tabs, device=r))
            if n > 1:
                uid = ixs[0].comm_unique_id()
                run_ranks(n, lambda r: ixs[r].comm_init(uid, r, n))
            steps = []
            for step in range(a.steps + 1):
                def rank(r):
                    ix = ixs[r]
                    ix.reset()
                    t1 = time.perf_counter()
                    if n > 1:
                        ix.scan_alignments_shard(bam, opts)
                        t2 = time.perf_counter()
                        ix.allreduce_counts()
                    else:
                        ix.scan_alignments(bam, opts)
                        t2 = time.perf_counter()
                    ix._dirty = True
                    ix.sync()
                    p = ix.profile()
                    return {"wall_s": time.perf_counter() - t1, "scan_s": t2 - t1, "phase1_ms": p["rmdup_keys_ms"], "exchange_ms": p["rmdup_exchange_ms"],
                            "phase2_ms": p["rmdup_count_ms"], "bcast_bytes": p["rmdup_bcast_bytes"]}
                per = run_ranks(n, rank)
                if step:
                    steps.append(per)
            got = (list(ixs[0].cnt), tables_of(ixs[0]))
            if ref is None and n == 1:
                ref = got
            run = {"n_gpus": n, "api": "itx_scan_alignments_shard + itx_comm_allreduce_counts + itx_sync_counts" if n > 1 else "itx_scan_alignments + itx_sync_counts (the whole file on one device)",
                   "wall_s_per_rank": [[round(x["wall_s"], 3) for x in per] for per in steps],
                   "wall_s_slowest_rank_mean": round(sum(max(x["wall_s"] for x in per) for per in steps) / len(steps), 3),
                   "counters": {"records": got[0][0] + got[0][1], "fragments": got[0][6], "unique_kept": got[0][11], "in_repeats": got[0][9]},
                   "parity_with_one_device": None if ref is None else (got == ref)}
            if n > 1:
                run["phase_ms_per_rank"] = [[{k: round(x[k], 1) for k in ("phase1_ms", "exchange_ms", "phase2_ms")} for x in per] for per in steps]
                run["bytes_broadcast"] = steps[-1][0]["bcast_bytes"]
            res["runs"].append(run)
            for ix in ixs:
                ix.close()
    finally:
        shutil.rmtree(wd, ignore_errors=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    return 0 if all(r.get("parity_with_one_device") in (True, None) for r in res["runs"]) else 1


if __name__ == "__main__":
    sys.exit(main())
