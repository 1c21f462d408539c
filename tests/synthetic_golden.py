"""Stored outputs of the reference for the generated worlds of tests/test_emu_synth.py and tests/test_bigwig.py, so that
their comparisons with the reference run on every machine: tests/golden/synthetic/ holds, per case, the `stat` tables and
report (gzipped, byte for byte), the wiggles (sha256, size and a seeded sample of non-zero lines: 9 MB each) and, for the bigWig
cases, the sha256 and size of each wiggle and of the bigWig the reference built from it.

    python tests/synthetic_golden.py        # (re)record; uses the reference binary oracle/_ref/iteres when it is built

manifest.json names the source of what it holds.  Where the reference binary is not built, the recorder takes the files
from the code the tests pin to it: the oracle (tables, report, wiggles) and the product's bigWig writer (bigWig files)."""
import gzip
import hashlib
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import oracle_lib as O  # noqa: E402
import runners  # noqa: E402
import synth  # noqa: E402

DIR = os.path.join(HERE, "golden", "synthetic")
MANIFEST = os.path.join(DIR, "manifest.json")
STAT_WORLD = (1, 60000, 7)               # shape, rmsk rows, seed of test_emu_synth's worlds(1, 60000)
STAT_CASES = [(0, 20000, []), (1, 20000, []), (2, 10000, []), (1, 10000, ["-x", "-E", "0"])]
STAT_TEXT = ["out.iteres.subfamily.stat", "out.iteres.family.stat", "out.iteres.class.stat", "out.iteres.report"]
STAT_WIG = ["out.iteres.wig", "out.iteres.unique.wig"]
BIGWIG_SEED = 11
BIGWIG_CASES = [(1, 60000, 0, 150000), (0, 20000, 2, 30000)]
BIGWIG_STEMS = ["ref.iteres", "ref.iteres.unique"]
SAMPLE_LINES = 100


def stat_case(mode, n_units, args):
    return "_".join(["m%d" % mode, str(n_units)] + [a.strip("-") for a in args])


def bigwig_case(shape, n_rmsk, mode, n_units):
    return "s%d_%d_m%d_%d" % (shape, n_rmsk, mode, n_units)


def digest(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 20), b""):
            h.update(b)
    return {"sha256": h.hexdigest(), "size": os.path.getsize(path)}


def load():
    with open(MANIFEST) as f:
        return json.load(f)


def write_bam(world, path, mode, n_units):
    world.write_bam(path, mode, n_units, level=1, threads=4)


def oracle_stat(tables, bam, args, outdir, prefix="out"):
    """what `iteres stat -o <prefix> <args>` writes for the tables and the report, from the oracle"""
    o = runners.parse("stat", args)
    ix = O.OracleIndex(*tables)
    try:
        ix.scan_file(bam, runners.ora_opts(o))
        p = os.path.join(outdir, prefix)
        ix.write_stat(p, o["nindex"], o["nindex2"])
        ix.write_report(p + ".iteres.report", o["Q"], "ALL")
    finally:
        ix.close()


def reference_stat(tables, bam, args, outdir, prefix="out"):
    p = subprocess.run([O.REF_BIN, "stat", "-w", "-o", prefix] + args + list(tables) + [bam], cwd=outdir, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:]


def check_stat(case, outdir):
    """the files of `iteres stat` in outdir against the stored ones of `case`: the tables and the report byte for byte, the
    wiggles by sha256 and size (a mismatch names the first sampled line that differs)"""
    want = load()["stat"][case]
    for fn in STAT_TEXT:
        with gzip.open(os.path.join(DIR, case, fn + ".gz"), "rb") as f:
            exp = f.read()
        with open(os.path.join(outdir, fn), "rb") as f:
            got = f.read()
        if got != exp:
            bad = next((i for i, (x, y) in enumerate(zip(got.split(b"\n"), exp.split(b"\n"))) if x != y), None)
            raise AssertionError("%s differs from the reference's (first differing line %s)" % (fn, bad))
    for fn in STAT_WIG:
        w = want["wig"][fn]
        if digest(os.path.join(outdir, fn)) != {"sha256": w["sha256"], "size": w["size"]}:
            with open(os.path.join(outdir, fn), "rb") as f:
                lines = f.read().split(b"\n")
            bad = [(i, s) for i, s in w["sample"] if i >= len(lines) or lines[i].decode() != s]
            raise AssertionError("%s differs from the reference's (sampled lines that differ: %s)" % (fn, bad[:3]))


def record():
    import tempfile
    import numpy as np
    use_ref = os.path.exists(O.REF_BIN)
    man = {"source": ("the reference binary (oracle/_ref/iteres stat -w)" if use_ref else
                      "the oracle (oracle/iteres_oracle.c: tables, report, wiggles) and the product's bigWig writer (itx_wig_to_bigwig)"),
           "stat": {}, "bigwig": {}}
    with tempfile.TemporaryDirectory() as d:
        shape, n_rmsk, seed = STAT_WORLD
        s = synth.Synth(shape, n_rmsk, seed=seed)
        tables = s.write_tables(os.path.join(d, "tables"))
        for mode, n_units, args in STAT_CASES:
            case = stat_case(mode, n_units, args)
            od = os.path.join(d, case)
            os.makedirs(od)
            bam = os.path.join(d, "reads.bam")
            write_bam(s, bam, mode, n_units)
            (reference_stat if use_ref else oracle_stat)(tables, bam, args, od)
            os.makedirs(os.path.join(DIR, case), exist_ok=True)
            for fn in STAT_TEXT:
                with open(os.path.join(od, fn), "rb") as f, open(os.path.join(DIR, case, fn + ".gz"), "wb") as g:
                    with gzip.GzipFile(filename=fn, mode="wb", fileobj=g, mtime=0) as z:
                        z.write(f.read())
            wigs = {}
            for fn in STAT_WIG:
                with open(os.path.join(od, fn), "rb") as f:
                    lines = f.read().split(b"\n")
                lit = [i for i, x in enumerate(lines) if x not in (b"", b"0")]          # the wiggle is mostly zero lines
                idx = np.sort(np.random.default_rng(len(lines)).choice(lit, min(SAMPLE_LINES, len(lit)), replace=False))
                wigs[fn] = dict(digest(os.path.join(od, fn)), sample=[[int(i), lines[i].decode()] for i in idx])
            man["stat"][case] = {"mode": mode, "n_units": n_units, "args": args, "wig": wigs}
        s.close()
        for shape, n_rmsk, mode, n_units in BIGWIG_CASES:
            case = bigwig_case(shape, n_rmsk, mode, n_units)
            od = os.path.join(d, "bw_" + case)
            os.makedirs(od)
            s = synth.Synth(shape, n_rmsk, seed=BIGWIG_SEED)
            tables = s.write_tables(od)
            bam = os.path.join(od, "reads.bam")
            write_bam(s, bam, mode, n_units)
            s.close()
            if use_ref:
                reference_stat(tables, bam, [], od, prefix="ref")
            else:
                oracle_stat(tables, bam, [], od, prefix="ref")
            man["bigwig"][case] = {}
            for stem in BIGWIG_STEMS:
                bw = os.path.join(od, stem + ".bigWig")
                if not use_ref:
                    runners.wig_to_bigwig(os.path.join(od, stem + ".wig"), tables[1], bw)
                man["bigwig"][case][stem] = {"wig": digest(os.path.join(od, stem + ".wig")), "bigWig": digest(bw)}
    with open(MANIFEST, "w") as f:
        json.dump(man, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    record()
