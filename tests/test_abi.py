"""The C-ABI library loads on a box without a GPU and exports every symbol include/iteres_gpu.h
declares; without a device the product refuses to work instead of falling back to anything."""
import ctypes as C
import os
import re
import subprocess
import sys

from iteres_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    h = open(os.path.join(ROOT, "include", "iteres_gpu.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return sorted(set(re.findall(r"\b(itx_[a-z0-9_]+)\s*\(", h)))


def test_library_exports_every_declared_symbol():
    L = C.CDLL(capi.lib_path())
    decl = declared_symbols()
    assert len(decl) >= 40
    for s in decl:
        assert hasattr(L, s), s
    assert set(decl) == set(capi.SYMBOLS)


def test_struct_layout_matches_header():
    assert C.sizeof(capi.ScanOpts) == 64 and C.sizeof(capi.Trace) == 20      # 10 scalars, readNames, isSam, two path pointers
    o = capi.ScanOpts()
    capi.lib().itx_scan_opts_default(C.byref(o))
    assert (o.mapQ, o.iSize, o.extension, o.diffSubfam, o.filter, o.readNames, o.outbed, o.outbed_unique) == (10, 500, 150, 1, 0, 0, None, None)
    assert abs(o.minCoverage - 1e-4) < 1e-10


def test_no_device_means_error_not_fallback(tmp_path):
    """in processes that see no CUDA device (an empty CUDA_VISIBLE_DEVICES hides any the machine has)"""
    gold = os.path.join(ROOT, "tests", "golden", "kat1_basic", "input")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    probe = ("import sys\nsys.path.insert(0, %r)\nfrom iteres_b200 import capi\nassert capi.lib().itx_device_count() == 0\n"
             "try:\n    capi.Index(*sys.argv[1:])\nexcept capi.ItxError as e:\n    print(e)\n" % ROOT)
    p = subprocess.run([sys.executable, "-c", probe] + [os.path.join(gold, f) for f in ("chrom.sizes", "rep.sizes", "rmsk.txt")],
                       env=env, capture_output=True, text=True)
    assert p.returncode == 0 and "no usable CUDA device" in p.stdout, p.stdout + p.stderr
    cli = os.path.join(ROOT, "iteres_b200", "csrc", "iteres")
    p = subprocess.run([cli, "stat", "-o", str(tmp_path / "x")] + [os.path.join(gold, f) for f in ("chrom.sizes", "rep.sizes", "rmsk.txt", "reads.bam")],
                       env=env, capture_output=True, text=True)
    assert p.returncode == 255 and "no usable CUDA device" in p.stderr


def test_product_never_touches_the_oracle():
    """nothing under iteres_b200/ or include/ may name, link or load the checker"""
    for d in ("iteres_b200", "include"):
        for base, _, files in os.walk(os.path.join(ROOT, d)):
            for f in files:
                if f.endswith((".c", ".cu", ".cuh", ".h", ".py")) or f == "Makefile":
                    txt = open(os.path.join(base, f), errors="ignore").read()
                    assert "liboracle" not in txt and "ora_" not in txt and "oracle/" not in txt, os.path.join(base, f)
    out = subprocess.run(["ldd", capi.lib_path()], capture_output=True, text=True).stdout
    assert "oracle" not in out and "emu" not in out


def test_cli_usage_and_exit_codes():
    cli = os.path.join(ROOT, "iteres_b200", "csrc", "iteres")
    p = subprocess.run([cli], capture_output=True, text=True)
    assert p.returncode == 1 and "Usage:   iteres <command> [options]" in p.stderr
    for cmd in ("stat", "filter", "cpgstat", "cpgfilter"):
        p = subprocess.run([cli, cmd], capture_output=True, text=True)
        assert p.returncode == 1 and "Usage:   iteres %s" % cmd in p.stderr
    p = subprocess.run([cli, "bogus"], capture_output=True, text=True)
    assert p.returncode == 1 and "unrecognized command 'bogus'" in p.stderr
