"""The bigWig writer (iteres_b200/csrc/itx_bigwig.c, host C, the product's bigWigFileCreate) against the reference:
the committed golden .bigWig files of every `stat` / `cpgstat` known-answer variant are covered by the golden
suites; here a hg19-shaped world (1395 subfamilies: several sections per consensus, multi-level R and B+ trees,
several zoom levels) is compared with what the UNMODIFIED reference binary wrote for it, as stored under
tests/golden/synthetic/ (and with the binary itself where it is built: oracle/_ref/iteres), and the error paths are checked."""
import ctypes as C
import filecmp
import os

import pytest

import oracle_lib as O
import synth
import synthetic_golden as SG
from iteres_b200 import capi


def to_bigwig(wig, sizes, out):
    err = C.create_string_buffer(capi.ERRLEN)
    rc = capi.lib().itx_wig_to_bigwig(wig.encode(), sizes.encode(), out.encode(), err)
    return rc, err.value.decode()


@pytest.mark.skipif(not os.path.exists(SG.MANIFEST), reason="no stored outputs of the reference under tests/golden/synthetic")
@pytest.mark.parametrize("shape,n_rmsk,mode,n_units", SG.BIGWIG_CASES)
def test_same_bytes_as_the_reference_binary(shape, n_rmsk, mode, n_units, tmp_path):
    d = str(tmp_path)
    s = synth.Synth(shape, n_rmsk, seed=SG.BIGWIG_SEED)
    cs, rs, rm = s.write_tables(d)
    bam = os.path.join(d, "reads.bam")
    SG.write_bam(s, bam, mode, n_units)
    s.close()
    have_ref = os.path.exists(O.REF_BIN)
    (SG.reference_stat if have_ref else SG.oracle_stat)((cs, rs, rm), bam, [], d, prefix="ref")
    want = SG.load()["bigwig"][SG.bigwig_case(shape, n_rmsk, mode, n_units)]
    for stem in SG.BIGWIG_STEMS:
        wig = os.path.join(d, stem + ".wig")
        assert SG.digest(wig) == want[stem]["wig"], stem          # the wiggle the reference built its bigWig from
        mine = os.path.join(d, stem + ".mine.bigWig")
        assert to_bigwig(wig, rs, mine) == (0, "")
        assert SG.digest(mine) == want[stem]["bigWig"], stem
        if have_ref:
            assert filecmp.cmp(mine, os.path.join(d, stem + ".bigWig"), shallow=False), stem


def test_errors_follow_the_reference(tmp_path):
    sizes = tmp_path / "rep.sizes"
    sizes.write_text("AluY\t300\nL1\t10\nAluY\t5\n")               # a later row of the same name wins
    wig = tmp_path / "x.wig"
    wig.write_text("")
    rc, msg = to_bigwig(str(wig), str(sizes), str(tmp_path / "x.bigWig"))
    assert rc == -2 and msg.endswith("is empty of data")         # bwgCreate.c:1108-1109
    wig.write_text("fixedStep chrom=L1 start=1 step=1 span=1\n" + "1\n" * 11)
    rc, msg = to_bigwig(str(wig), str(sizes), str(tmp_path / "x.bigWig"))
    assert rc == -2 and "has 10 bases, but item ends at 11" in msg
    wig.write_text("fixedStep chrom=AluY start=1 step=1 span=1\n" + "1\n" * 6)
    rc, msg = to_bigwig(str(wig), str(sizes), str(tmp_path / "x.bigWig"))
    assert rc == -2 and "has 5 bases" in msg
    wig.write_text("fixedStep chrom=MIR start=1 step=1 span=1\n1\n")
    rc, msg = to_bigwig(str(wig), str(sizes), str(tmp_path / "x.bigWig"))
    assert rc == -2 and "'MIR' not found" in msg
    wig.write_text("fixedStep chrom=L1 start=1 step=1 span=1\n" + "2\n" * 10)
    assert to_bigwig(str(wig), str(sizes), str(tmp_path / "x.bigWig")) == (0, "")
    assert to_bigwig(str(tmp_path / "nope.wig"), str(sizes), str(tmp_path / "x.bigWig"))[0] == -1
