"""-R on ONE BGZF file split across ranks (itx_shard_dedup_keys, itx_shard_dedup_fetch, itx_dedup_admit, itx_scan_shard_file_rmdup):
phase 1 settles every part and collects its unique fragments' keys, counting nothing; every rank admits the keys and flags of the
parts before its own with an ordinal below all of its own, counts its part with -R, and admits those of the parts after it.  The
summed counts are those of the single-device -R scan of the whole file, bit for bit.  The ranks run in turn on ONE device here, each
on an index of its own and the keys moved through the host, as tests/test_gpu_shard.py runs the plain protocol; the last tests run
itx_scan_alignments_shard (NCCL) and the command line on two devices."""
import filecmp
import os
import struct
import subprocess
import threading

import numpy as np
import pytest

import bamio
import kats
import oracle_lib as O
import synth
from iteres_b200 import capi
from test_gpu_parity import assert_same_tables
from test_gpu_shard import _kat_tables, assert_parts_equal_whole, run_parts

pytestmark = pytest.mark.gpu

RMDUP = dict(rmDup=1)


def or_flags(fl):
    out = 0
    for f in fl:
        out |= f
    return out


def phase1(tabs, path, nranks, opts, ixs=None):
    """phase 1 with the chain check, the ranks in turn -> (indexes, reports, keys per part, flags per part, ranks that ran again,
    keys each rank exported before it ran again)"""
    ixs = ixs or [capi.Index(*tabs) for _ in range(nranks)]
    res = [ixs[r].shard_dedup_keys(path, opts, r, nranks) for r in range(nranks)]
    first_keys = {}
    redone = []
    for _ in range(nranks + 1):
        bad, forced = capi.shard_chain_check([x[0] for x in res])
        if bad < 0:
            break
        first_keys.setdefault(bad, ixs[bad].shard_dedup_fetch(res[bad][1]))
        res[bad] = ixs[bad].shard_dedup_keys(path, opts, bad, nranks, forced)
        redone.append(bad)
    else:
        raise AssertionError("the parts do not chain: %r" % ([x[0] for x in res],))
    keys = [ixs[r].shard_dedup_fetch(res[r][1]) for r in range(nranks)]
    assert [len(k) for k in keys] == [x[1] for x in res]
    return ixs, [x[0] for x in res], keys, [x[2] for x in res], redone, first_keys


def run_file(tabs, path, nranks, opts, ixs=None, exchange=True):
    """one file of a run: phase 1, the keys through the host, phase 2 -> (indexes, keys per part, ranks that ran phase 1 again,
    keys exported before that)"""
    ixs, reps, keys, flags, redone, first_keys = phase1(tabs, path, nranks, opts, ixs)
    none = np.zeros((0, 2), dtype=np.uint64)
    for r in range(nranks):
        if exchange:
            ixs[r].dedup_admit(np.concatenate(keys[:r]) if r else none, or_flags(flags[:r]))
        _, rep = ixs[r].scan_shard_file_rmdup(path, opts, r, nranks, reps[r][0])
        assert rep == reps[r]
        if exchange:
            ixs[r].dedup_admit(np.concatenate(keys[r + 1:]) if r + 1 < nranks else none, or_flags(flags[r + 1:]))
    return ixs, keys, redone, first_keys


def write_stream(path, raw, level=1):
    with open(path, "wb") as f:
        for i in range(0, len(raw), 0xFF00):
            f.write(bamio.bgzf_block(raw[i:i + 0xFF00], level))
        f.write(bamio.EOF_BLOCK)


def doubled_bam(d, shape, n_rmsk, mode, n_units, seed):
    """a BAM whose reads come twice over (the second copy after the first): every key has a copy far from its first, in other
    parts than the first's whatever the number of ranks"""
    s = synth.Synth(shape, n_rmsk, seed=seed)
    tabs = s.write_tables(d)
    buf, n, _ = s.stream(mode, n_units)
    hdr_len = len(s.header())
    raw = buf[:n].tobytes()
    raw += raw[hdr_len:]
    bam = os.path.join(d, "reads.bam")
    write_stream(bam, raw)
    s.close()
    return tabs, bam


def close(ixs):
    for ix in ixs:
        ix.close()


@pytest.mark.parametrize("nranks", [2, 3, 5, 8])
@pytest.mark.parametrize("shape,mode,n_rmsk,n_units", [(2, 0, 3000, 150000), (1, 2, 60000, 100000)], ids=["chrM_se50", "pe100"])
def test_rmdup_parts_sum_to_the_whole(shape, mode, n_rmsk, n_units, nranks, tmp_path):
    d = str(tmp_path)
    tabs, bam = doubled_bam(d, shape, n_rmsk, mode, n_units, seed=41)
    opts = capi.default_opts(**RMDUP)
    whole = capi.Index(*tabs)
    want = whole.scan_alignments(bam, opts)
    ora = O.OracleIndex(*tabs)
    assert ora.scan_file(bam, O.default_opts(**RMDUP)) == want
    assert_same_tables(whole, ora)
    ixs, keys, redone, _ = run_file(tabs, bam, nranks, opts)
    assert_parts_equal_whole(ixs, whole)
    close(ixs)
    # phase 1 settles every part as the plain protocol does: from the same guesses, with the same ranks scanning again
    plain, _, plain_redone = run_parts(tabs, bam, nranks, capi.default_opts())
    close(plain)
    assert redone == plain_redone
    # the exchange is what makes them equal: keys are shared between parts, and the parts alone keep more reads
    allk = np.concatenate([k for k in keys if len(k)])
    assert len(np.unique(allk, axis=0)) < len(allk)
    alone, _, _, _ = run_file(tabs, bam, nranks, opts, exchange=False)
    assert sum(int(ix.cnt[11]) for ix in alone) > want[11]
    close(alone + [whole])
    ora.close()


def test_filter_rmdup_on_four_ranks(tmp_path):
    d = str(tmp_path)
    tabs, bam = doubled_bam(d, 1, 60000, 1, 60000, seed=42)
    opts = capi.default_opts(filter=1, diffSubfam=0, **RMDUP)
    whole = capi.Index(*tabs)
    want = whole.scan_alignments(bam, opts)
    ixs, _, _, _ = run_file(tabs, bam, 4, opts)
    assert [sum(int(ix.cnt[k]) for ix in ixs) for k in range(13)] == want
    got = sum((ix.elem_counts_by_row(0).astype(np.uint64) for ix in ixs), np.zeros(len(whole.elem_counts_by_row(0)), dtype=np.uint64))
    assert np.array_equal(got.astype(np.uint32), whole.elem_counts_by_row(0)) and int(got.sum()) == want[9] > 0
    gu = sum((ix.elem_counts_by_row(1).astype(np.uint64) for ix in ixs), np.zeros(len(whole.elem_counts_by_row(1)), dtype=np.uint64))
    assert np.array_equal(gu.astype(np.uint32), whole.elem_counts_by_row(1))
    close(ixs + [whole])


@pytest.mark.parametrize("first", ["unmapped", "unique", "nonunique"])
def test_the_nonunique_rule_across_a_part_boundary(first, tmp_path):
    """two parts in stored blocks (one BGZF block each, the first the larger, so that the second rank owns exactly the second):
    rank 1's part starts with a non-unique read.  It is the run's first non-unique read and comes before every unique read --
    kept -- only when rank 0's part holds neither kind of fragment."""
    d = str(tmp_path)
    tabs = _kat_tables(d)
    pad = [kats.se("u%d" % j, 4, 0, 0) for j in range(400)]                 # unmapped: not fragments
    lead = {"unmapped": [], "unique": [kats.se("x", 0, 900000, 37)], "nonunique": [kats.se("x", 0, 900000, 3)]}[first]
    part1 = [kats.se("n0", 0, 1050, 3)] + [kats.se("b%d" % j, 16 if j % 2 else 0, 1100 + 5 * j, 30) for j in range(40)]
    raw0 = bamio.encode_header([("chr1", 1000000)]) + b"".join(bamio.encode_record(r) for r in lead + pad)
    raw1 = b"".join(bamio.encode_record(r) for r in part1)
    assert len(raw0) < 0xFF00 and len(raw0) > 2 * len(raw1)
    bam = os.path.join(d, "reads.bam")
    with open(bam, "wb") as f:
        f.write(bamio.bgzf_block(raw0, 0) + bamio.bgzf_block(raw1, 0) + bamio.EOF_BLOCK)
    opts = capi.default_opts(**RMDUP)
    ora = O.OracleIndex(*tabs)
    want = ora.scan_stream(raw0 + raw1, O.default_opts(**RMDUP))
    whole = capi.Index(*tabs)
    assert whole.scan_alignments(bam, opts) == want
    ixs, _, _, _ = run_file(tabs, bam, 2, opts)
    assert int(ixs[0].cnt[0] + ixs[0].cnt[1]) == len(lead + pad) and int(ixs[1].cnt[0] + ixs[1].cnt[1]) == len(part1)   # each part holds what was put there
    assert_parts_equal_whole(ixs, whole)
    # n0 overlaps the AluY element, so it is counted exactly when it is kept; rank 1 alone (no admission) always keeps it
    solo, _, _, _ = run_file(tabs, bam, 2, opts, exchange=False)
    assert int(solo[1].cnt[9]) == int(ixs[1].cnt[9]) + (0 if first == "unmapped" else 1)
    close(ixs + solo + [whole])
    ora.close()


@pytest.mark.parametrize("second", ["other", "same"])
def test_rmdup_keys_persist_across_the_files_of_a_run(second, tmp_path):
    """a list a.bam,b.bam (or a.bam,a.bam) on 3 ranks: the second file's parts find every key of the first in their tables"""
    d = str(tmp_path)
    s = synth.Synth(2, 3000, seed=43)
    tabs = s.write_tables(d)
    a, b = os.path.join(d, "a.bam"), os.path.join(d, "b.bam")
    s.write_bam(a, 0, 60000, level=1, threads=4)
    synth.Synth(2, 3000, seed=44).write_bam(b, 0, 50000, level=1, threads=4)
    files = [a, b if second == "other" else a]
    opts = capi.default_opts(**RMDUP)
    whole = capi.Index(*tabs)
    want = whole.scan_alignments(",".join(files), opts)
    once = capi.Index(*tabs)
    first = once.scan_alignments(a, opts)
    if second == "same":
        assert want[11] == first[11]                            # the repeated file keeps none of its unique reads
    ixs = [capi.Index(*tabs) for _ in range(3)]
    for f in files:
        run_file(tabs, f, 3, opts, ixs)
    assert_parts_equal_whole(ixs, whole)
    close(ixs + [whole, once])
    s.close()


def test_a_wrong_first_record_guess_is_caught_between_ranks_with_rmdup(tmp_path):
    """the decoy carrier of test_gpu_shard.py: rank 1 guesses a decoy record inside the carrier's byte array, phase 1 collects the
    decoys' keys, the chain check sends it back -- and the keys it exports then are its real reads' alone"""
    d = str(tmp_path)
    tabs = _kat_tables(d)
    small = bamio.encode_record(kats.se("decoy", 0, 5100, 37))
    payload = small * (200 * 1024 // len(small))
    carrier = kats.se("carrier", 0, 1050, 37, aux=[("NM", "C", 0), ("ZB", "B", b"C" + struct.pack("<i", len(payload)) + payload)])
    reads = [kats.se("a%d" % j, 16 if j % 2 else 0, 1000 + 7 * (j % 40), 30 + j % 3, aux=[("NM", "C", 1)]) for j in range(300)]
    reads.append(carrier)
    reads += [kats.se("b%d" % j, 16 if j % 2 else 0, 1000 + 7 * (j % 40), 30 + j % 3, aux=[("NM", "C", 1)]) for j in range(300)]
    bam = os.path.join(d, "reads.bam")
    raw = bamio.write_bam(bam, [("chr1", 1000000)], reads, level=1)
    opts = capi.default_opts(**RMDUP)
    ora = O.OracleIndex(*tabs)
    want = ora.scan_stream(raw, O.default_opts(**RMDUP))
    whole = capi.Index(*tabs)
    assert whole.scan_alignments(bam, opts) == want
    ixs, keys, redone, first_keys = run_file(tabs, bam, 2, opts)
    assert redone == [1]
    starts = lambda k: set((k[:, 0] & 0xffffffff).tolist()) if len(k) else set()     # noqa: E731
    assert any(x >= 5000 for x in starts(first_keys[1]))          # the decoys' keys were collected by the guess ...
    assert not any(x >= 5000 for x in starts(keys[1]))            # ... and are gone after the second phase 1
    assert_parts_equal_whole(ixs, whole)
    close(ixs + [whole])
    ora.close()


def test_an_admission_that_makes_the_table_grow(tmp_path):
    """1.5 M keys admitted into a table made for 1 M (loads above 0.7 move it into one twice the size): the admission goes through
    and a -R scan afterwards judges its reads as before -- none of the admitted keys is a real read's"""
    d = str(tmp_path)
    s = synth.Synth(2, 3000, seed=45)
    tabs = s.write_tables(d)
    bam = os.path.join(d, "reads.bam")
    s.write_bam(bam, 0, 60000, level=1, threads=4)
    opts = capi.default_opts(**RMDUP)
    fresh = capi.Index(*tabs)
    want = fresh.scan_alignments(bam, opts)
    ix = capi.Index(*tabs)
    rng = np.random.RandomState(7)
    k = np.empty((1500000, 2), dtype=np.uint64)
    k[:, 0] = rng.randint(0, 1 << 62, size=len(k), dtype=np.int64).astype(np.uint64)
    k[:, 1] = np.uint64(0xfffff) << np.uint64(1)                  # a chromosome identity no reference has
    ix.dedup_admit(k[:700000], 0)
    ix.dedup_admit(k[700000:], 0)
    assert ix.scan_alignments(bam, opts) == want
    for which in range(3):
        assert ix.table(which) == fresh.table(which)
    close([ix, fresh])
    s.close()


def _ranks(ixs, fn):
    errs = []

    def rank(r):
        try:
            fn(r)
        except Exception as e:           # noqa: BLE001
            errs.append((r, e))
    th = [threading.Thread(target=rank, args=(r,)) for r in range(len(ixs))]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs


def test_two_gpus_rmdup(tmp_path):
    """itx_scan_alignments_shard with -R on two devices (NCCL all-gathers and broadcasts) + ONE allreduce = the single-device -R scan"""
    if capi.lib().itx_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    d = str(tmp_path)
    tabs, bam = doubled_bam(d, 2, 3000, 0, 150000, seed=46)
    opts = capi.default_opts(**RMDUP)
    whole = capi.Index(*tabs, device=0)
    want = whole.scan_alignments(bam, opts)
    world = 2
    ixs = [capi.Index(*tabs, device=r) for r in range(world)]
    uid = ixs[0].comm_unique_id()

    def run(r):
        ixs[r].comm_init(uid, r, world)
        ixs[r].scan_alignments_shard(bam + "," + bam, opts)
        ixs[r].allreduce_counts()
    _ranks(ixs, run)
    whole2 = capi.Index(*tabs, device=0)
    want2 = whole2.scan_alignments(bam + "," + bam, opts)
    assert want2[11] == want[11]
    for r in range(world):
        assert list(ixs[r].cnt) == want2, r
    assert ixs[0].profile()["rmdup_bcast_bytes"] > 0
    for which in range(3):
        assert ixs[0].table(which) == whole2.table(which)
    close(ixs + [whole, whole2])


def test_command_line_rmdup_on_two_gpus(tmp_path):
    """ITERES_GPUS=2 iteres stat -R / filter -R write the files ITERES_GPUS=1 writes"""
    if capi.lib().itx_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    d = str(tmp_path)
    tabs, bam = doubled_bam(d, 1, 60000, 2, 100000, seed=47)
    exe = os.path.join(os.path.dirname(capi.lib_path()), "iteres")
    for cmd in ("stat", "filter"):
        outs = []
        for n in (1, 2):
            od = os.path.join(d, "%s_%d" % (cmd, n))
            os.makedirs(od)
            p = subprocess.run([exe, cmd, "-R", "-o", "out", *tabs, bam], cwd=od, env=dict(os.environ, ITERES_GPUS=str(n)), capture_output=True, text=True)
            assert p.returncode == 0, p.stderr[-2000:]
            assert "one GPU" not in p.stderr
            outs.append(od)
        names = sorted(os.listdir(outs[0]))
        assert names == sorted(os.listdir(outs[1])) and names
        for fn in names:
            assert filecmp.cmp(os.path.join(outs[0], fn), os.path.join(outs[1], fn), shallow=False), (cmd, fn)
