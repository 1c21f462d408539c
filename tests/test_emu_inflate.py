"""The device DEFLATE decoder (iteres_b200/csrc/itx_inflate.cuh, host build) against zlib: stored, fixed and
dynamic blocks, every compression level, several kinds of content incl. the BAM streams the generator makes,
and damaged input (must report an error, never run away).  Besides zlib's own streams, the decoder gets the shapes of
tests/deflate_shapes.py -- streams other BGZF writers produce and zlib never does -- and its invalid set."""
import functools
import random
import struct
import zlib

import numpy as np
import pytest

import deflate_shapes as DS
import emu_lib
import synth


def deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return co.compress(data) + co.flush()


def samples():
    rnd = random.Random(4)
    out = {
        "empty": b"",
        "one": b"A",
        "zeros": bytes(65280),
        "run": b"ab" * 30000,
        "random": bytes(rnd.getrandbits(8) for _ in range(40000)),
        "text": (b"the quick brown fox jumps over the lazy dog, " * 1400)[:65000],
        "lowent": bytes(rnd.choice(b"ACGT") for _ in range(65280)),
        "ramp": bytes(range(256)) * 250,
        "short_periods": b"".join(bytes([65 + i % 26]) * (3 + i % 7) + b"xyz" * (2 + i % 5) + b"abcdefg" * 3 for i in range(2500))[:65000],
        "triples": bytes(rnd.choice(b"ab") for _ in range(65000)),       # dense 3..6-byte matches: long match lists
        # the largest block BGZF allows (ISIZE 65536: positions fill 16 bits, the last window of the match copies is cut short)
        "max_block": (b"".join(bytes([65 + i % 26]) * (3 + i % 7) + b"xyz" * (2 + i % 5) + bytes(rnd.randrange(256) for _ in range(i % 11)) for i in range(4000)))[:65536],
        # runs of period 1..9 and far copies through every edge of the match-copy windows (1536, 3072, 6144 bytes)
        "windows": DS.periodic_runs(65536, 1),
        "far": DS.far_copies(65536, 2),                                   # every match 32768 bytes back
    }
    s = synth.Synth(0, 2000, seed=5)
    for mode in (0, 1, 2):
        buf, n, _ = s.stream(mode, 3000)
        out["bam%d" % mode] = buf[:n].tobytes()[: 0xff00]
        out["bam%d_tail" % mode] = buf[:n].tobytes()[0xff00: 2 * 0xff00]
    s.close()
    return out


SAMPLES = samples()


# every second pass the host build has: in line, listed, pointer jumping, and itx_lzw_resolve at 8192 / 2048 / 256 bytes and at
# the device's windows of 6144 / 3072 / 1536 bytes
DEFERS = [0, 1, 2, 3, 4, 5, 6, 7, 8]
SHAPE_SAMPLES = ["bam0", "text", "random", "run", "windows", "far", "max_block"]


@functools.lru_cache(maxsize=None)
def tokens(name):
    return DS.lz77(SAMPLES[name])


@functools.lru_cache(maxsize=None)
def shaped(name, shape):
    """SAMPLES[name] written by the shape (zlib has checked that it decodes to the sample)"""
    return DS.SHAPES[shape](tokens(name))


@pytest.mark.parametrize("defer", DEFERS)
@pytest.mark.parametrize("name,level", [(n, lv) for n in sorted(SAMPLES) for lv in (0, 1, 6, 9)] +
                         [(n, sh) for n in SHAPE_SAMPLES for sh in DS.SHAPES])
def test_matches_zlib(name, level, defer):
    """level 0..9: zlib's stream; a shape name: the stream deflate_shapes writes in that shape"""
    data = SAMPLES[name]
    comp = deflate(data, level) if isinstance(level, int) else shaped(name, level)
    rc, got = emu_lib.inflate(comp, len(data), defer=defer)
    assert rc == 0 and got == data


def test_shapes_hold_what_they_are_written_for():
    """the shapes above really contain the rare constructs, and the window samples really cross the windows.  FEATURES is
    emptied and every stream written again here (not taken from the cache), so the check sees only what these writes emit."""
    DS.FEATURES.clear()
    for n in SHAPE_SAMPLES:
        for sh in DS.SHAPES:
            DS.SHAPES[sh](tokens(n))
    assert DS.FEATURES >= {"16_across_trees", "16_after_17", "18_at_11", "18_at_138", "258_as_284+31", "lit_code_13_15",
                           "dist_code_13_15", "distance_32768", "empty_distance_tree", "empty_dynamic", "empty_stored",
                           "final_empty_fixed", "hclen_below_19", "single_incomplete_distance_code"}, DS.FEATURES
    for w in (1536, 3072, 6144):
        crossing, runs = DS.windows_crossed(tokens("windows"), w)
        assert crossing >= 5 and runs >= 3, (w, crossing, runs)
    assert len(SAMPLES["windows"]) == len(SAMPLES["max_block"]) == 65536
    assert sum(m[0] for m in tokens("far") if type(m) is tuple and m[1] == 32768) > 32000


@pytest.mark.parametrize("name", ["text", "bam0", "lowent", "one"])
def test_fixed_huffman_and_other_strategies(name):
    data = SAMPLES[name]
    for strat in (zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED):
        rc, got = emu_lib.inflate(deflate(data, 6, strat), len(data))
        assert rc == 0 and got == data, strat


def test_multi_block_stream_with_sync_flushes():
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    data = SAMPLES["text"]
    comp = b""
    for i in range(0, len(data), 7000):
        comp += co.compress(data[i:i + 7000]) + co.flush(zlib.Z_SYNC_FLUSH)      # stored empty blocks in between
    comp += co.flush()
    rc, got = emu_lib.inflate(comp, len(data))
    assert rc == 0 and got == data


def test_wrong_isize_and_damaged_streams_are_errors():
    data = SAMPLES["bam0"]
    comp = deflate(data, 6)
    assert emu_lib.inflate(comp, len(data) + 1, cap=len(data) + 1)[0] == 2           # ISIZE mismatch
    assert emu_lib.inflate(comp, len(data) - 5, cap=len(data) - 5)[0] != 0           # would overflow the block: refused
    assert emu_lib.inflate(comp[: len(comp) // 2], len(data))[0] != 0                # truncated
    rnd = random.Random(9)
    bad = 0
    for _ in range(200):
        b = bytearray(comp)
        for _ in range(3):
            b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
        rc, got = emu_lib.inflate(bytes(b), len(data))
        if rc != 0 or got != data:
            bad += 1
    assert bad > 150                                                                   # and none of them hung or crashed
    for _ in range(100):                                                               # pure noise
        junk = bytes(rnd.getrandbits(8) for _ in range(rnd.randrange(1, 300)))
        emu_lib.inflate(junk, 1000)
    # streams zlib rejects, each for one reason: a data error, or an output that is not ISIZE long
    for name, (stream, isize, want) in DS.invalid_streams().items():
        for defer in DEFERS:
            rc = emu_lib.inflate(stream, isize, defer=defer)[0]
            assert rc in ((1, 2) if want is None else (want,)), (name, defer, rc)


def test_bgzf_blocks_of_a_generated_bam(tmp_path):
    s = synth.Synth(1, 5000, seed=8)
    bam = str(tmp_path / "x.bam")
    n, nrec = s.write_bam(bam, 2, 4000, level=1, threads=2)
    buf, n2, _ = s.stream(2, 4000)
    raw = open(bam, "rb").read()
    off, out = 0, b""
    while off + 18 <= len(raw):
        bsize = struct.unpack_from("<H", raw, off + 16)[0] + 1
        isize = struct.unpack_from("<I", raw, off + bsize - 4)[0]
        rc, got = emu_lib.inflate(raw[off + 18: off + bsize - 8], isize)
        assert rc == 0
        out += got
        off += bsize
    assert out == buf[:n2].tobytes()
    s.close()
