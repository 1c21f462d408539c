"""k_inflate on DEFLATE streams that zlib never writes (tests/deflate_shapes.py): deep and flat codes, a single incomplete
distance code, literal-only blocks, many short blocks of mixed types, 258 as 284 + 31, matches 32768 bytes back and runs through
the edges of the match-copy windows.  A real BAM stream from the generator is cut into BGZF blocks of 40 bytes to 64 KiB and
block i is written in shape i mod S, so every warp of 8, 16 or 32 blocks decodes a mix of shapes in lock step.  The stream on
the device must be the stream that was compressed, byte for byte, and the counts and tables those of the host scan and the
oracle, through every second pass (ITX_LZ), every block density of the warp, the file and the pinned-image entry and the host
inflate.  Invalid streams in the middle of a valid file must fail the scan as a damaged block, and leave the index usable."""
import ctypes as C
import math
import struct
import zlib

import numpy as np
import pytest

import bamio
import deflate_shapes as DS
import oracle_lib as O
import synth
from iteres_b200 import capi
from test_gpu_parity import assert_same_tables

pytestmark = pytest.mark.gpu
SHAPES = list(DS.SHAPES)
# raw block sizes, cycled: the edges of the match-copy windows (1536 / 3072 / 6144), a few bytes, the largest block BGZF allows
SIZES_SMALL_FILE = [40, 65536, 257, 1536, 1537, 3072, 3073, 6144, 6145, 700, 20000, 12289, 100, 40000, 333, 32768, 9000]
SIZES_LARGE_FILE = [40, 257, 1536, 1537, 3072, 3073, 700, 2000, 1000, 333, 2500, 1200, 600]


def bgzf_block(comp, raw, isize=None):
    """one BGZF block around a raw-deflate stream; isize: the footer's ISIZE when it is not len(raw)"""
    bsize = 18 + len(comp) + 8 - 1
    assert bsize < 65536
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize) + comp +
            struct.pack("<II", zlib.crc32(raw) & 0xFFFFFFFF, len(raw) if isize is None else isize))


def shaped_blocks(raw, sizes, first=0):
    """raw cut into blocks of sizes[i % len] bytes (halved while the shape does not fit a BGZF block), block i written in shape
    SHAPES[(first + i) % S]"""
    out, off, i = [], 0, 0
    while off < len(raw):
        size, shape = sizes[i % len(sizes)], SHAPES[(first + i) % len(SHAPES)]
        while True:
            piece = raw[off:off + size]
            comp = DS.SHAPES[shape](DS.lz77(piece))
            if len(comp) + 26 <= 65536:
                break
            size //= 2
        out.append(bgzf_block(comp, piece))
        off += len(piece)
        i += 1
    return out


class World:
    def __init__(self, d):
        self.s = synth.Synth(1, 60000, seed=7)
        self.tables = self.s.write_tables(d)
        self.d = d
        self.files = {}

    def add(self, name, raw, blocks):
        path = "%s/%s.bam" % (self.d, name)
        with open(path, "wb") as f:
            for b in blocks:
                f.write(b)
            f.write(bamio.EOF_BLOCK)
        ix = capi.Index(*self.tables)
        a = np.frombuffer(raw + b"\0" * 64, dtype=np.uint8)
        want = ix.scan_bam_host(a.ctypes.data, len(raw), capi.default_opts())
        ix.close()
        ora = O.OracleIndex(*self.tables)
        assert ora.scan_stream(raw, O.default_opts()) == want
        self.files[name] = (path, raw, want, ora, len(blocks))


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    w = World(str(tmp_path_factory.mktemp("shapes")))
    # small: fewer than 4096 blocks, so the file is one short group (the tail launch, ITX_INF_TAIL_LANES blocks per warp)
    buf, n, _ = w.s.stream(1, 6000)
    raw = buf[:n].tobytes()
    hl = len(w.s.header())
    small = shaped_blocks(raw[:hl], [65536]) + shaped_blocks(raw[hl:], SIZES_SMALL_FILE, first=1)
    assert len(small) < 4096
    w.add("small", raw, small)
    # large: a group of more than 4096 blocks (ITX_INF_LANES blocks per warp).  The host caps a group at the file's bytes / 2048
    # + 64 blocks (the small-file estimate in scan_bgzf_device_inflate, iteres_b200/csrc/itx_gpu.cu), so the file needs more than
    # 8.4 MB of blocks of less than 2 KiB on average; the assert below restates that formula and fails if the estimate changes.
    # Its records are one piece of the generator's stream repeated: the repeats have the same blocks, so each block is written once.
    buf, n, _ = w.s.stream(1, 2000)
    rec = buf[hl:n].tobytes()
    period = shaped_blocks(rec, SIZES_LARGE_FILE)
    head = shaped_blocks(raw[:hl], [65536])
    per_bytes = sum(len(b) for b in period)
    m = max(math.ceil(8.8e6 / per_bytes), math.ceil(4400 / len(period)))
    large = head + period * m
    flen = sum(len(b) for b in large) + len(bamio.EOF_BLOCK)
    assert flen // 2048 + 64 > 4096 and len(large) > flen // 2048 + 64 + 32, (flen, len(large))
    w.add("large", raw[:hl] + rec * m, large)
    yield w
    for f in w.files.values():
        f[3].close()
    w.s.close()


def scan_checked(world, name, entry):
    path, raw, want, ora, _ = world.files[name]
    ix = capi.Index(*world.tables)
    if entry == "file":
        got = ix.scan_alignments(path, capi.default_opts())
    else:
        L = capi.lib()
        img = open(path, "rb").read()
        pin = L.itx_host_alloc_pinned(len(img) + 64)
        try:
            C.memmove(pin, img, len(img))
            got = ix.scan_bgzf_memory(pin, len(img), capi.default_opts())
        finally:
            L.itx_host_free_pinned(pin)
    assert got == want
    assert ix.stream_fetch(len(raw) + 100) == raw
    assert_same_tables(ix, ora)
    ix.close()


@pytest.mark.parametrize("entry", ["file", "pinned"])
@pytest.mark.parametrize("lanes", [8, 16, 32])
@pytest.mark.parametrize("lz", ["2", "0", "1"])
def test_mixed_shapes_small_file(lz, lanes, entry, world, monkeypatch):
    monkeypatch.delenv("ITX_INFLATE", raising=False)
    monkeypatch.setenv("ITX_LZ", lz)
    monkeypatch.setenv("ITX_INF_TAIL_LANES", str(lanes))
    scan_checked(world, "small", entry)


@pytest.mark.parametrize("lanes", [8, 16, 32])
@pytest.mark.parametrize("lz", ["2", "0", "1"])
def test_mixed_shapes_large_file(lz, lanes, world, monkeypatch):
    monkeypatch.delenv("ITX_INFLATE", raising=False)
    monkeypatch.setenv("ITX_LZ", lz)
    monkeypatch.setenv("ITX_INF_LANES", str(lanes))
    scan_checked(world, "large", "pinned" if lanes == 16 else "file")


@pytest.mark.parametrize("name", ["small", "large"])
def test_host_inflate_reads_the_shapes_too(name, world, monkeypatch):
    monkeypatch.setenv("ITX_INFLATE", "host")
    scan_checked(world, name, "file")


INVALID = DS.invalid_streams()


@pytest.mark.parametrize("inflate", ["device", "host"])
@pytest.mark.parametrize("bad", sorted(INVALID))
def test_invalid_block_fails_the_scan_and_the_index_recovers(bad, inflate, world, tmp_path, monkeypatch):
    monkeypatch.setenv("ITX_INFLATE", inflate)
    path, raw, want, ora, _ = world.files["small"]
    blocks = []
    with open(path, "rb") as f:
        img = f.read()
    off = 0
    while off < len(img):
        bsize = struct.unpack_from("<H", img, off + 16)[0] + 1
        blocks.append(img[off:off + bsize])
        off += bsize
    stream, isize, _ = INVALID[bad]
    k = len(blocks) // 2
    broken = str(tmp_path / "broken.bam")
    with open(broken, "wb") as f:
        f.write(b"".join(blocks[:k]) + bgzf_block(stream, b"", isize) + b"".join(blocks[k:]))
    ix = capi.Index(*world.tables)
    with pytest.raises(capi.ItxError) as e:
        ix.scan_alignments(broken, capi.default_opts())
    assert e.value.code == -2 and "inflate failed" in str(e.value)
    ix.reset()
    assert ix.scan_alignments(path, capi.default_opts()) == want
    assert ix.stream_fetch(len(raw) + 100) == raw
    ix.close()
