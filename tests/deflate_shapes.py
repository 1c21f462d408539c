"""Raw DEFLATE (RFC 1951) written in plain Python, in shapes that zlib's compressor never produces but other BGZF writers do
(libdeflate, Intel's deflater, ...): deep and flat Huffman codes, a single incomplete distance code, literal-only blocks with an
empty distance tree, many short blocks of mixed types, code-length headers with other repeat patterns, 258 as 284 + 31.  A TEST
HELPER, not product code: the tests feed these streams to the device inflater and compare its output with the input bytes.

zlib writes none of these streams; it only checks them.  Every positive stream is decoded by zlib.decompressobj(-15) to exactly
its input before it is returned, and every stream of the invalid set is asserted to be rejected by zlib.

Tokens: a literal is an int 0..255, a match a tuple (length, distance).  `lz77` makes them for one BGZF block; every shape is a
function tokens -> raw-deflate bytes.  FEATURES collects which rare constructs the writer emitted, so that a test can check that
the shapes still cover what they are meant to cover."""
import bisect
import random
import zlib

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
             8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8          # symbols 0..287 (286/287 have codes but are invalid)
FIXED_DIST = [5] * 32                                             # codes 0..31 (30/31 invalid)

FEATURES = set()


def _len_code(n, via284=False):
    """length 3..258 -> (symbol, extra bits, extra value)"""
    if n == 258 and via284:
        FEATURES.add("258_as_284+31")
        return 284, 5, 31
    k = bisect.bisect_right(LEN_BASE, n) - 1
    if n == 258:
        k = 28
    return 257 + k, LEN_EXTRA[k], n - LEN_BASE[k]


def _dist_code(d):
    k = bisect.bisect_right(DIST_BASE, d) - 1
    return k, DIST_EXTRA[k], d - DIST_BASE[k]


def _rev(c, n):
    r = 0
    for _ in range(n):
        r = (r << 1) | (c & 1)
        c >>= 1
    return r


class BitWriter:
    """LSB-first bit packing (RFC 1951 3.1.1); Huffman codes go MSB-first, so `canonical` hands them out bit-reversed"""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def bits(self, v, n):
        assert 0 <= v < (1 << n) or n == 0 and v == 0, (v, n)
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)

    def raw(self, data):
        assert self.n == 0
        self.out += data

    def getvalue(self):
        self.align()
        return bytes(self.out)


def canonical(lengths):
    """RFC 1951 3.2.2: the canonical code of every symbol, bit-reversed for BitWriter.bits"""
    count = [0] * 16
    for ln in lengths:
        count[ln] += 1
    count[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    out = [0] * len(lengths)
    for s, ln in enumerate(lengths):
        if ln:
            out[s] = _rev(nxt[ln], ln)
            nxt[ln] += 1
    return out


def kraft_left(lengths, maxbits=15):
    """code space left over, in units of 2^-maxbits: 0 complete, < 0 over-subscribed, > 0 incomplete"""
    return (1 << maxbits) - sum((1 << maxbits) >> ln for ln in lengths if ln)


def fit_lengths(lengths, maxbits, keep=(), prefer=()):
    """Make the code lengths a complete prefix code of at most maxbits bits: over-subscription is removed by lengthening the longest
    codes still below maxbits, the rest of the code space is handed out by shortening codes (those in `prefer` first, the shortest
    that fits first).  Symbols in `keep` are left alone."""
    L = [min(ln, maxbits) for ln in lengths]
    K = 1 << maxbits
    left = kraft_left(L, maxbits)
    while left < 0:
        ln, s = max((ln, s) for s, ln in enumerate(L) if 0 < ln < maxbits and s not in keep)
        L[s] += 1
        left += K >> (ln + 1)
    while left > 0:
        cand = [(s not in prefer, ln, s) for s, ln in enumerate(L) if ln > 1 and (K >> ln) <= left and s not in keep]
        if not cand:                                                # nothing left to shorten: code an unused symbol too
            s = next(s for s, ln in enumerate(L) if not ln and s not in keep)
            L[s] = maxbits
            left -= 1
            continue
        _, ln, s = min(cand)
        L[s] -= 1
        left -= K >> ln
    return L


def huffman_lengths(freqs, maxbits):
    """Huffman code lengths of the used symbols, limited to maxbits; one used symbol gets a 1-bit code"""
    import heapq
    used = [s for s, f in enumerate(freqs) if f]
    L = [0] * len(freqs)
    if len(used) == 1:
        L[used[0]] = 1
    if len(used) <= 1:
        return L
    heap = [(freqs[s], s, [s]) for s in used]
    heapq.heapify(heap)
    while len(heap) > 1:
        fa, ta, a = heapq.heappop(heap)
        fb, tb, b = heapq.heappop(heap)
        for s in a + b:
            L[s] += 1
        heapq.heappush(heap, (fa + fb, min(ta, tb), a + b))
    return fit_lengths(L, maxbits) if max(L) > maxbits else L


def deep_lengths(freqs):
    """a complete code that puts the frequent symbols on 13..15-bit codes: the frequent seven eighths ask for 13, 14, 15 bits in
    turn and the rest of the code space goes to the rare symbols"""
    used = sorted((s for s, f in enumerate(freqs) if f), key=lambda s: (-freqs[s], s))
    L = [0] * len(freqs)
    if len(used) <= 2:
        for s in used:
            L[s] = 1
        return L
    n_rare = max(1, len(used) // 8)
    for i, s in enumerate(used):
        L[s] = 13 + i % 3
    return fit_lengths(L, 15, prefer=set(used[len(used) - n_rare:]))


# ---------------------------------------------------------------------------------------------------------------- token source
def lz77(data, chain=8, max_dist=32768):
    """greedy LZ77 over one block: hash of three bytes, the `chain` most recent candidates, the nearest of the longest matches"""
    data = bytes(data)
    n = len(data)
    head, prev = {}, [-1] * n
    toks = []
    i = 0

    def insert(p):
        if p + 3 <= n:
            k = data[p:p + 3]
            prev[p] = head.get(k, -1)
            head[k] = p

    while i < n:
        best, bd = 0, 0
        lim = min(258, n - i)
        if lim >= 3:
            j, c = head.get(data[i:i + 3], -1), chain
            while j >= 0 and c and i - j <= max_dist:
                if data[j + best] == data[i + best] if best < lim else False:
                    ln = 0
                    while ln + 16 <= lim and data[j + ln:j + ln + 16] == data[i + ln:i + ln + 16]:
                        ln += 16
                    while ln < lim and data[j + ln] == data[i + ln]:
                        ln += 1
                    if ln > best:
                        best, bd = ln, i - j
                        if ln == lim:
                            break
                j, c = prev[j], c - 1
        if best >= 3:
            toks.append((best, bd))
            for p in range(i, i + best):
                insert(p)
            i += best
        else:
            toks.append(data[i])
            insert(i)
            i += 1
    return toks


def expand(tokens):
    out = bytearray()
    for t in tokens:
        if type(t) is int:
            out.append(t)
        else:
            ln, d = t
            assert 1 <= d <= len(out) and d <= 32768
            for _ in range(ln):
                out.append(out[-d])
    return bytes(out)


def windows_crossed(tokens, w):
    """matches that start before a multiple of w (counted from the block's start) and end after it, and how many of them are runs"""
    pos, cross, runs = 0, 0, 0
    for t in tokens:
        if type(t) is int:
            pos += 1
            continue
        ln, d = t
        if (pos // w) != ((pos + ln - 1) // w):
            cross += 1
            runs += d < ln
        pos += ln
    return cross, runs


# ---------------------------------------------------------------------------------------------------------------- block writers
def _freqs(tokens, via284):
    lf, df = [0] * 286, [0] * 30
    for t in tokens:
        if type(t) is int:
            lf[t] += 1
        else:
            lf[_len_code(t[0], via284)[0]] += 1
            df[_dist_code(t[1])[0]] += 1
    lf[256] += 1
    return lf, df


def _body(bw, tokens, llens, dlens, via284):
    lc, dc = canonical(llens), canonical(dlens)
    for t in tokens:
        if type(t) is int:
            assert llens[t]
            bw.bits(lc[t], llens[t])
        else:
            s, ne, ev = _len_code(t[0], via284)
            d, dne, dev = _dist_code(t[1])
            assert llens[s] and dlens[d], (s, d)
            bw.bits(lc[s], llens[s])
            bw.bits(ev, ne)
            bw.bits(dc[d], dlens[d])
            bw.bits(dev, dne)
            if t[1] == 32768:
                FEATURES.add("distance_32768")
    bw.bits(lc[256], llens[256])


def stored_block(bw, data, final, nlen_xor=0):
    """data <= 65535 bytes; nlen_xor != 0 writes a wrong NLEN"""
    bw.bits(final, 1)
    bw.bits(0, 2)
    bw.align()
    bw.bits(len(data), 16)
    bw.bits((len(data) ^ 0xffff) ^ nlen_xor, 16)
    bw.raw(data)
    if not data:
        FEATURES.add("empty_stored")


def fixed_block(bw, tokens, final, via284=False):
    bw.bits(final, 1)
    bw.bits(1, 2)
    _body(bw, tokens, FIXED_LIT, FIXED_DIST, via284)
    if not tokens and final:
        FEATURES.add("final_empty_fixed")


def rle(seq, mode, boundary):
    """the code-length sequence as (symbol, repeat extra) pairs.  zlib: runs inside each tree, 17/18 for zeros, value + 16s
    otherwise.  cross: the same over the whole sequence, so a run may go from the literal/length lengths into the distance ones.
    plain: no repeat codes.  zero16: a run of zeros as 17 (3 zeros) followed by 16s, which repeat the zero of the 17.  edge18: zero
    runs as 18 at 138 and 18 at 11."""
    out = []
    parts = [seq] if mode in ("cross", "plain") else [seq[:boundary], seq[boundary:]]
    for part in parts:
        i = 0
        while i < len(part):
            v, r = part[i], 1
            while i + r < len(part) and part[i + r] == v:
                r += 1
            i += r
            if mode == "plain":
                out += [(v, 0)] * r
                continue
            if v == 0 and mode == "zero16" and r >= 6:
                out.append((17, 0))
                r -= 3
                FEATURES.add("16_after_17")
                while r >= 3:
                    k = min(r, 6)
                    out.append((16, k - 3))
                    r -= k
                out += [(0, 0)] * r
                continue
            if v == 0 and mode == "edge18":
                while r >= 138:
                    out.append((18, 127))
                    r -= 138
                    FEATURES.add("18_at_138")
                while r >= 11:
                    out.append((18, 0))
                    r -= 11
                    FEATURES.add("18_at_11")
                if r >= 3:
                    out.append((17, r - 3))
                    r = 0
                out += [(0, 0)] * r
                continue
            if v == 0:
                while r >= 11:
                    k = min(r, 138)
                    out.append((18, k - 11))
                    r -= k
                if r >= 3:
                    out.append((17, r - 3))
                    r = 0
                out += [(0, 0)] * r
                continue
            out.append((v, 0))
            r -= 1
            while r >= 3:
                k = min(r, 6)
                out.append((16, k - 3))
                r -= k
            out += [(v, 0)] * r
    return out


def _rle_covers(syms):
    """(first position, count) of the lengths each (symbol, extra) pair of an rle list stands for"""
    pos, i = [], 0
    for s, e in syms:
        n = 1 if s < 16 else (3 + e if s < 18 else 11 + e)
        pos.append((i, n))
        i += n
    return pos


def dynamic_header(bw, llens, dlens, final, mode="zlib", hclen=None, hlit=None, hdist=None, syms=None, cl_lens=None):
    """BFINAL, BTYPE 2 and the code-length header.  hlit / hdist are the 5-bit field values (default: as few as the lengths
    need); syms / cl_lens override the repeat-coded sequence and the code-length code (invalid streams)"""
    nl = len(llens) if hlit is None else hlit + 257
    nd = len(dlens) if hdist is None else hdist + 1
    seq = (list(llens) + [0] * 32)[:nl] + (list(dlens) + [0] * 32)[:nd]
    if syms is None:
        syms = rle(seq, mode, nl)
        for (a, n), (s, _) in zip(_rle_covers(syms), syms):
            if s == 16 and a < nl < a + n:
                FEATURES.add("16_across_trees")
    if cl_lens is None:
        f = [0] * 19
        for s, _ in syms:
            f[s] += 1
        if sum(1 for x in f if x) == 1:                       # a code of one symbol would be incomplete: give it a partner
            f[0 if not f[0] else 8] += 1
        cl_lens = huffman_lengths(f, 7)
    n_cl = max([i + 1 for i, s in enumerate(CL_ORDER) if cl_lens[s]] + [4])
    if hclen is not None:
        n_cl = max(n_cl, hclen)
    if n_cl < 19:
        FEATURES.add("hclen_below_19")
    bw.bits(final, 1)
    bw.bits(2, 2)
    bw.bits(nl - 257, 5)
    bw.bits(nd - 1, 5)
    bw.bits(n_cl - 4, 4)
    for i in range(n_cl):
        bw.bits(cl_lens[CL_ORDER[i]], 3)
    cc = canonical(cl_lens)
    for s, e in syms:
        assert cl_lens[s], s
        bw.bits(cc[s], cl_lens[s])
        if s == 16:
            bw.bits(e, 2)
        elif s == 17:
            bw.bits(e, 3)
        elif s == 18:
            bw.bits(e, 7)


def _trim(lens, minimum):
    n = len(lens)
    while n > minimum and lens[n - 1] == 0:
        n -= 1
    return list(lens[:n])


def dynamic_block(bw, tokens, final, llens, dlens, via284=False, **hdr):
    for k, ln in enumerate(llens):
        if ln >= 13:
            FEATURES.add("lit_code_13_15")
    for ln in dlens:
        if ln >= 13:
            FEATURES.add("dist_code_13_15")
    if sum(1 for x in dlens if x) == 1 and kraft_left(dlens) > 0:
        FEATURES.add("single_incomplete_distance_code")
    if not any(dlens):
        FEATURES.add("empty_distance_tree")
    if not tokens:
        FEATURES.add("empty_dynamic")
    dynamic_header(bw, _trim(llens, 257), _trim(dlens, 1), final, **hdr)
    _body(bw, tokens, llens, dlens, via284)


# ---------------------------------------------------------------------------------------------------------------- shapes
def checked(stream, data):
    """zlib decodes the stream to exactly `data` and reaches its end: the writer wrote a valid stream"""
    d = zlib.decompressobj(-15)
    got = d.decompress(stream) + d.flush()
    assert got == data and d.eof and not d.unused_data, "the helper wrote a stream zlib does not decode to its input"
    return stream


def _one_dynamic(tokens, llens_of, dlens_of, via284=False, **hdr):
    lf, df = _freqs(tokens, via284)
    bw = BitWriter()
    dynamic_block(bw, tokens, 1, llens_of(lf), dlens_of(df), via284, **hdr)
    return checked(bw.getvalue(), expand(tokens))


def shape_optimal(tokens):
    """one dynamic block, Huffman lengths limited to 15 bits, the header coded as zlib codes it"""
    return _one_dynamic(tokens, lambda f: huffman_lengths(f, 15), lambda f: huffman_lengths(f, 15))


def shape_deep(tokens):
    """frequent literal/length and distance symbols on 13..15-bit codes; zero runs as 18 at 11 and at 138"""
    return _one_dynamic(tokens, deep_lengths, deep_lengths, mode="edge18")


def shape_flat(tokens):
    """every literal/length symbol coded, on 8 or 9 bits (the 60 most frequent on 9: past the 8-bit look-up table), every
    distance symbol on 4 or 5 bits; no repeat codes in the header"""
    def ll(f):
        order = sorted(range(286), key=lambda s: (-f[s], s))
        L = [8] * 286
        for s in order[:60]:
            L[s] = 9
        return L

    def dl(f):
        order = sorted(range(30), key=lambda s: (f[s], s))
        L = [5] * 30
        for s in order[:2]:
            L[s] = 4
        return L
    return _one_dynamic(tokens, ll, dl, mode="plain")


def shape_single_distance_code(tokens):
    """only the matches of the most frequent distance code stay, and that code is the distance tree's only one (1 bit: an
    incomplete code, which RFC 1951 allows for one distance code); zero runs as a 17 followed by 16s"""
    toks, c = _keep_one_distance_code(tokens, expand(tokens))
    return _one_dynamic(toks, lambda f: huffman_lengths(f, 15), lambda f: [0] * c + [1], mode="zero16")


def _keep_one_distance_code(tokens, data):
    """the matches whose distance code is the most frequent one, every other match spelled out as literals"""
    df = [0] * 30
    for t in tokens:
        if type(t) is not int:
            df[_dist_code(t[1])[0]] += 1
    c = max(range(30), key=lambda d: (df[d], -d))
    out, pos = [], 0
    for t in tokens:
        if type(t) is int:
            out.append(t)
            pos += 1
        else:
            if _dist_code(t[1])[0] == c:
                out.append(t)
            else:
                out += list(data[pos:pos + t[0]])
            pos += t[0]
    return out, c


def shape_literal_only(tokens):
    """every match spelled out as literals, the distance tree empty (HDIST 1, length 0); the header's runs cross from the
    literal/length lengths into the distance lengths"""
    toks = list(expand(tokens))
    return _one_dynamic(toks, lambda f: huffman_lengths(f, 15), lambda f: [0], mode="cross")


def shape_fixed(tokens):
    """fixed Huffman codes only, in three blocks"""
    bw = BitWriter()
    k = len(tokens)
    cuts = [0, k // 3, 2 * k // 3, k]
    for i in range(3):
        fixed_block(bw, tokens[cuts[i]:cuts[i + 1]], int(i == 2))
    return checked(bw.getvalue(), expand(tokens))


def shape_via284(tokens):
    """optimal codes, but every length 258 written as code 284 with extra bits 31; all 19 code-length code lengths sent"""
    return _one_dynamic(tokens, lambda f: huffman_lengths(f, 15), lambda f: huffman_lengths(f, 15), via284=True, hclen=19)


def shape_cross16(tokens):
    """a 16 that repeats the last literal/length length into the first distance lengths: HLIT 286, literal/length symbols 284
    and 285 and distance symbols 0 and 1 all on 5 bits (every distance symbol coded, 28 on 5 bits and 2 on 4)"""
    def ll(f):
        L = huffman_lengths(f, 15)
        L[284] = L[285] = 5
        return fit_lengths(L, 15, keep={284, 285})
    return _one_dynamic(tokens, ll, lambda f: [5] * 28 + [4, 4], mode="cross")


def shape_split(k, seed):
    """k blocks (k up to a few hundred) of mixed types -- stored, fixed, dynamic with each header style, an empty dynamic block,
    empty stored blocks in between -- and a final empty fixed block"""
    def make(tokens):
        rnd = random.Random(seed * 7919 + len(tokens))
        n = len(tokens)
        cuts = sorted([0, n] + [rnd.randrange(n + 1) for _ in range(k - 1)])
        data = expand(tokens)
        bw = BitWriter()
        pos = 0
        modes = ["zlib", "plain", "zero16", "edge18", "cross"]
        for i in range(k):
            piece = tokens[cuts[i]:cuts[i + 1]]
            nbytes = sum(1 if type(t) is int else t[0] for t in piece)
            kind = i % 4
            if kind == 0:
                chunk = data[pos:pos + nbytes]
                for a in range(0, max(len(chunk), 1), 65535):
                    stored_block(bw, chunk[a:a + 65535], 0)
            elif kind == 1:
                fixed_block(bw, piece, 0, via284=bool(i & 4))
            else:
                lf, df = _freqs(piece, False)
                dyn = deep_lengths if i % 3 == 0 else (lambda f: huffman_lengths(f, 15))
                dl = dyn(df)
                if not any(dl):
                    dl = [0] if i % 2 else [1]                   # no match in the piece: an empty tree or one unused 1-bit code
                dynamic_block(bw, piece, 0, dyn(lf), dl, mode=modes[i % 5], hclen=19 if i % 7 == 0 else None)
            pos += nbytes
            if i % 7 == 3:
                stored_block(bw, b"", 0)
            if i == k // 2:
                dynamic_block(bw, [], 0, [0] * 256 + [1], [0])   # an empty dynamic block: only the end-of-block code, 1 bit
        fixed_block(bw, [], 1)
        return checked(bw.getvalue(), data)
    make.__name__ = "shape_split%d" % k
    return make


SHAPES = {
    "optimal": shape_optimal,
    "deep": shape_deep,
    "flat": shape_flat,
    "single_dist": shape_single_distance_code,
    "literal_only": shape_literal_only,
    "fixed": shape_fixed,
    "split200": shape_split(200, 1),
    "split9": shape_split(9, 2),
    "via284": shape_via284,
    "cross16": shape_cross16,
}


# ---------------------------------------------------------------------------------------------------------------- contents
def periodic_runs(size, seed, edges=(1536, 3072, 6144)):
    """random bytes with runs of period 1..9 that straddle every multiple of the match-copy windows, and copies of earlier
    bytes across them: the matches the greedy matcher finds there cross the window edges"""
    rnd = random.Random(seed)
    out = bytearray(rnd.getrandbits(8) for _ in range(min(size, 64)))
    step = min(edges)
    edge = step
    k = 0
    while len(out) < size:
        # up to a few bytes before the edge, then a run (or a far copy) through it
        lead = rnd.randrange(1, 12)
        while len(out) < edge - lead and len(out) < size:
            out += bytes(rnd.getrandbits(8) for _ in range(min(edge - lead - len(out), 97)))
            if rnd.random() < 0.3 and len(out) > 400:
                a = rnd.randrange(len(out) - 300)
                out += out[a:a + rnd.randrange(3, 40)]
        p = 1 + k % 9
        unit = bytes(rnd.getrandbits(8) for _ in range(p))
        if k % 5 == 4 and len(out) > 2000:
            a = rnd.randrange(len(out) - 1500)
            out += out[a:a + rnd.randrange(20, 300)]              # a copy from far back across the edge
        else:
            out += (unit * (300 // p + 2))[:rnd.randrange(12, 290)]
        edge += step
        k += 1
    return bytes(out[:size])


def far_copies(size, seed):
    """32768 random bytes and then the same bytes again: every match is 32768 bytes back"""
    rnd = random.Random(seed)
    head = bytes(rnd.getrandbits(8) for _ in range(32768))
    return (head + head)[:size]


# ---------------------------------------------------------------------------------------------------------------- invalid streams
def _dyn_stream(llens, dlens, tokens=(), **hdr):
    bw = BitWriter()
    dynamic_header(bw, llens, dlens, 1, **hdr)
    lc = canonical(llens)
    for t in tokens:
        bw.bits(lc[t], llens[t])
    bw.bits(0x2b5, 10)                                             # a few more bits: the stream does not simply run out
    return bw.getvalue() + b"\x5a\xa5\x33"


def _rejected(stream, isize):
    d = zlib.decompressobj(-15)
    try:
        got = d.decompress(stream) + d.flush()
    except zlib.error:
        return True
    return not d.eof or len(got) != isize


def invalid_streams(seed=3):
    """name -> (raw deflate, ISIZE, expected status).  Status 1 is a data error (ITX_INF_EDATA), 2 an output of another size
    than ISIZE (ITX_INF_ESIZE), None either of the two (output longer than ISIZE: the decoder may stop at the first byte too
    many or at the end of the stream).  zlib rejects every one of them."""
    rnd = random.Random(seed)
    text = b"the quick brown fox jumps over the lazy dog " * 40
    good_tokens = lz77(text)
    lf, df = _freqs(good_tokens, False)
    L, D = _trim(huffman_lengths(lf, 15), 257), _trim(huffman_lengths(df, 15), 1)
    out = {}

    ll = [8] * 286                                                  # 286 codes of 8 bits: 30 too many
    out["oversubscribed_literal_tree"] = (_dyn_stream(ll, [1, 1]), 100, 1)
    ll = [0] * 286
    ll[65], ll[256] = 2, 1                                          # two codes, a quarter of the code space unused
    out["incomplete_literal_tree"] = (_dyn_stream(ll, [1, 1], [65, 65, 256]), 2, 1)
    ll = [0] * 286
    ll[97], ll[98], ll[256], ll[258], ll[260] = 2, 2, 2, 3, 3
    dl = [1, 2]                                                     # two distance codes, a quarter unused
    bw = BitWriter()
    dynamic_block(bw, [97, 98, (6, 2), (4, 1)], 1, ll, dl)
    out["incomplete_distance_tree"] = (bw.getvalue(), 12, 1)
    ll = [0] * 286
    ll[97], ll[98] = 1, 1                                           # no end-of-block code
    out["missing_end_of_block"] = (_dyn_stream(ll, [1, 1], [97, 98, 97]), 3, 1)
    out["repeat_code_16_first"] = (_dyn_stream(L, D, syms=[(16, 1)] + rle(L + D, "zlib", len(L))), len(text), 1)
    short = rle(L + D[:-1], "zlib", len(L))                         # all lengths but the last, then three zeros
    out["repeat_past_the_last_length"] = (_dyn_stream(L, D, syms=short + [(17, 0)]), len(text), 1)
    for f in (30, 31):
        out["hlit_%d" % (f + 257)] = (_dyn_stream(L + [0] * 2, D, hlit=f), len(text), 1)
        out["hdist_%d" % (f + 1)] = (_dyn_stream(L, D + [0] * 2, hdist=f), len(text), 1)
    out["oversubscribed_code_length_code"] = (_dyn_stream(L, D, cl_lens=[1] * 19), len(text), 1)
    cl = [0] * 19
    cl[0], cl[8] = 2, 1                                             # one code of 1 bit and one of 2: incomplete
    out["incomplete_code_length_code"] = (_dyn_stream([8] * 256 + [8], [0], syms=[(8, 0)] * 257 + [(0, 0)], cl_lens=cl), 1, 1)
    for s in (286, 287):
        bw = BitWriter()
        bw.bits(1, 1)
        bw.bits(1, 2)
        fc = canonical(FIXED_LIT)
        for b in b"abc":
            bw.bits(fc[b], 8)
        bw.bits(fc[s], 8)                                           # a length code beyond 285
        bw.bits(0, 5)
        bw.bits(fc[256], 7)
        out["fixed_symbol_%d" % s] = (bw.getvalue(), 6, 1)
    hist = bytes(rnd.getrandbits(8) for _ in range(60000))
    for d in (30, 31):
        bw = BitWriter()
        stored_block(bw, hist, 0)
        bw.bits(1, 1)
        bw.bits(1, 2)
        fc, dc = canonical(FIXED_LIT), canonical(FIXED_DIST)
        bw.bits(fc[257], 7)                                         # length 3
        bw.bits(dc[d], 5)                                           # distance code 30 / 31, whose base (32769 / 49153) lies within the
        bw.bits(0, 14)                                              # 60000 bytes written so far: only the code check refuses it
        bw.bits(fc[256], 7)
        out["fixed_distance_code_%d" % d] = (bw.getvalue(), 60003, 1)
    bw = BitWriter()
    fixed_block(bw, list(b"0123456789") + [(3, 11)], 1)             # 11 bytes back after 10
    out["distance_beyond_output"] = (bw.getvalue(), 13, 1)
    bw = BitWriter()
    stored_block(bw, b"stored bytes", 1, nlen_xor=0x10)
    out["stored_len_nlen_mismatch"] = (bw.getvalue(), 12, 1)
    good = shape_optimal(good_tokens)
    out["output_shorter_than_isize"] = (good, len(text) + 1, 2)
    out["output_longer_than_isize"] = (good, len(text) - 1, None)
    for name, (stream, isize, _) in out.items():
        assert _rejected(stream, isize), "zlib accepts the invalid stream " + name
    return out
