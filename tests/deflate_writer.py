"""Designed deflate streams for the PNG decoder (test-only).

Every file the rest of the suite decodes was written by zlib (``zlib.compressobj``, ``cv2.imencode``).  zlib never writes
several shapes inflate accepts and other encoders do write: single-code or empty distance trees, code-length repeats that
cross from the literal / length lengths into the distance lengths (zopfli, libdeflate), literal-only blocks with HLIT 257,
an empty dynamic block, length symbol 284 with extra bits 31, codes of 11 - 15 bits in use.  ``Stream`` builds a zlib
stream from an explicit list of blocks - stored, fixed or dynamic, with the exact code lengths of both trees, the exact
code-length run encoding and HCLEN, and tokens whose symbols and extra bits may be chosen - and ``png_file`` wraps the
inflated bytes in a PNG file whose rows are exactly those bytes (8-bit gray, or RGB / RGBA for long rows).

``corpus()`` yields the designs: header shapes, block layouts (a dynamic block at every residue of a stream word, stored
blocks behind Huffman blocks ending at every residue), symbolic history across block and group starts and the 32 KiB edge,
decoys (stored payloads made of real dynamic headers: false candidates of the device's block-start search) and the
files the decoder declines on purpose.  What each design reaches is not taken on trust: the tests read it from the block
records ``Stream`` keeps.
"""
from __future__ import annotations

import heapq
import zlib
from dataclasses import dataclass, field
from functools import lru_cache

import numpy as np

from oracle import png_decode_model as M
from oracle.png_model import BitOut

# RFC 1951 3.2.5: length symbols 257 .. 285 and distance codes 0 .. 29 (base value, extra bits)
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
             8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
CL_EXTRA = {16: 2, 17: 3, 18: 7}

# the decoder's limits (csrc/p2p_pngdec.cuh kMaxSyms, kWindow; p2p_api_pngdec.inl kPdHostBudget, pd_layout)
MAX_SYMS = 1 << 20
WINDOW = 32768
HOST_BUDGET = 8 << 20


def cap_list(stream_len):
    return min(max(stream_len // 8, 1 << 16), 1 << 26)


def cap_cand(stream_len):
    return min(stream_len // 512 + 1024, 1 << 24)


def cap_blocks(stream_len, raw_bytes):
    return cap_cand(stream_len) + min(raw_bytes // 65535 + 1024, 1 << 24)


def group_size(nb):
    m = 1
    while m * m < nb:
        m += 1
    return m


def len_symbol(length):
    """(symbol, extra bits, extra value) zlib would use for a match length 3 .. 258"""
    if length == 258:
        return 285, 0, 0
    i = max(k for k in range(28) if LEN_BASE[k] <= length)
    return 257 + i, LEN_EXTRA[i], length - LEN_BASE[i]


def dist_symbol(dist):
    i = max(k for k in range(30) if DIST_BASE[k] <= dist)
    return i, DIST_EXTRA[i], dist - DIST_BASE[i]


def match_length(sym, extra):
    return LEN_BASE[sym - 257] + extra


def match_dist(code, extra):
    return DIST_BASE[code] + extra


def canonical(lens):
    """Canonical Huffman codes of a list of code lengths (0 = no code), bit-reversed for the LSB-first stream."""
    maxl = max(lens) if lens else 0
    bl_count = [0] * (maxl + 2)
    for l in lens:
        if l:
            bl_count[l] += 1
    code, nxt = 0, [0] * (maxl + 2)
    for bits in range(1, maxl + 1):
        code = (code + bl_count[bits - 1]) << 1
        nxt[bits] = code
    out = {}
    for s, l in enumerate(lens):
        if l:
            c = nxt[l]
            nxt[l] += 1
            out[s] = int(format(c, f"0{l}b")[::-1], 2)
    return out


def kraft(lens):
    return sum(2.0 ** -l for l in lens if l)


def chain_lengths(n, maxlen=None):
    """Lengths of a complete code of n >= 2 codes whose longest code has maxlen bits (default n - 1): the chain 1, 2, ..,
    maxlen, maxlen, then the shortest leaf split in two until there are n."""
    maxlen = maxlen or n - 1
    assert n <= 1 << maxlen
    lens = list(range(1, maxlen)) + [maxlen, maxlen]
    while len(lens) < n:
        l = min(x for x in lens if x < maxlen)
        lens.remove(l)
        lens += [l + 1, l + 1]
    return sorted(lens)


def flat_lengths(n):
    """Lengths of a complete code of n codes, as equal as possible (n = 1: the single code of length 1)."""
    if n == 1:
        return [1]
    k = (n - 1).bit_length()
    short = (1 << k) - n
    return [k - 1] * short + [k] * (n - short)


def huff_lengths(freq, limit):
    """{symbol: code length} of a Huffman code for {symbol: count}; a flat complete code when the tree is deeper than limit."""
    syms = sorted(freq)
    if len(syms) == 1:
        return {syms[0]: 1}
    heap = [(freq[s], i, (s,)) for i, s in enumerate(syms)]
    heapq.heapify(heap)
    depth = {s: 0 for s in syms}
    k = len(heap)
    while len(heap) > 1:
        f1, _, a = heapq.heappop(heap)
        f2, _, b = heapq.heappop(heap)
        for s in a + b:
            depth[s] += 1
        heapq.heappush(heap, (f1 + f2, k, a + b))
        k += 1
    if max(depth.values()) <= limit:
        return depth
    return dict(zip(syms, flat_lengths(len(syms))))


def rle_lengths(seq):
    """The code-length run encoding of seq as one sequence: [(symbol, extra)].  Runs cross from the literal / length lengths
    into the distance lengths wherever the values continue (zlib encodes the two trees apart; zopfli and libdeflate do not)."""
    out, i, n = [], 0, len(seq)
    while i < n:
        v = seq[i]
        j = i
        while j < n and seq[j] == v:
            j += 1
        r = j - i
        if v == 0:
            while r >= 11:
                k = min(r, 138)
                out.append((18, k - 11))
                r -= k
            if r >= 3:
                out.append((17, r - 3))
                r = 0
            out += [(0, 0)] * r
        else:
            out.append((v, 0))
            r -= 1
            while r >= 3:
                k = min(r, 6)
                out.append((16, k - 3))
                r -= k
            out += [(v, 0)] * r
        i = j
    return out


def expand_runs(runs):
    seq = []
    for s, e in runs:
        if s < 16:
            seq.append(s)
        elif s == 16:
            seq += [seq[-1]] * (3 + e)
        elif s == 17:
            seq += [0] * (3 + e)
        else:
            seq += [0] * (11 + e)
    return seq


FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 30


@dataclass
class Rec:
    """What one block of a designed stream is: the tests read coverage from these."""
    kind: str
    final: bool
    start: int
    end: int = 0
    out_off: int = 0
    out_len: int = 0
    n_tokens: int = 0
    hlit: int = 0
    hdist: int = 0
    hclen: int = 0
    litlens: list = field(default_factory=list)
    distlens: list = field(default_factory=list)
    cl_runs: list = field(default_factory=list)
    cl_lens: list = field(default_factory=list)
    lsyms: set = field(default_factory=set)    # (length symbol, extra value) pairs used
    dsyms: set = field(default_factory=set)    # (distance code, extra value) pairs used
    lits: set = field(default_factory=set)
    match_srcs: list = field(default_factory=list)   # (offset in the block, distance, length)


class Stream:
    """A zlib stream built block by block.  Tokens: an int (literal) or (length, distance) or (length, distance, length
    symbol, length extra) to choose the symbol (284 + 31 for 258).  The inflated bytes are kept (``data``)."""

    def __init__(self, cmf=0x78, flevel=2):
        self.bo = BitOut()
        flg = flevel << 6
        flg |= (31 - ((cmf << 8) | flg) % 31) % 31
        self.bo.send(cmf, 8)
        self.bo.send(flg, 8)
        self.cmf, self.flg = cmf, flg
        self.data = bytearray()
        self.recs: list[Rec] = []

    def bit(self):
        return self.bo.tell()

    def _start(self, kind, final, btype):
        r = Rec(kind, bool(final), self.bit(), out_off=len(self.data))
        self.bo.send(1 if final else 0, 1)
        self.bo.send(btype, 2)
        return r

    def _end(self, r):
        r.end = self.bit()
        r.out_len = len(self.data) - r.out_off
        self.recs.append(r)
        return r

    def stored(self, payload, final=False, nlen=None):
        r = self._start("stored", final, 0)
        pad = (-self.bit()) & 7
        self.bo.send(0, pad)
        n = len(payload)
        self.bo.send(n, 16)
        self.bo.send((n ^ 0xFFFF) if nlen is None else nlen, 16)
        for b in payload:
            self.bo.send(b, 8)
        self.data += bytes(payload)
        return self._end(r)

    def _tokens(self, r, tokens, lcode, llen, dcode, dlen):
        bo, data = self.bo, self.data
        for t in tokens:
            if isinstance(t, int):
                bo.send(lcode[t], llen[t])
                data.append(t)
                r.lits.add(t)
                continue
            L, D = t[0], t[1]
            if len(t) > 2:
                ls, le = t[2], t[3]
                assert match_length(ls, le) == L
                lx = LEN_EXTRA[ls - 257]
            else:
                ls, lx, le = len_symbol(L)
            ds, dx, de = dist_symbol(D)
            bo.send(lcode[ls], llen[ls])
            bo.send(le, lx)
            bo.send(dcode[ds], dlen[ds])
            bo.send(de, dx)
            r.lsyms.add((ls, le))
            r.dsyms.add((ds, de))
            r.match_srcs.append((len(data) - r.out_off, D, L))
            if D <= len(data):
                for _ in range(L):
                    data.append(data[-D])
            else:   # a designed invalid distance: nothing sensible to produce
                data += bytes(L)
        bo.send(lcode[256], llen[256])
        r.n_tokens = len(tokens)

    def fixed(self, tokens, final=False):
        r = self._start("fixed", final, 1)
        lc, dc = canonical(FIXED_LIT), canonical(FIXED_DIST + [5, 5])
        self._tokens(r, tokens, lc, FIXED_LIT, dc, FIXED_DIST + [5, 5])
        return self._end(r)

    def dynamic(self, tokens, final=False, litlens=None, distlens=None, cl_runs=None, cl_lens=None, hclen=None, hlit=None,
                hdist=None):
        """A dynamic block.  litlens / distlens: the exact code lengths (their lengths are HLIT / HDIST), else Huffman codes
        of the tokens (HLIT / HDIST as small as possible unless given; no distance used: the empty distance tree);
        cl_runs: the exact code-length run encoding, else ``rle_lengths``; cl_lens: the 19 code-length code lengths by
        symbol, else a Huffman code of the runs (a second code when only one symbol is used: that code must be complete);
        hclen: code-length code lengths sent (default: as few as possible)."""
        if litlens is None:
            f = {256: 1}
            for t in tokens:
                s = t if isinstance(t, int) else (t[2] if len(t) > 2 else len_symbol(t[0])[0])
                f[s] = f.get(s, 0) + 1
            hl = huff_lengths(f, 15)
            n = hlit or max(257, max(hl) + 1)
            litlens = [hl.get(s, 0) for s in range(n)]
        if distlens is None:
            f = {}
            for t in tokens:
                if not isinstance(t, int):
                    d = dist_symbol(t[1])[0]
                    f[d] = f.get(d, 0) + 1
            hd = huff_lengths(f, 15) if f else {}
            n = hdist or max(1, max(hd, default=0) + 1)
            distlens = [hd.get(s, 0) for s in range(n)]
        seq = list(litlens) + list(distlens)
        if cl_runs is None:
            cl_runs = rle_lengths(seq)
        assert expand_runs(cl_runs) == seq, "the code-length runs do not spell the code lengths"
        if cl_lens is None:
            f = {}
            for s, _ in cl_runs:
                f[s] = f.get(s, 0) + 1
            if len(f) == 1:
                f[next(s for s in (0, 1, 2) if s not in f)] = 1
            h = huff_lengths(f, 7)
            cl_lens = [h.get(s, 0) for s in range(19)]
        need = max(i for i in range(19) if cl_lens[CL_ORDER[i]]) + 1
        hclen = max(4, need) if hclen is None else hclen
        assert hclen >= need
        r = self._start("dynamic", final, 2)
        bo = self.bo
        bo.send(len(litlens) - 257, 5)
        bo.send(len(distlens) - 1, 5)
        bo.send(hclen - 4, 4)
        for i in range(hclen):
            bo.send(cl_lens[CL_ORDER[i]], 3)
        cc = canonical(cl_lens)
        for s, e in cl_runs:
            bo.send(cc[s], cl_lens[s])
            if s >= 16:
                bo.send(e, CL_EXTRA[s])
        r.hlit, r.hdist, r.hclen = len(litlens), len(distlens), hclen
        r.litlens, r.distlens, r.cl_runs, r.cl_lens = list(litlens), list(distlens), list(cl_runs), list(cl_lens)
        lc, dc = canonical(list(litlens)), canonical(list(distlens))
        self._tokens(r, tokens, lc, list(litlens), dc, list(distlens))
        return self._end(r)

    def pad_to(self, residue, final=False):
        """A fixed block of literals 0 (8 bits) and 144 (9 bits) after which the next block starts at stream bit
        residue (mod 32)."""
        delta = (residue - self.bit()) % 32
        b = (delta - 10) % 8
        a8 = delta - 10 - 9 * b
        while a8 < 0:
            a8 += 32
        return self.fixed([144] * b + [0] * (a8 // 8), final=final)

    def zlib(self):
        bo = BitOut()
        bo.buf, bo.acc, bo.n = bytearray(self.bo.buf), self.bo.acc, self.bo.n
        bo.windup()
        return bytes(bo.buf) + (zlib.adler32(bytes(self.data)) & 0xFFFFFFFF).to_bytes(4, "big")


def png_file(data, z, stride=None, idat=1 << 20):
    """A PNG file whose zlib stream is z and whose inflated image is data: rows of ``stride`` bytes (default: one row),
    8-bit gray when the row fits, else RGB / RGBA / gray + alpha.  Every row must start with a filter type 0 .. 4."""
    data = bytes(data)
    stride = stride or len(data)
    assert len(data) % stride == 0, (len(data), stride)
    assert all(data[k] <= 4 for k in range(0, len(data), stride)), "a row starts with a byte that is not a filter type"
    rb = stride - 1
    for ctype, bpp in ((0, 1), (6, 4), (2, 3), (4, 2)):
        if rb % bpp == 0 and rb // bpp < 32767:
            break
    else:
        raise ValueError(f"no 8-bit PNG format has rows of {rb} bytes")
    ihdr = rb // bpp, len(data) // stride
    out = M.SIG + M.chunk(b"IHDR", ihdr[0].to_bytes(4, "big") + ihdr[1].to_bytes(4, "big") + bytes([8, ctype, 0, 0, 0]))
    for at in range(0, len(z), idat):
        out += M.chunk(b"IDAT", z[at:at + idat])
    return out + M.chunk(b"IEND", b"")


@dataclass
class Design:
    name: str
    png: bytes
    z: bytes
    data: bytes
    recs: list
    features: tuple
    expect: str = "decode"   # decode | decline:<class> | overflow | invalid
    decoys: list = field(default_factory=list)   # (stream bit, kind) of the false candidates placed on purpose

    @property
    def n_blocks(self):
        return len(self.recs)


def _design(name, s, features, stride=None, expect="decode", decoys=()):
    z = s.zlib()
    return Design(name, png_file(s.data, z, stride), z, bytes(s.data), s.recs, tuple(features), expect, list(decoys))


def _rand(rng, n, hi=256):
    return [int(v) for v in rng.integers(0, hi, n)]


def _fill(s, stride, final=True):
    """A last fixed block of zeros that completes the last row (rows of ``stride`` bytes)."""
    m = (-len(s.data)) % stride
    toks = [0] if m else []
    m -= len(toks)
    while m >= 3:
        k = min(258, m)
        if 0 < m - k < 3:
            k -= 3
        toks.append((k, 1))
        m -= k
    return s.fixed(toks + [0] * m, final=final)


# ---- headers -----------------------------------------------------------------------------------------------------
def headers():
    rng = np.random.default_rng(1)
    out = []
    # literal-only blocks with HLIT 257 and an empty distance tree (HDIST 1 / 30, all zero); a single-code distance tree;
    # a literal tree holding only end-of-block; HLIT 286 / HDIST 30 with repeats across their boundary
    s = Stream()
    s.dynamic([0] + _rand(rng, 600))
    s.dynamic(_rand(rng, 300), distlens=[0] * 30)
    s.dynamic(_rand(rng, 40, 16) + [(10, 7), (20, 7), (3, 7)], distlens=[0, 0, 0, 0, 0, 1])          # one distance code, 1 bit
    s.dynamic([], litlens=[0] * 256 + [1], distlens=[0])                                               # only end-of-block
    s.dynamic([], litlens=[0] * 256 + [1], distlens=[0] * 30)
    s.dynamic(_rand(rng, 200, 8) + [(5, 3), (7, 100)], hlit=286, hdist=30)                             # zero run 262 .. 301
    # a 16 run across HLIT / HDIST: literal / length lengths end in 5s (280 .. 285), the distance lengths start with 5s
    lit = [0] * 286
    lit[0:12] = [4] * 12
    lit[256] = 4
    lit[280:286] = [5] * 6
    dist = [5] * 28 + [4] * 2
    assert kraft(lit) == 1.0 and kraft(dist) == 1.0
    s.dynamic(_rand(rng, 300, 12) + [(131, 1), (200, 2), (258, 40), (227, 250), (258, 300), (194, 1000)], litlens=lit, distlens=dist)
    # exact code-length runs: 18 x 138 (extra 127), a 16 run of threes across HLIT / HDIST
    lit = [3] * 6 + [0] * 250 + [3, 3]                      # HLIT 258: literals 0 .. 5, end-of-block, length 3
    dist = [3] * 4 + [2] * 2
    runs = [(3, 0), (16, 2), (18, 127), (18, 101), (3, 0), (16, 2), (2, 0), (2, 0)]
    s.dynamic(_rand(rng, 50, 6) + [(3, 1), (3, 2), (3, 3), (3, 4), (3, 5), (3, 7)], litlens=lit, distlens=dist, cl_runs=runs)
    # every literal / length code length 1 .. 15 in use, and distance codes of 1 .. 15 bits in use
    syms = list(range(13)) + [256, 257, 258]       # 16 symbols: chain 1 .. 15, 15
    lit = [0] * 259
    for sym, l in zip(syms, chain_lengths(16)):
        lit[sym] = l
    dist = [0] * 16
    for d, l in zip(range(16), chain_lengths(16)):
        dist[d] = l
    toks = list(range(13)) * 2 + [(3, DIST_BASE[d]) for d in range(16)] + [(4, DIST_BASE[d] + (DIST_EXTRA[d] and 1)) for d in range(16)]
    s.dynamic(toks, litlens=lit, distlens=dist)
    # a code-length code with 7-bit codes (19 code-length symbols, the longest 7 bits); HCLEN 19
    lit = [0] * 286
    vals = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 15]
    for sym, l in zip(list(range(15)) + [256], vals):
        lit[sym] = l
    dist = [0] * 30
    cl = [0] * 19
    for sym, l in zip(range(19), chain_lengths(19, 7)):
        cl[sym] = l
    s.dynamic(list(range(15)) * 2, litlens=lit, distlens=dist, cl_lens=cl)
    # HCLEN 5 .. 19: literal lengths all 8 (255 literals + end-of-block), empty distance tree: code-length symbols 8 and 0
    lit = [8] * 255 + [0] + [8]
    for h in range(5, 20):
        s.dynamic(_rand(rng, 20, 255), litlens=lit, distlens=[0], hclen=h, final=h == 19)
    out.append(_design("headers", s, ["hlit257", "hlit286", "hdist1", "hdist30", "empty_dist_tree", "single_code_dist_tree",
                                      "eob_only_literal_tree", "cross_boundary_repeats", "18x138", "lit_lengths_1_15",
                                      "dist_lengths_9_15", "cl_7bit", "hclen_5_19"]))
    # all 29 length symbols and all 30 distance codes at their smallest and largest extra values (distance 32768, 284 + 31)
    s = Stream()
    s.dynamic([0] + _rand(rng, 33000, 5))
    toks = []
    for k in range(29):
        for le in sorted({0, (1 << LEN_EXTRA[k]) - 1}):
            for de_max in (False, True):
                d = (k * 2 + de_max) % 30
                de = (1 << DIST_EXTRA[d]) - 1 if de_max else 0
                toks.append((match_length(257 + k, le), match_dist(d, de)))
    for d in range(30):
        for de in sorted({0, (1 << DIST_EXTRA[d]) - 1}):
            toks.append((3 + d % 5, match_dist(d, de)))
    toks.append((258, 32768, 284, 31))
    toks += [(258, 32768), (258, 1, 284, 31)]
    s.dynamic(toks, hlit=286, hdist=30)
    s.fixed([(258, 32768, 284, 31), (258, 32768)] + _rand(rng, 10, 5))
    _fill(s, 4096)
    out.append(_design("all_lengths_and_distances", s, ["all_length_symbols", "all_distance_codes", "284+31", "dist32768"], 4096))
    return out


# ---- layout --------------------------------------------------------------------------------------------------------
def layout():
    rng = np.random.default_rng(2)
    out = []
    # a dynamic block starting at every residue 0 .. 31 of a stream word (fixed pads in between), each reaching back
    s = Stream()
    s.dynamic([0] + _rand(rng, 500))
    for r in rng.permutation(32):
        s.pad_to(int(r))
        assert s.bit() % 32 == r
        s.dynamic(_rand(rng, int(rng.integers(20, 200))) + [(int(rng.integers(3, 259)), int(rng.integers(1, 400)))])
    s.fixed([], final=True)
    out.append(_design("dynamic_at_every_residue", s, ["residues_0_31", "fixed_between_dynamic", "dynamic_first_at_16"]))
    # stored blocks behind Huffman blocks ending at every residue; LEN 0; empty fixed blocks (the Z_PARTIAL_FLUSH shape)
    s = Stream()
    s.dynamic([0] + _rand(rng, 300))
    for r in range(32):
        s.pad_to(r)
        s.stored(bytes(_rand(rng, int(rng.integers(0, 40)))))
        s.dynamic(_rand(rng, 50) + [(20, 51)])
        s.fixed([])
        s.stored(b"")
    s.dynamic(_rand(rng, 30), final=True)
    out.append(_design("stored_after_every_residue", s, ["stored_after_huffman_residues", "stored_len0", "empty_fixed"]))
    # stored blocks of LEN 65535 (two, then a match of distance 32768 into them), an empty final stored block
    s = Stream()
    s.stored(bytes([0]) + bytes(_rand(rng, 65534, 5)))
    s.dynamic([(258, 32768)] * 3 + _rand(rng, 100, 5))
    s.stored(bytes(_rand(rng, 65535, 5)))
    n = (-(len(s.data) + 1)) % 4096
    s.fixed([(258, 32768)] * (n // 258) + [1] * (n % 258) + [2])
    s.stored(b"", final=True)
    out.append(_design("stored_65535", s, ["stored_len65535", "empty_final_stored"], 4096))
    # empty final blocks of every kind; the shortest final dynamic block right in front of the Adler-32
    for kind in ("fixed", "dynamic"):
        s = Stream()
        s.dynamic([0] + _rand(rng, 700) + [(40, 300)])
        if kind == "fixed":
            s.fixed([], final=True)
        else:
            s.dynamic([], final=True, litlens=[0] * 256 + [1], distlens=[0])
        out.append(_design(f"empty_final_{kind}", s, [f"empty_final_{kind}", "final_dynamic_last_word"]))
    return out


# ---- history -------------------------------------------------------------------------------------------------------
def history():
    rng = np.random.default_rng(3)
    out = []
    # matches whose source straddles the block start, distance below the length; a source at the block's first byte
    s = Stream()
    s.dynamic([0] + _rand(rng, 400))
    for d in (1, 2, 3, 31, 32, 33, 257, 258):
        s.dynamic([(258, d), (d, 258 + d) if d >= 3 else (3, 258 + 3), (10, 258 + 3 + max(d, 3))] + _rand(rng, 30) +
                  [(5, 300), (7, 43)])
        s.dynamic(_rand(rng, 5) + [(40, 5), (40, 45 + d)] + [(int(rng.integers(3, 100)), int(rng.integers(1, 600))) for _ in range(20)])
    s.fixed([], final=True)
    out.append(_design("straddling_matches", s, ["straddle_1_2_3_31_32_33_257_258", "source_at_block_start"]))
    # blocks of exactly 32767, 32768, 32769 output bytes, each followed by distance-32768 matches
    for n in (32767, 32768, 32769):
        s = Stream()
        s.dynamic([0] + _rand(rng, 5000, 5))
        toks = []
        while sum(1 if isinstance(t, int) else t[0] for t in toks) < n - 300:
            toks += _rand(rng, 20, 5) + [(int(rng.integers(3, 259)), int(rng.integers(1, 5000)))]
        rest = n - sum(1 if isinstance(t, int) else t[0] for t in toks)
        toks += _rand(rng, rest, 5)
        r = s.dynamic(toks)
        assert r.out_len == n
        s.dynamic([(258, 32768)] * 200 + [(100, 32768), (3, 32767), (4, 32769 - 1)] + _rand(rng, 10, 5))
        _fill(s, 4096)
        out.append(_design(f"block_of_{n}", s, [f"out_len_{n}", "dist32768_after"], 4096))
    # the first byte of a block's last 32 KiB as a history source: seven blocks (groups of three); block 4 is 33,000 bytes of
    # history marks (distance-32768 matches from its first byte on), block 5 is empty, and block 6 opens with a
    # distance-32768 match whose source is exactly that byte - re-based by the group walk, made final by the chain walk
    s = Stream()
    for n in (11000, 11000, 11000, 5):
        s.dynamic(_row_literals(rng, len(s.data), n))
    s.dynamic([(258, 32768)] * 127 + [(234, 32768)])
    s.dynamic([], litlens=[0] * 256 + [1], distlens=[0])
    s.dynamic([(258, 32768)] + _row_literals(rng, len(s.data) + 258, 100))
    _fill(s, 4096)
    out.append(_design("tail_window_edges", s, ["tail_window_first_byte", "chain_window_first_byte"], 4096))
    # nb = k^2 - 1, k^2, k^2 + 1 tiny blocks: chains through every group, marks at exactly the group start and one before
    for k in (2, 3, 5, 8):
        for nb in (k * k - 1, k * k, k * k + 1):
            out.append(_groups(nb, rng))
    for nb in (1, 2, 3):
        out.append(_groups(nb, rng, name=f"nb_{nb}"))
    return out


def _groups(nb, rng, name=None):
    per = group_size(nb)
    s = Stream()
    starts = []
    for i in range(nb):
        starts.append(len(s.data))
        n_out = int(rng.integers(150, 400))
        toks, o = [], 0
        if i == 0:
            toks, o = [0] + _rand(rng, 40), 41
        gs = starts[(i // per) * per]
        if i % per == 1:   # the group's second block opens with marks at exactly its group start and one in front of it
            toks, o = [(3, starts[i] - gs)] + ([(4, starts[i] + 3 - gs + 1)] if gs else []), 3 + (4 if gs else 0)
        while o < n_out:
            here = starts[i] + o
            pick = int(rng.integers(0, 6))
            if i % per and pick == 0 and here - gs <= WINDOW:                 # a mark at exactly the group start
                toks.append((int(rng.integers(3, 12)), here - gs))
            elif i % per and pick == 1 and 0 < gs and here - gs + 1 <= WINDOW:   # one in front of it
                toks.append((int(rng.integers(3, 12)), here - gs + 1))
            elif pick in (2, 3) and here > 0:                              # into the block before, or far back
                toks.append((int(rng.integers(3, 40)), int(rng.integers(1, min(here, WINDOW) + 1))))
            elif pick == 4 and i > 0:                                         # just in front of this block's start
                toks.append((int(rng.integers(3, 30)), o + int(rng.integers(1, 8))))
            else:
                toks.append(int(rng.integers(0, 256)))
            o += 1 if isinstance(toks[-1], int) else toks[-1][0]
        s.dynamic(toks, final=i == nb - 1)
    return _design(name or f"groups_nb_{nb}", s, [f"nb_{nb}", f"group_size_{per}", "mark_at_gs", "mark_at_gs_minus_1"])


def _row_literals(rng, at, n, row=4096):
    """n random literals written from output position at on: 0 at the row starts (rows of ``row`` bytes)."""
    return [0 if (at + i) % row == 0 else int(v) for i, v in enumerate(rng.integers(0, 256, n))]


def _row_tokens(rng, at, n, far=4096):
    """Tokens of exactly n output bytes starting at output position at (a row start: the first byte is literal 0),
    literals and matches reaching up to ``far`` bytes back."""
    toks, o = [0], 1
    while o < n:
        if n - o >= 3 and rng.integers(0, 3) == 0:
            L = int(rng.integers(3, min(258, n - o) + 1))
            toks.append((L, int(rng.integers(1, min(far, at + o) + 1))))
            o += L
        else:
            toks.append(int(rng.integers(0, 256)))
            o += 1
    return toks


# ---- decoys --------------------------------------------------------------------------------------------------------
def _decoy_bits(kind, rng):
    """The bits (LSB first) of a dynamic block used as a false candidate: 'block' decodes to its end-of-block (a different
    block); 'bad' is the header of a tree that holds only end-of-block (code '0') followed by a '1' (no such code); 'long'
    is a header without its end-of-block code whose tree is literal 0 = '0', literal 1 = '10', end-of-block = '11': zeros
    and isolated ones decode as literals for ever."""
    s = Stream()
    s.bo = BitOut()
    if kind == "block":
        s.dynamic(_rand(rng, 12, 4) + [(3, 2)])
    elif kind == "bad":
        s.dynamic([], litlens=[0] * 256 + [1], distlens=[0])
    else:
        lit = [0] * 257
        lit[0], lit[1], lit[256] = 1, 2, 2
        s.dynamic([], litlens=lit, distlens=[0])
    bo = s.bo
    bits = [(byte >> k) & 1 for byte in bo.buf for k in range(8)] + [(bo.acc >> k) & 1 for k in range(bo.n)]
    if kind == "bad":
        bits[-1] = 1
    elif kind == "long":
        bits = bits[:-2]
    return bits


def _pack(bits):
    bits = bits + [0] * ((-len(bits)) % 8)
    return bytes(sum(b << k for k, b in enumerate(bits[i:i + 8])) for i in range(0, len(bits), 8))


def decoy_payload(n_units, kinds, rng, unit=24, row=4096, shift0=0):
    """(stored data, [(bit in the data, kind)]): rows of ``row`` bytes, each a 0 and then as many whole decoy units of
    ``unit`` bytes as fit; the header of unit k sits at bit shift (shift0 + k) mod 32 of the unit's first byte."""
    per_row = (row - 1) // unit
    out, at = bytearray(), []
    for k in range(n_units):
        if k % per_row == 0:
            if out:
                out += bytes((-len(out)) % row)
            out.append(0)
        sh = (shift0 + k) % 32
        kind = kinds[k % len(kinds)]
        b = _pack([0] * sh + _decoy_bits(kind, rng))
        assert len(b) <= unit, len(b)
        at.append((8 * len(out) + sh, kind))
        out += b + bytes(unit - len(b))
    out += bytes((-len(out)) % row)
    return bytes(out), at


def stream_bits(z):
    """The deflate data of zlib stream z as a list of bits in stream order (LSB first), the Adler-32 left out."""
    return np.unpackbits(np.frombuffer(z[:-4], np.uint8), bitorder="little").tolist()


def _complete_or_single(lens):
    """inftrees.c's rule for literal / length and distance codes: not over-subscribed, and complete unless the code is a
    single code of length 1 (or empty)."""
    left, used = 1.0, [l for l in lens if l]
    for l in used:
        left -= 2.0 ** -l
    return left >= 0 and (left == 0 or used in ([], [1]))


def _decoder(lens):
    return {(l, int(format(c, f"0{l}b")[::-1], 2)): s for s, c in canonical(lens).items() for l in [lens[s]]}


def measure(bits, bit, out_cap, wsize=WINDOW):
    """A one-block inflate of the dynamic block at stream bit ``bit`` (bits: ``stream_bits``), the way the decoder
    measures a candidate: ('ok', end bit, bytes) at its end-of-block; ('bad', ..) at whatever inflate rejects, at more
    bytes than out_cap or past the end of the data; ('long', ..) when MAX_SYMS symbols pass without end-of-block."""
    n_bits, pos = len(bits), bit

    def get(n):
        nonlocal pos
        v = sum(bits[pos + k] << k for k in range(n) if pos + k < n_bits)
        pos += n
        return v

    def sym(dec):
        nonlocal pos
        code = 0
        for l in range(1, 16):
            code = (code << 1) | (bits[pos] if pos < n_bits else 0)
            pos += 1
            s = dec.get((l, code))
            if s is not None:
                return s
        return None

    if get(3) >> 1 != 2:
        return "bad", pos, 0
    hlit, hdist, hclen = get(5) + 257, get(5) + 1, get(4) + 4
    if hlit > 286 or hdist > 30:
        return "bad", pos, 0
    cl = [0] * 19
    for i in range(hclen):
        cl[CL_ORDER[i]] = get(3)
    if kraft(cl) != 1.0:
        return "bad", pos, 0
    cdec, lens = _decoder(cl), []
    while len(lens) < hlit + hdist:
        s = sym(cdec)
        if s < 16:
            lens.append(s)
            continue
        if s == 16 and not lens:
            return "bad", pos, 0
        v, rep = (lens[-1], 3 + get(2)) if s == 16 else (0, 3 + get(3)) if s == 17 else (0, 11 + get(7))
        if len(lens) + rep > hlit + hdist:
            return "bad", pos, 0
        lens += [v] * rep
    ll, dl = lens[:hlit], lens[hlit:]
    if not ll[256] or not _complete_or_single(ll) or not _complete_or_single(dl):
        return "bad", pos, 0
    ldec, ddec, o = _decoder(ll), _decoder(dl), 0
    for n in range(MAX_SYMS + 1):
        if n == MAX_SYMS:
            return "long", pos, o
        s = sym(ldec)
        if s is None or s > 285:
            return "bad", pos, o
        if s < 256:
            if o >= out_cap:
                return "bad", pos, o
            o += 1
            continue
        if s == 256:
            break
        L = LEN_BASE[s - 257] + get(LEN_EXTRA[s - 257])
        d = sym(ddec)
        if d is None or d > 29:
            return "bad", pos, o
        dist = DIST_BASE[d] + get(DIST_EXTRA[d])
        if dist > wsize or o + L > out_cap:
            return "bad", pos, o
        o += L
    return ("ok" if pos <= n_bits else "bad"), pos, o


def _stored_decoys(s, payload_and_at, decoys):
    """A stored block of decoy data; the decoys' stream bits are appended to ``decoys``."""
    payload, at = payload_and_at
    r = s.stored(payload)
    base = r.end - 8 * len(payload)
    decoys += [(base + b, kind) for b, kind in at]


def decoys():
    rng = np.random.default_rng(4)
    out = []
    # false candidates at every bit shift inside stored blocks, between true dynamic blocks
    s, dec = Stream(), []
    s.dynamic([0] + _rand(rng, 4095, 5))
    for part in range(3):
        _stored_decoys(s, decoy_payload(160, ["block", "bad", "block"], rng, unit=24, row=4096, shift0=part * 11), dec)
        s.dynamic(_row_tokens(rng, len(s.data), 4096))
    _fill(s, 4096)
    out.append(_design("decoys_every_shift", s, ["decoys_bad", "decoys_block", "decoy_shifts_0_31"], 4096, decoys=dec))
    # a false candidate that measures long (PD_LONG): the 'long' header, then more than 2^20 symbols of zero bits across
    # stored blocks whose LEN / NLEN (0x5555 / 0xAAAA) hold no two adjacent 1 bits (each 1 starts a '10', never the
    # end-of-block '11'); the image is larger than 2^20 bytes, else the decoy would measure bad (more bytes than the image)
    s = Stream()
    s.dynamic([0] + _rand(rng, 4095, 5))
    head = _pack(_decoy_bits("long", rng))
    r = s.stored(bytes(8) + head + bytes(0x5555 - 8 - len(head)))
    dec = [(r.end - 8 * 0x5555 + 64, "long")]
    for _ in range(50):
        s.stored(bytes(0x5555))
    s.dynamic([(258, 32768)] * 30 + _rand(rng, 50, 5))
    _fill(s, 4096)
    out.append(_design("decoy_long", s, ["decoy_long"], 4096, decoys=dec))
    # decoy densities just below and above the candidate capacity (stream_len / 512 + 1024)
    for name in ("cand_below", "cand_above"):
        unit = 24   # a candidate per unit: the capacity is reached at stream_len / 512 + 1024 = units
        units = int(1024 * 512 / (512 - unit) * (0.93 if name == "cand_below" else 1.12))
        s, dec = Stream(), []
        s.dynamic([0] + _rand(rng, 4095, 5))
        per = (4095 // unit) * 10
        for b0 in range(0, units, per):
            _stored_decoys(s, decoy_payload(min(per, units - b0), ["block", "bad"], rng, unit=unit, row=4096, shift0=b0), dec)
            s.dynamic(_row_tokens(rng, len(s.data), 4096))
        _fill(s, 4096)
        out.append(_design(f"decoys_{name}", s, [f"decoys_{name}"], 4096, expect="decode" if name == "cand_below" else "overflow",
                           decoys=dec))
    # quick-test passes just below and above the list capacity (stream_len / 8, at least 65,536): the two-byte pattern
    # b5 ed passes the first header test at 3 of its 16 bit positions (and the full test at none)
    for name, rows in (("list_below", 10), ("list_above", 12)):
        s = Stream()
        s.dynamic([0] + _rand(rng, 4095, 5))
        s.stored(b"".join(b"\0" + (b"\xb5\xed" * 2048)[:4095] for _ in range(rows)))
        s.dynamic(_row_tokens(rng, len(s.data), 4096))
        _fill(s, 4096)
        out.append(_design(f"decoys_{name}", s, [f"decoys_{name}"], 4096, expect="decode" if name == "list_below" else "overflow"))
    return out


# ---- declined on purpose: the present limits, pinned ---------------------------------------------------------------
def declines():
    rng = np.random.default_rng(5)
    out = []
    # one block of kMaxSyms symbols (end-of-block included: decodes) and of one more (declined)
    for extra, expect in ((0, "decode"), (1, "decline:max_syms")):
        s = Stream()
        s.stored(b"\0" + bytes(_rand(rng, 4095, 5)))
        lit = [0] * 257
        lit[0], lit[256] = 1, 1
        s.dynamic([0] * (MAX_SYMS - 1 + extra), litlens=lit, distlens=[0])
        _fill(s, 4096)
        out.append(_design(f"max_syms_{'plus1' if extra else 'exact'}", s, ["max_syms"], 4096, expect))
    # fixed-Huffman data just under and just over the host budget: the walk measures a first fixed block of 2^23 (+ 1)
    # bits, then refuses to measure the next one
    for over in (0, 1):
        s = Stream()
        bits = HOST_BUDGET + over
        j = (bits - 10) % 8
        k = (bits - 10 - 9 * j) // 8
        s.fixed([0] + [144] * j + [0] * (k - 1))
        assert s.recs[-1].end - s.recs[-1].start == bits
        s.fixed([1, 2, 3])
        s.stored(bytes((-len(s.data)) % 4096), final=True)
        out.append(_design(f"host_budget_{'over' if over else 'under'}", s, ["host_budget"], 4096,
                           "decline:host_budget" if over else "decode"))
    # more blocks than the chain may have (cap_blocks), and exactly as many
    for over in (0, 1):
        nb = 2000
        while True:
            s = Stream()
            s.fixed([0, 7])
            for _ in range(nb - 2):
                s.fixed([])
            s.fixed([], final=True)
            cap = cap_blocks(len(s.zlib()), len(s.data))
            if nb == cap + over:
                break
            nb = cap + over
        out.append(_design(f"blocks_{'over' if over else 'at'}_cap", s, ["cap_blocks"], None,
                           "decline:cap_blocks" if over else "decode"))
    # a distance beyond the window the zlib header declares (CINFO 0: 256 bytes)
    s = Stream(cmf=0x08)
    s.dynamic([0] + _rand(rng, 299) + [(10, 280)], final=True)
    out.append(_design("distance_beyond_cinfo_window", s, ["cinfo_window"], None, "decline:cinfo_window"))
    return out


# ---- invalid on purpose: inflate rejects them, so must the decoder ------------------------------------------------
def invalid():
    rng = np.random.default_rng(6)
    out = []
    # an over-subscribed distance tree (three codes of one bit) between valid blocks
    s = Stream()
    s.dynamic([0] + _rand(rng, 300))
    s.dynamic(_rand(rng, 40) + [(10, 1), (12, 2)], distlens=[1, 1, 1])
    s.dynamic(_rand(rng, 40), final=True)
    out.append(_design("invalid_oversubscribed_distances", s, ["oversubscribed_dist_tree"], None, "invalid"))
    # a stored block whose NLEN is not the complement of LEN
    s = Stream()
    s.dynamic([0] + _rand(rng, 300))
    s.stored(bytes(_rand(rng, 100)), nlen=0x1234)
    s.dynamic(_rand(rng, 40), final=True)
    out.append(_design("invalid_stored_nlen", s, ["stored_nlen"], None, "invalid"))
    return out


@lru_cache(maxsize=None)
def corpus():
    """Every design, by family."""
    return {"headers": headers(), "layout": layout(), "history": history(), "decoys": decoys(), "declines": declines(),
            "invalid": invalid()}


def all_designs():
    return [d for fam in corpus().values() for d in fam]


# ---- scale: an 8192 x 4096 panorama in a shape zlib only writes when told to flush after every row ------------------
def panorama_flushed_per_row(W=8192, H=4096, seed=8):
    """(BGR panorama, PNG file): RGB rows filtered Sub, one zlib partial flush per row - a dynamic block and an empty
    fixed block per row (libpng writers that flush every row produce this shape)."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W]
    base = np.stack([(x // 3 + y // 5) & 255, (x // 7 - y // 2) & 255, ((x + y) // 11) & 255], axis=2)
    img = (base + rng.integers(-4, 5, (H, W, 3))) & 255
    rgb = img.astype(np.uint8)
    d = rgb.astype(np.int16)
    sub = np.empty((H, 1 + 3 * W), np.uint8)
    sub[:, 0] = 1
    flat = d.reshape(H, 3 * W)
    f = flat.copy()
    f[:, 3:] = flat[:, 3:] - flat[:, :-3]
    sub[:, 1:] = (f & 255).astype(np.uint8)
    co = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY)
    parts = []
    for r in range(H):
        parts.append(co.compress(sub[r].tobytes()))
        parts.append(co.flush(zlib.Z_PARTIAL_FLUSH))
    parts.append(co.flush())
    z = b"".join(parts)
    png = M.SIG + M.chunk(b"IHDR", W.to_bytes(4, "big") + H.to_bytes(4, "big") + bytes([8, 2, 0, 0, 0]))
    for at in range(0, len(z), 1 << 20):
        png += M.chunk(b"IDAT", z[at:at + (1 << 20)])
    return np.ascontiguousarray(rgb[:, :, ::-1]), png + M.chunk(b"IEND", b"")
