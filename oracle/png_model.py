"""Step-by-step model of the PNG encoder behind ``cv2.imwrite(path.png, bgr)`` (ref ``app/panorama_to_plane-pitch.py:277``, the
default ``--output_format png``, ref :400-405).  TEST INFRASTRUCTURE (see ``oracle/__init__.py``).

The arithmetic lives in libpng + zlib (linked by ``opencv-python``; not under ``/root/reference``).  OpenCV's defaults are:
filter Sub on every row (``png_set_filter(PNG_FILTER_SUB)``), zlib level 1 (``Z_BEST_SPEED``), strategy ``Z_RLE``, memLevel 8,
32 KiB window, IDAT chunks of 8192 bytes.  Restated here from the published sources:

* ``deflate.c``  deflate_rle: greedy run-length matches at distance 1 (3..258 bytes), blocks of 16383 symbols
* ``trees.c``    build_tree / gen_bitlen / gen_codes (heap order and depth tie-breaks included), scan_tree / send_tree,
                 build_bl_tree, the stored / static / dynamic decision, compress_block, LSB-first bit packing
* ``pngwrite.c`` signature, IHDR, IDAT chunking (8192-byte zbuffer), IEND; CRC-32 per chunk, Adler-32 trailer

``deflate_rle`` is pinned against ``zlib.compressobj(1, DEFLATED, 15, 8, Z_RLE)`` and ``encode_png`` against ``cv2.imencode('.png')``
in ``tests/test_png_oracle.py``."""
import zlib, numpy as np

MAX_BITS, BL_CODES, D_CODES, LITERALS, LENGTH_CODES = 15, 19, 30, 256, 29
L_CODES = LITERALS + 1 + LENGTH_CODES
HEAP_SIZE = 2 * L_CODES + 1
END_BLOCK, REP_3_6, REPZ_3_10, REPZ_11_138 = 256, 16, 17, 18
extra_lbits = [0,0,0,0,0,0,0,0,1,1,1,1,2,2,2,2,3,3,3,3,4,4,4,4,5,5,5,5,0]
extra_dbits = [0,0,0,0,1,1,2,2,3,3,4,4,5,5,6,6,7,7,8,8,9,9,10,10,11,11,12,12,13,13]
extra_blbits = [0]*16 + [2,3,7]
bl_order = [16,17,18,0,8,7,9,6,10,5,11,4,12,3,13,2,14,1,15]
base_length = [0]*LENGTH_CODES
length_code = [0]*256
def _init():
    length = 0
    for code in range(LENGTH_CODES-1):
        base_length[code] = length
        for n in range(1 << extra_lbits[code]):
            length_code[length] = code; length += 1
    length_code[length-1] = LENGTH_CODES-1   # length 258 -> code 28
    base_length[LENGTH_CODES-1] = 255  # unused extra (0 bits)
_init()
static_l_len = [8]*144 + [9]*112 + [7]*24 + [8]*8
static_d_len = [5]*30

def bi_reverse(code, length):
    r = 0
    for _ in range(length):
        r = (r << 1) | (code & 1); code >>= 1
    return r

class BitOut:
    def __init__(self): self.buf = bytearray(); self.acc = 0; self.n = 0
    def send(self, value, length):
        self.acc |= (value & ((1 << length) - 1)) << self.n; self.n += length
        while self.n >= 8:
            self.buf.append(self.acc & 0xFF); self.acc >>= 8; self.n -= 8
    def tell(self): return 8 * len(self.buf) + self.n
    def windup(self):
        if self.n: self.buf.append(self.acc & 0xFF)
        self.acc = 0; self.n = 0

def build_tree(freq, elems, stree_len, extra, base, max_length, st):
    """returns (lens, codes, max_code); st = dict with opt_len/static_len updated, st['overflow'] = gen_bitlen's count of
    nodes deeper than max_length (0: the tree needed no repair)"""
    Freq = list(freq) + [0]*(HEAP_SIZE)   # room for internal nodes
    Len = [0]*(len(Freq)); Dad = [0]*len(Freq); depth = [0]*len(Freq)
    heap = [0]*(HEAP_SIZE+1); heap_len = 0; heap_max = HEAP_SIZE; max_code = -1
    for n in range(elems):
        if Freq[n] != 0:
            heap_len += 1; heap[heap_len] = max_code = n; depth[n] = 0
        else: Len[n] = 0
    while heap_len < 2:
        if max_code < 2: max_code += 1; node = max_code
        else: node = 0
        heap_len += 1; heap[heap_len] = node
        Freq[node] = 1; depth[node] = 0; st['opt_len'] -= 1
        if stree_len is not None: st['static_len'] -= stree_len[node]
    def smaller(n, m): return Freq[n] < Freq[m] or (Freq[n] == Freq[m] and depth[n] <= depth[m])
    def pqdownheap(k):
        nonlocal heap_len
        v = heap[k]; j = k << 1
        while j <= heap_len:
            if j < heap_len and smaller(heap[j+1], heap[j]): j += 1
            if smaller(v, heap[j]): break
            heap[k] = heap[j]; k = j; j <<= 1
        heap[k] = v
    for n in range(heap_len // 2, 0, -1): pqdownheap(n)
    node = elems
    while True:
        n = heap[1]; heap[1] = heap[heap_len]; heap_len -= 1; pqdownheap(1)
        m = heap[1]
        heap_max -= 1; heap[heap_max] = n
        heap_max -= 1; heap[heap_max] = m
        Freq[node] = Freq[n] + Freq[m]
        depth[node] = max(depth[n], depth[m]) + 1
        Dad[n] = Dad[m] = node
        heap[1] = node; node += 1
        pqdownheap(1)
        if heap_len < 2: break
    heap_max -= 1; heap[heap_max] = heap[1]
    # gen_bitlen
    bl_count = [0]*(MAX_BITS+1); overflow = 0
    Len[heap[heap_max]] = 0
    h = heap_max + 1
    while h < HEAP_SIZE:
        n = heap[h]; bits = Len[Dad[n]] + 1
        if bits > max_length: bits = max_length; overflow += 1
        Len[n] = bits
        if n <= max_code:
            bl_count[bits] += 1
            xbits = extra[n-base] if n >= base else 0
            f = Freq[n]; st['opt_len'] += f * (bits + xbits)
            if stree_len is not None: st['static_len'] += f * (stree_len[n] + xbits)
        h += 1
    st['overflow'] = overflow
    if overflow > 0:
        while True:
            bits = max_length - 1
            while bl_count[bits] == 0: bits -= 1
            bl_count[bits] -= 1; bl_count[bits+1] += 2; bl_count[max_length] -= 1
            overflow -= 2
            if overflow <= 0: break
        h = HEAP_SIZE
        for bits in range(max_length, 0, -1):
            n = bl_count[bits]
            while n != 0:
                h -= 1; m = heap[h]
                if m > max_code: continue
                if Len[m] != bits:
                    st['opt_len'] += (bits - Len[m]) * Freq[m]; Len[m] = bits
                n -= 1
    # gen_codes
    next_code = [0]*(MAX_BITS+1); code = 0
    for bits in range(1, MAX_BITS+1):
        code = (code + bl_count[bits-1]) << 1; next_code[bits] = code
    codes = [0]*elems
    for n in range(max_code+1):
        l = Len[n]
        if l: codes[n] = bi_reverse(next_code[l], l); next_code[l] += 1
    return Len[:elems], codes, max_code

def scan_tree(lens, max_code, blfreq):
    prevlen = -1; nextlen = lens[0]; count = 0
    max_count, min_count = (138, 3) if nextlen == 0 else (7, 4)
    ext = list(lens[:max_code+1]) + [0xffff]
    for n in range(max_code+1):
        curlen = nextlen; nextlen = ext[n+1]
        count += 1
        if count < max_count and curlen == nextlen: continue
        elif count < min_count: blfreq[curlen] += count
        elif curlen != 0:
            if curlen != prevlen: blfreq[curlen] += 1
            blfreq[REP_3_6] += 1
        elif count <= 10: blfreq[REPZ_3_10] += 1
        else: blfreq[REPZ_11_138] += 1
        count = 0; prevlen = curlen
        if nextlen == 0: max_count, min_count = 138, 3
        elif curlen == nextlen: max_count, min_count = 6, 3
        else: max_count, min_count = 7, 4

def send_tree(out, lens, max_code, bllen, blcode):
    prevlen = -1; nextlen = lens[0]; count = 0
    max_count, min_count = (138, 3) if nextlen == 0 else (7, 4)
    ext = list(lens[:max_code+1]) + [0xffff]
    for n in range(max_code+1):
        curlen = nextlen; nextlen = ext[n+1]
        count += 1
        if count < max_count and curlen == nextlen: continue
        elif count < min_count:
            for _ in range(count): out.send(blcode[curlen], bllen[curlen])
        elif curlen != 0:
            if curlen != prevlen:
                out.send(blcode[curlen], bllen[curlen]); count -= 1
            out.send(blcode[REP_3_6], bllen[REP_3_6]); out.send(count-3, 2)
        elif count <= 10:
            out.send(blcode[REPZ_3_10], bllen[REPZ_3_10]); out.send(count-3, 3)
        else:
            out.send(blcode[REPZ_11_138], bllen[REPZ_11_138]); out.send(count-11, 7)
        count = 0; prevlen = curlen
        if nextlen == 0: max_count, min_count = 138, 3
        elif curlen == nextlen: max_count, min_count = 6, 3
        else: max_count, min_count = 7, 4

def tokenize_rle(data):
    """deflate_rle: list of tokens: ('L', byte) or ('M', length)"""
    n = len(data); toks = []; i = 0
    while i < n:
        ml = 0
        if n - i >= 3 and i > 0:
            prev = data[i-1]
            if data[i] == prev and data[i+1] == prev and data[i+2] == prev:
                j = i + 3; lim = min(n, i + 258)
                while j < lim and data[j] == prev: j += 1
                ml = j - i
        if ml >= 3: toks.append(('M', ml)); i += ml
        else: toks.append(('L', data[i])); i += 1
    return toks

def flush_block(out, toks, stored_bytes, last, buf_available=True, rec=None):
    """_tr_flush_block; returns the block kind.  ``rec`` (a dict) receives the block's record, see ``deflate_rle``."""
    start = out.tell()
    lfreq = [0]*L_CODES; dfreq = [0]*D_CODES
    lfreq[END_BLOCK] = 1
    for t, v in toks:
        if t == 'L': lfreq[v] += 1
        else:
            lfreq[length_code[v-3] + LITERALS + 1] += 1; dfreq[0] += 1
    st = {'opt_len': 0, 'static_len': 0}
    llen, lcode, lmax = build_tree(lfreq, L_CODES, static_l_len, extra_lbits, LITERALS+1, MAX_BITS, st)
    l_overflow = st['overflow']
    dlen, dcode, dmax = build_tree(dfreq, D_CODES, static_d_len, extra_dbits, 0, MAX_BITS, st)
    blfreq = [0]*BL_CODES
    scan_tree(llen, lmax, blfreq); scan_tree(dlen, dmax, blfreq)
    bllen, blcode, _ = build_tree(blfreq, BL_CODES, None, extra_blbits, 0, 7, st)
    if rec is not None:
        rec.update(tokens=len(toks), bytes=len(stored_bytes), start_bit=start, l_overflow=l_overflow,
                   bl_overflow=st['overflow'], hdr_bits=0, last=last,
                   lengths=sorted({v for t, v in toks if t == 'M'}), lmax=lmax)
    max_blindex = BL_CODES - 1
    while max_blindex >= 3 and bllen[bl_order[max_blindex]] == 0: max_blindex -= 1
    st['opt_len'] += 3*(max_blindex+1) + 5 + 5 + 4
    opt_lenb = (st['opt_len'] + 3 + 7) >> 3; static_lenb = (st['static_len'] + 3 + 7) >> 3
    if static_lenb <= opt_lenb: opt_lenb = static_lenb
    if len(stored_bytes) + 4 <= opt_lenb and buf_available:
        out.send((0 << 1) + last, 3); out.windup()
        L = len(stored_bytes); out.buf += bytes([L & 0xFF, L >> 8, (~L) & 0xFF, ((~L) >> 8) & 0xFF]); out.buf += stored_bytes
        if rec is not None: rec['kind'] = 'stored'
        return 'stored'
    if static_lenb == opt_lenb:
        out.send((1 << 1) + last, 3)
        ll, lc, dl, dc = static_l_len, None, static_d_len, None
        # static codes
        blc = [0]*(MAX_BITS+1)
        for l in static_l_len: blc[l] += 1
        nc = [0]*(MAX_BITS+1); code = 0
        for bits in range(1, MAX_BITS+1): code = (code + blc[bits-1]) << 1; nc[bits] = code
        lc = [0]*288
        for n in range(288): lc[n] = bi_reverse(nc[static_l_len[n]], static_l_len[n]); nc[static_l_len[n]] += 1
        dc = [bi_reverse(n, 5) for n in range(30)]
        kind = 'static'
    else:
        out.send((2 << 1) + last, 3)
        out.send(lmax + 1 - 257, 5); out.send(dmax + 1 - 1, 5); out.send(max_blindex + 1 - 4, 4)
        for rank in range(max_blindex + 1): out.send(bllen[bl_order[rank]], 3)
        send_tree(out, llen, lmax, bllen, blcode); send_tree(out, dlen, dmax, bllen, blcode)
        ll, lc, dl, dc = llen, lcode, dlen, dcode
        kind = 'dynamic'
        if rec is not None: rec['hdr_bits'] = out.tell() - start
    for t, v in toks:
        if t == 'L': out.send(lc[v], ll[v])
        else:
            code = length_code[v-3]
            out.send(lc[code + LITERALS + 1], ll[code + LITERALS + 1])
            if extra_lbits[code]: out.send(v - 3 - base_length[code], extra_lbits[code])
            out.send(dc[0], dl[0])
    out.send(lc[END_BLOCK], ll[END_BLOCK])
    if rec is not None: rec['kind'] = kind
    return kind

def deflate_rle(data, lit_bufsize=16384, stats=None):
    """(zlib stream, block kinds).  ``stats``, if a list, receives one dict per deflate block: ``kind`` ('stored', 'static'
    or 'dynamic'), ``tokens`` and ``bytes`` (symbols and input bytes of the block, END_BLOCK not counted), ``l_overflow``
    and ``bl_overflow`` (gen_bitlen's overflow count of the literal / length and of the bit-length tree: > 0 when the tree
    was deeper than 15 / 7 bits and got repaired), ``hdr_bits`` (3 block-type bits + tree description of a dynamic block,
    else 0), ``start_bit`` (bit offset of the block in the stream, the 16 bits of CMF / FLG included), ``last``, ``lmax``
    (the largest literal / length symbol used) and ``lengths`` (the match lengths it holds)."""
    out = BitOut(); out.buf += b'\x78\x01'
    toks = tokenize_rle(data)
    sym_end = lit_bufsize - 1
    pos = 0; i = 0; kinds = []
    nblocks = 0
    while True:
        blk = toks[i:i+sym_end]
        nbytes = sum(1 if t == 'L' else v for t, v in blk)
        full = len(blk) == sym_end
        i += len(blk)
        rec = {} if stats is not None else None
        kinds.append(flush_block(out, blk, data[pos:pos+nbytes], 0 if full else 1, rec=rec)); pos += nbytes
        if rec is not None: stats.append(rec)
        if full: continue
        out.windup(); break
    a = zlib.adler32(data)
    out.buf += a.to_bytes(4, 'big')
    return bytes(out.buf), kinds

def sub_filter(bgr: np.ndarray) -> bytes:
    """PNG rows of an 8-bit BGR image as OpenCV writes them: RGB order (png_set_bgr), filter type 1 (Sub) on every row -
    type 0 (None) for images one pixel wide, where libpng drops the Sub filter (pngwrite.c png_set_filter /
    png_write_start_row: ``width == 1`` clears SUB, AVG and PAETH; the bytes are the same, only the type differs)."""
    H, W, _ = bgr.shape
    rgb = bgr[..., ::-1].astype(np.int16)
    f = rgb.copy()
    f[:, 1:] -= rgb[:, :-1]
    ftype = np.full((H, 1), 0 if W == 1 else 1, np.uint8)
    rows = np.concatenate([ftype, (f & 255).astype(np.uint8).reshape(H, 3 * W)], axis=1)
    return rows.tobytes()


def zlib_header(data_size: int) -> bytes:
    """CMF / FLG of the stream: 78 01 (32 KB window, level flags 0), with the window bits libpng writes for small
    images (pngwutil.c optimize_cmf: for at most 16384 bytes of data, the smallest window that still holds them)."""
    cinfo = 7
    half = 1 << (cinfo + 7)
    if data_size <= 16384 and data_size <= half:
        while True:
            half >>= 1
            cinfo -= 1
            if not (cinfo > 0 and data_size <= half):
                break
    cmf = 0x08 | (cinfo << 4)
    flg = 0x1F - ((cmf << 8) % 0x1F)
    return bytes([cmf, flg])


def encode_png(bgr: np.ndarray) -> bytes:
    """The bytes ``cv2.imencode('.png', bgr)`` produces (default parameters)."""
    import struct

    H, W, _ = bgr.shape
    raw = sub_filter(bgr)
    z, _ = deflate_rle(raw)
    z = zlib_header(len(raw)) + z[2:]

    def chunk(typ, data):
        return struct.pack(">I", len(data)) + typ + data + struct.pack(">I", zlib.crc32(typ + data) & 0xFFFFFFFF)

    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 0))
    for i in range(0, len(z), 8192):
        out += chunk(b"IDAT", z[i:i + 8192])
    return out + chunk(b"IEND", b"")


if __name__ == "__main__":
    import sys; sys.path.insert(0, '/root/repo')
    from tools import synth_inputs as synth
    rng = np.random.default_rng(0)
    def sub_filter(img):
        H, W, _ = img.shape
        rgb = img[..., ::-1].astype(np.int16)
        f = rgb.copy(); f[:, 1:] -= rgb[:, :-1]
        rows = np.concatenate([np.ones((H, 1), np.uint8), (f & 255).astype(np.uint8).reshape(H, 3*W)], axis=1)
        return rows.tobytes()
    cases = {"smooth": synth.smooth(300, 200, 1), "flat": np.full((120, 200, 3), 77, np.uint8),
             "textured": np.clip(synth.smooth(320, 160, 2).astype(int) + rng.integers(-6, 7, (160, 320, 3)), 0, 255).astype(np.uint8),
             "stripes": np.repeat(rng.integers(0, 256, (90, 30, 3), dtype=np.uint8), 10, axis=1),
             "tiny": rng.integers(0, 256, (3, 5, 3), dtype=np.uint8)}
    for name, img in cases.items():
        raw = sub_filter(img)
        co = zlib.compressobj(1, zlib.DEFLATED, 15, 8, zlib.Z_RLE)
        ref = co.compress(raw) + co.flush()
        got, kinds = deflate_rle(raw)
        print(name, len(raw), len(ref), len(got), got == ref, {k: kinds.count(k) for k in set(kinds)})
        if got != ref:
            d = next(i for i in range(min(len(got), len(ref))) if got[i] != ref[i]); print("  first diff at byte", d)
