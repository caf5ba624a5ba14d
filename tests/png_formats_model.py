"""CPU reference of the PNG decoder's wider subset (P2P_OPT_PNG_FORMATS = 1; TEST INFRASTRUCTURE ONLY - never imported by
the product package): every colour type and bit depth of the PNG specification (11.2.2) and Adam7 interlacing (8.2), built on
the chunk walk and the scanline filters of ``oracle/png_decode_model.py``.

* ``in_subset``: the chunk rules of ``parse_png`` with ``formats = 1`` (PLTE and tRNS where the specification puts them);
* ``decode``: zlib, the filters pass by pass, then what ``cv2.imread(path)`` (``IMREAD_COLOR``) makes of the samples - libpng's
  ``png_do_read_interlace``, ``png_do_unpack`` / ``png_do_expand`` (1/2/4-bit gray scaled), ``png_do_expand_palette``
  (palette alpha dropped) and ``png_do_strip_16`` (the high byte);
* ``write_png``: files of any of these formats (sub-byte packing, 16-bit big-endian samples, Adam7 passes, PLTE / tRNS).

Pinned against ``cv2.imdecode`` itself in ``tests/test_png_decode_formats_oracle.py``.
"""
from __future__ import annotations

import struct
import zlib

import numpy as np

from oracle import png_decode_model as M

CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
DEPTHS = {0: (1, 2, 4, 8, 16), 2: (8, 16), 3: (1, 2, 4, 8), 4: (8, 16), 6: (8, 16)}   # PNG specification 11.2.2
ADAM7 = [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)]  # x0, y0, dx, dy


def in_subset(data: bytes):
    """(W, H, colour type) if the device decoder accepts the file's structure with formats = 1, else None."""
    try:
        ch = M.chunks(data)
    except ValueError:
        return None
    if not ch or ch[0][0] != b"IHDR" or len(ch[0][1]) != 13 or ch[-1][0] != b"IEND":
        return None
    if not all(ok for _, _, _, ok in ch):
        return None
    W, H, depth, ctype, comp, filt, lace = struct.unpack(">IIBBBBB", ch[0][1])
    if depth not in DEPTHS.get(ctype, ()) or comp or filt or lace > 1 or not (0 < W < 32767 and 0 < H < 32767):
        return None
    names = [c[0] for c in ch]
    if b"IDAT" not in names:
        return None
    first = names.index(b"IDAT")
    last = len(names) - 1 - names[::-1].index(b"IDAT")
    if any(n != b"IDAT" for n in names[first:last + 1]):
        return None
    n_plte = 0
    for k, (n, body, _, _) in enumerate(ch[1:-1], 1):
        if n == b"IDAT":
            continue
        if n == b"PLTE":
            if ctype in (0, 4) or n_plte or k > first or not body or len(body) % 3 or len(body) > 768:
                return None
            if ctype == 3 and len(body) // 3 > (1 << depth):
                return None
            n_plte = len(body) // 3
            continue
        if n == b"tRNS":
            if names[1:k].count(b"tRNS") or k > first:
                return None
            lim = (1 << depth) - 1
            vals = struct.unpack(f">{len(body) // 2}H", body[:len(body) // 2 * 2])
            if ctype == 0 and (len(body) != 2 or vals[0] > lim):
                return None
            if ctype == 2 and (len(body) != 6 or max(vals) > lim):
                return None
            if ctype == 3 and not (n_plte and 0 < len(body) <= n_plte):
                return None
            if ctype in (4, 6):
                return None
            continue
        if n in (b"acTL", b"fcTL", b"fdAT", b"eXIf", b"IHDR") or not (n[0] & 0x20) or not n.isalpha():
            return None
    if ctype == 3 and not n_plte:
        return None
    return W, H, ctype


def passes(W: int, H: int, lace: int):
    """[(x0, y0, dx, dy, w, h)] of the non-empty passes (the whole image when not interlaced)."""
    out = []
    for x0, y0, dx, dy in (ADAM7 if lace else [(0, 0, 1, 1)]):
        w, h = max(0, (W - x0 + dx - 1) // dx), max(0, (H - y0 + dy - 1) // dy)
        if w and h:
            out.append((x0, y0, dx, dy, w, h))
    return out


def unpack(rows: np.ndarray, w: int, depth: int, channels: int) -> np.ndarray:
    """Samples [h, w, channels] (u16 values) of reconstructed rows [h, row_bytes]: sub-byte samples MSB first, 16-bit big-endian."""
    h = rows.shape[0]
    if depth == 16:
        return (rows[:, :w * channels * 2].reshape(h, w * channels, 2).astype(np.uint16) @ np.array([256, 1], np.uint16)).reshape(h, w, channels)
    if depth == 8:
        return rows[:, :w * channels].reshape(h, w, channels).astype(np.uint16)
    bits = np.unpackbits(rows, axis=1)[:, :w * depth].reshape(h, w, depth)
    return (bits.astype(np.uint16) @ (1 << np.arange(depth - 1, -1, -1)).astype(np.uint16)).reshape(h, w, 1)


def decode(data: bytes) -> np.ndarray:
    """BGR u8 [H, W, 3] of a file inside the wider subset (ValueError otherwise, also for a palette index without a PLTE
    entry; zlib.error for a damaged stream)."""
    sub = in_subset(data)
    if sub is None:
        raise ValueError("outside the subset")
    W, H, ctype = sub
    ch = M.chunks(data)
    raw = np.frombuffer(zlib.decompress(b"".join(body for typ, body, _, _ in ch if typ == b"IDAT")), np.uint8)
    depth, lace = ch[0][1][8], ch[0][1][12]
    nch = CHANNELS[ctype]
    bits = depth * nch
    bpp = max(1, bits // 8)
    samples = np.zeros((H, W, nch), np.uint16)
    at = 0
    for x0, y0, dx, dy, w, h in passes(W, H, lace):
        rb = (w * bits + 7) // 8
        part = raw[at:at + h * (1 + rb)]
        if part.size != h * (1 + rb):
            raise ValueError("wrong amount of image data")
        samples[y0::dy, x0::dx] = unpack(M.unfilter(part, h, rb, bpp), w, depth, nch)
        at += h * (1 + rb)
    if at != raw.size:
        raise ValueError("wrong amount of image data")
    if ctype == 3:
        plte = np.frombuffer(next(b for t, b, _, _ in ch if t == b"PLTE"), np.uint8).reshape(-1, 3)
        idx = samples[:, :, 0]
        if idx.max() >= len(plte):
            raise ValueError("palette index without a PLTE entry")
        return plte[idx][:, :, ::-1].copy()
    v = (samples >> 8).astype(np.uint8) if depth == 16 else (samples * (255 // ((1 << depth) - 1))).astype(np.uint8)
    if ctype in (0, 4):
        return np.repeat(v[:, :, :1], 3, axis=2)
    return v[:, :, 2::-1].copy()


def pack_rows(samples: np.ndarray, depth: int) -> np.ndarray:
    """Bytes [h, row_bytes] of samples [h, n] (values < 2^depth): big-endian 16-bit, sub-byte samples MSB first."""
    h, n = samples.shape
    if depth == 16:
        return samples.astype(">u2").view(np.uint8).reshape(h, 2 * n)
    if depth == 8:
        return samples.astype(np.uint8)
    bits = (samples[:, :, None].astype(np.uint16) >> np.arange(depth - 1, -1, -1)) & 1
    return np.packbits(bits.reshape(h, n * depth).astype(np.uint8), axis=1)


def write_png(img: np.ndarray, ctype: int = 2, filters="adaptive", level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY,
              wbits: int = 15, idat: int | list = 8192, extra_chunks=(), depth: int = 8, interlace: int = 0, palette=None,
              trns=None) -> bytes:
    """A PNG file of img (sample values: [H, W] for gray / palette indices, [H, W, C] in PNG channel order otherwise).
    filters: 'adaptive' (libpng's heuristic, ``oracle/png_decode_model.py`` filter_rows) or a list of row filters used
    cyclically in every pass; interlace: 1 = Adam7; palette: [n, 3] RGB (a PLTE chunk); trns: bytes of a tRNS chunk."""
    H, W = img.shape[:2]
    nch = CHANNELS[ctype]
    bpp = max(1, depth * nch // 8)
    im = np.asarray(img).reshape(H, W, nch)
    raw = b""
    for x0, y0, dx, dy, w, h in passes(W, H, interlace):
        sub = im[y0::dy, x0::dx].reshape(h, w * nch)
        f = filters if isinstance(filters, str) else [filters[i % len(filters)] for i in range(h)]
        raw += M.filter_rows(pack_rows(sub, depth), bpp, f)
    co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
    z = co.compress(raw) + co.flush()
    out = M.SIG + M.chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, depth, ctype, 0, 0, interlace))
    if palette is not None:
        out += M.chunk(b"PLTE", np.asarray(palette, np.uint8).tobytes())
    if trns is not None:
        out += M.chunk(b"tRNS", bytes(trns))
    for typ, body in extra_chunks:
        out += M.chunk(typ, body)
    sizes = idat if isinstance(idat, list) else [idat]
    at, k = 0, 0
    while at < len(z):
        out += M.chunk(b"IDAT", z[at:at + sizes[k % len(sizes)]])
        at += sizes[k % len(sizes)]
        k += 1
    return out + M.chunk(b"IEND", b"")
