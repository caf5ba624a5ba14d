"""PNG files of every colour type / bit depth / interlace method (the decoder's subset with P2P_OPT_PNG_FORMATS = 1), the
files that subset must still decline, and seeded damage of new-format files.  Shared by the CPU and the GPU tests."""
import struct
import zlib

import numpy as np

import png_formats_model as X
from oracle import png_decode_model as M

FORMATS = [(ct, d) for ct, ds in X.DEPTHS.items() for d in ds]   # every valid (colour type, bit depth)
SIZES = [(1, 1), (1, 9), (9, 1), (5, 5), (33, 17), (257, 129)]  # (W, H)
FILTERS = ["adaptive", [0], [1], [2], [3], [4], "rows"]
KINDS = ["noise", "smooth", "mixed"]


def samples(H: int, W: int, ct: int, depth: int, seed: int, kind: str, n_plte: int = 0) -> np.ndarray:
    """Sample values of an image ([H, W] or [H, W, C]): below 2^depth, palette indices below n_plte."""
    top = n_plte if ct == 3 else 1 << depth
    rng = np.random.default_rng(seed)
    ch = X.CHANNELS[ct]
    y, x = np.mgrid[0:H, 0:W]
    base = np.stack([(x * (3 + k) + y * (5 - k)) * top // (4 * max(W + H, 1)) + k * top // 5 for k in range(ch)], axis=2)
    if kind == "noise":
        img = rng.integers(0, top, (H, W, ch))
    elif kind == "smooth":
        img = base
    else:
        img = base + rng.integers(-2, 3, (H, W, ch)) * max(1, top // 64)
        img[:, 3 * W // 4:] = rng.integers(0, top, (H, W - 3 * W // 4, ch))
    img = np.mod(img, top).astype(np.uint16)
    return img[:, :, 0] if ch == 1 else img


def palette(n: int, seed: int) -> np.ndarray:
    return np.random.default_rng(seed).integers(0, 256, (n, 3), dtype=np.uint8)


def make(ct: int, depth: int, lace: int, W: int, H: int, k: int, extra=(), n_plte=None, trns=None, suggested=False, **kw) -> bytes:
    """File k of a (colour type, depth, interlace, size) cell: filter and content chosen by k."""
    filt = FILTERS[k % len(FILTERS)]
    if filt == "rows":
        filt = [int(v) for v in np.random.default_rng(k).integers(0, 5, 7)]
    kind = KINDS[k % len(KINDS)]
    pal = None
    if ct == 3:
        n_plte = n_plte or (1 << depth)
        pal = palette(n_plte, k)
    elif suggested:
        pal = palette(7, k)
    img = samples(H, W, ct, depth, 1000 + k, kind, n_plte or 0)
    return X.write_png(img, ct, filters=filt, depth=depth, interlace=lace, palette=pal, trns=trns, extra_chunks=extra, **kw)


def ancillary(ct: int, depth: int, n_plte: int) -> list:
    """gAMA, sBIT, bKGD and iCCP chunks valid for the format."""
    ch = X.CHANNELS[ct]
    sbit = bytes([min(depth, 8) if ct == 3 else depth] * (3 if ct == 3 else ch))
    bkgd = bytes([n_plte - 1]) if ct == 3 else struct.pack(">" + "H" * (1 if ct in (0, 4) else 3), *([(1 << depth) - 1] * (1 if ct in (0, 4) else 3)))
    iccp = b"icc\0\0" + zlib.compress(bytes(range(256)) * 2)
    return [(b"gAMA", struct.pack(">I", 45455)), (b"sBIT", sbit), (b"bKGD", bkgd), (b"iCCP", iccp)]


def matrix(sizes=SIZES) -> list:
    """[(id, file)]: every format x interlace x size, filters and content rotating; then the PLTE / tRNS / ancillary
    variants at 33 x 17."""
    out = []
    k = 0
    for ct, d in FORMATS:
        for lace in (0, 1):
            for W, H in sizes:
                out.append((f"ct{ct}_d{d}_i{lace}_{W}x{H}", make(ct, d, lace, W, H, k)))
                k += 1
            tag = f"ct{ct}_d{d}_i{lace}"
            lim = (1 << d) - 1
            if ct == 3:
                short = max(1, (1 << d) * 3 // 4)
                out.append((tag + "_short_plte", make(ct, d, lace, 33, 17, k, n_plte=short)))
                out.append((tag + "_trns", make(ct, d, lace, 33, 17, k + 1, n_plte=short, trns=bytes(range(max(1, short - 1))))))
            elif ct == 0:
                out.append((tag + "_trns", make(ct, d, lace, 33, 17, k, trns=struct.pack(">H", lim // 3))))
            elif ct == 2:
                out.append((tag + "_trns", make(ct, d, lace, 33, 17, k, trns=struct.pack(">HHH", lim, 0, lim // 2))))
                out.append((tag + "_suggested_plte", make(ct, d, lace, 33, 17, k, suggested=True)))
            elif ct == 6:
                out.append((tag + "_suggested_plte", make(ct, d, lace, 33, 17, k, suggested=True)))
            n = max(1, (1 << d) * 3 // 4) if ct == 3 else 0
            out.append((tag + "_ancillary", make(ct, d, lace, 33, 17, k + 2, extra=ancillary(ct, d, n or 1), n_plte=n or None)))
            k += 3
    return out


def _ihdr(W, H, depth, ct, lace=0):
    return M.chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, depth, ct, 0, 0, lace))


def _file(ihdr: bytes, chunks_before=(), raw: bytes = b"", chunks_after=()) -> bytes:
    out = M.SIG + ihdr + b"".join(M.chunk(t, b) for t, b in chunks_before) + M.chunk(b"IDAT", zlib.compress(raw))
    return out + b"".join(M.chunk(t, b) for t, b in chunks_after) + M.chunk(b"IEND", b"")


def declines() -> dict:
    """name -> a file the extended subset must decline (P2P_ERR_UNSUPPORTED)."""
    W, H = 12, 10
    plte = palette(4, 0).tobytes()
    rows_pal8 = b"".join(b"\0" + bytes([(x + y) % 4 for x in range(W)]) for y in range(H))
    rows_gray8 = b"".join(b"\0" + bytes(range(y, y + W)) for y in range(H))
    rgb = samples(H, W, 2, 8, 3, "mixed")
    ga = samples(H, W, 4, 8, 3, "mixed")
    cases = {
        "palette index out of range": _file(_ihdr(W, H, 8, 3), [(b"PLTE", plte)],
                                            b"".join(b"\0" + bytes([(x + y) % 6 for x in range(W)]) for y in range(H))),
        "type 3 without PLTE": _file(_ihdr(W, H, 8, 3), [], rows_pal8),
        "PLTE in a gray file": _file(_ihdr(W, H, 8, 0), [(b"PLTE", plte)], rows_gray8),
        "PLTE in a gray + alpha file": X.write_png(ga, 4, palette=palette(4, 1)),
        "PLTE after IDAT": _file(_ihdr(W, H, 8, 2), [], b"".join(b"\0" + r.tobytes() for r in rgb.astype(np.uint8)),
                                 [(b"PLTE", plte)]),
        "two PLTE chunks": _file(_ihdr(W, H, 8, 3), [(b"PLTE", plte), (b"PLTE", plte)], rows_pal8),
        "more than 2^depth entries": _file(_ihdr(W, H, 2, 3), [(b"PLTE", palette(5, 2).tobytes())],
                                           b"".join(b"\0" + bytes(3) for _ in range(H))),
        "PLTE length not a multiple of 3": _file(_ihdr(W, H, 8, 3), [(b"PLTE", plte + b"\0")], rows_pal8),
        "tRNS on gray + alpha": X.write_png(ga, 4, trns=bytes(2)),
        "tRNS on RGBA": X.write_png(samples(H, W, 6, 8, 4, "mixed"), 6, trns=bytes(6)),
        "tRNS before PLTE": _file(_ihdr(W, H, 8, 3), [(b"tRNS", b"\0"), (b"PLTE", plte)], rows_pal8),
        "tRNS longer than PLTE": _file(_ihdr(W, H, 8, 3), [(b"PLTE", plte), (b"tRNS", bytes(5))], rows_pal8),
        "gray tRNS of the wrong length": _file(_ihdr(W, H, 8, 0), [(b"tRNS", bytes(3))], rows_gray8),
        "gray tRNS beyond the bit depth": X.write_png(samples(H, W, 0, 4, 5, "noise"), 0, depth=4, trns=struct.pack(">H", 16)),
        "RGB tRNS of the wrong length": X.write_png(rgb, 2, trns=bytes(4)),
        "invalid depth for RGB": _file(_ihdr(W, H, 4, 2), [], b"".join(b"\0" + bytes((W * 12 + 7) // 8) for _ in range(H))),
        "invalid depth for palette": _file(_ihdr(W, H, 16, 3), [(b"PLTE", plte)], b"".join(b"\0" + bytes(2 * W) for _ in range(H))),
        "invalid depth for gray": _file(_ihdr(W, H, 3, 0), [], b"".join(b"\0" + bytes(5) for _ in range(H))),
        "colour type 5": _file(_ihdr(W, H, 8, 5), [], b"".join(b"\0" + bytes(W) for _ in range(H))),
        "interlace method 2": _file(_ihdr(W, H, 8, 2, 2), [], b"".join(b"\0" + bytes(3 * W) for _ in range(H))),
        "eXIf": X.write_png(rgb, 2, depth=8, interlace=1, extra_chunks=[(b"eXIf", b"MM\0*\0\0\0\x08\0\0")]),
        "APNG": X.write_png(rgb, 2, depth=8, interlace=1, extra_chunks=[(b"acTL", struct.pack(">II", 1, 0))]),
    }
    # the data of a non-interlaced file behind an Adam7 header, and the reverse (wrong amount of image data)
    img16 = samples(H, W, 2, 16, 6, "mixed")
    flat = X.write_png(img16, 2, depth=16)
    laced = X.write_png(img16, 2, depth=16, interlace=1)
    cases["Adam7 header, non-interlaced data"] = flat[:8] + _ihdr(W, H, 16, 2, 1) + flat[33:]
    cases["non-interlaced header, Adam7 data"] = laced[:8] + _ihdr(W, H, 16, 2, 0) + laced[33:]
    return cases


def damaged(n: int, seed: int) -> list:
    """n seeded bit flips / byte overwrites / truncations of new-format files, half of them inside the deflate data with the
    chunk CRC recomputed."""
    rng = np.random.default_rng(seed)
    bases = [make(0, 16, 1, 40, 30, 0, level=6), make(2, 16, 0, 40, 30, 1, level=9, idat=[500]), make(3, 4, 1, 40, 30, 2),
             make(3, 8, 0, 40, 30, 3, n_plte=200), make(0, 2, 0, 40, 30, 4, level=1), make(6, 16, 1, 40, 30, 5, idat=[300])]
    out = []
    for i in range(n):
        base = bases[i % len(bases)]
        if i % 2:
            ch = M.chunks(base)
            z = bytearray(b"".join(b for t, b, _, _ in ch if t == b"IDAT"))
            at = int(rng.integers(2, len(z)))
            if rng.integers(0, 4) == 0:
                del z[at:]
            else:
                z[at] ^= 1 << int(rng.integers(0, 8))
            rest = b"".join(M.chunk(t, b) for t, b, _, _ in ch[1:] if t not in (b"IDAT", b"IEND"))
            out.append(M.SIG + M.chunk(b"IHDR", ch[0][1]) + rest + M.chunk(b"IDAT", bytes(z)) + M.chunk(b"IEND", b""))
        else:
            d = bytearray(base)
            at = int(rng.integers(8, len(d)))
            if rng.integers(0, 4) == 0:
                del d[at:]
            else:
                d[at] ^= 1 << int(rng.integers(0, 8))
            out.append(bytes(d))
    return out
