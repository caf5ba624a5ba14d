"""Random VALID PNG files against the library's host model of the device decoder (the kernels' own __host__ __device__
routines, run serially - no GPU needed): random sizes, colour types, filter choices, zlib levels / strategies / window
sizes / memory levels, IDAT splits and flushes; every file must decode to the pixels cv2.imdecode returns.

    python tools/fuzz_png_files.py [n_files] > profiles/r2_fuzz_png_files.jsonl
    python tools/fuzz_png_files.py --formats extended [n_files] > profiles/r3_fuzz_png_files_ext.jsonl

--formats extended: the decoder's wider subset (P2P_OPT_PNG_FORMATS = 1): every colour type / bit depth, Adam7 or not,
palettes of random length with or without tRNS, gray / RGB tRNS keys.
"""
import ctypes as C
import json
import struct
import sys
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402
from oracle import png_decode_model as M  # noqa: E402


def extended_file(rng, i):
    """A random valid file of the wider subset: format, interlace, size, palette / tRNS, content, filters and zlib settings."""
    sys.path.insert(0, str(ROOT / "tests"))
    import png_formats_model as X
    from png_formats import FORMATS, KINDS, palette, samples

    ct, depth = FORMATS[int(rng.integers(0, len(FORMATS)))]
    lace = int(rng.integers(0, 2))
    H, W = int(rng.integers(1, 120)), int(rng.integers(1, 200))
    n_plte = int(rng.integers(1, (1 << depth) + 1)) if ct == 3 else 0
    img = samples(H, W, ct, depth, int(rng.integers(0, 1 << 30)), KINDS[int(rng.integers(0, 3))], n_plte)
    lim = (1 << depth) - 1
    trns = None
    if rng.integers(0, 3) == 0:
        if ct == 3:
            trns = bytes(rng.integers(0, 256, int(rng.integers(1, n_plte + 1)), dtype=np.uint8))
        elif ct == 0:
            trns = struct.pack(">H", int(rng.integers(0, lim + 1)))
        elif ct == 2:
            trns = struct.pack(">HHH", *[int(v) for v in rng.integers(0, lim + 1, 3)])
    pal = palette(n_plte, i) if ct == 3 else (palette(int(rng.integers(1, 257)), i) if ct in (2, 6) and rng.integers(0, 4) == 0 else None)
    fsel = int(rng.integers(0, 3))
    filters = "adaptive" if fsel == 0 else ([int(rng.integers(0, 5))] if fsel == 1 else [int(v) for v in rng.integers(0, 5, 11)])
    kw = dict(filters=filters, level=int(rng.integers(0, 10)),
              strategy=[zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED][int(rng.integers(0, 5))],
              wbits=int(rng.integers(9, 16)), idat=[int(v) for v in rng.integers(1, 3000, int(rng.integers(1, 4)))])
    data = X.write_png(img, ct, depth=depth, interlace=lace, palette=pal, trns=trns, **kw)
    return data, dict(ct=ct, depth=depth, interlace=lace, W=W, H=H, n_plte=n_plte, trns=trns is not None)


def main():
    import cv2

    args = sys.argv[1:]
    formats = 0
    if "--formats" in args:
        k = args.index("--formats")
        formats = {"default": 0, "extended": 1}[args[k + 1]]
        del args[k:k + 2]
    n_files = int(args[0]) if args else 1500
    g.build()
    lib = g.load_package()._lib.load()
    rng = np.random.default_rng(4242 + formats)
    stats = {"files": 0, "identical": 0, "declined": 0, "different": 0, "blocks": 0, "blocks_found_by_search": 0, "bytes": 0}
    t0 = time.time()
    for i in range(n_files):
        if formats:
            data, kw = extended_file(rng, i)
            ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
            w, h = C.c_int(), C.c_int()
            stats["files"] += 1
            stats["bytes"] += len(data)
            if ref is None or lib.p2p_png_probe_ex(data, len(data), 1, C.byref(w), C.byref(h)):
                stats["declined"] += 1
                print(json.dumps({"declined_valid_file": i, "kw": kw, "cv2_none": ref is None}), flush=True)
                continue
            out = np.zeros((h.value, w.value, 3), np.uint8)
            st = (C.c_uint64 * 4)()
            rc = lib.p2p_png_decode_host_ex(data, len(data), 1, out.ctypes.data, out.strides[0], h.value, st)
            if rc:
                stats["declined"] += 1
                print(json.dumps({"declined_valid_file": i, "kw": kw}), flush=True)
            elif np.array_equal(out, ref):
                stats["identical"] += 1
                stats["blocks"] += st[2]
                stats["blocks_found_by_search"] += st[2] - st[3]
            else:
                stats["different"] += 1
                print(json.dumps({"different": i, "kw": kw}), flush=True)
            continue
        ctype, ch = [(0, 1), (2, 3), (4, 2), (6, 4)][int(rng.integers(0, 4))]
        H, W = int(rng.integers(1, 160)), int(rng.integers(1, 260))
        kind = ["mixed", "smooth", "noise"][int(rng.integers(0, 3))]
        img = M.test_image(H, W, ch, int(rng.integers(0, 1 << 30)), kind)
        fsel = int(rng.integers(0, 4))
        filters = "adaptive" if fsel == 0 else ([int(rng.integers(0, 5))] * H if fsel == 1 else list(rng.integers(0, 5, H)))
        kw = dict(
            filters=filters, level=int(rng.integers(0, 10)),
            strategy=[zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED][int(rng.integers(0, 5))],
            wbits=int(rng.integers(9, 16)), mem_level=int(rng.integers(1, 10)),
            idat=[int(v) for v in rng.integers(1, 5000, int(rng.integers(1, 4)))],
            flush_every=int(rng.integers(50, 20000)) if rng.integers(0, 3) == 0 else 0,
            flush_mode=[zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH][int(rng.integers(0, 2))],
        )
        data = M.write_png(img, ctype, **kw)
        ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
        w, h = C.c_int(), C.c_int()
        stats["files"] += 1
        stats["bytes"] += len(data)
        if ref is None or lib.p2p_png_probe(data, len(data), C.byref(w), C.byref(h)):
            stats["declined"] += 1
            continue
        out = np.zeros((h.value, w.value, 3), np.uint8)
        st = (C.c_uint64 * 4)()
        rc = lib.p2p_png_decode_host(data, len(data), out.ctypes.data, out.strides[0], h.value, st)
        if rc:
            stats["declined"] += 1
            print(json.dumps({"declined_valid_file": i, "kw": {k: (v if not isinstance(v, list) else "list") for k, v in kw.items()}}), flush=True)
        elif np.array_equal(out, ref):
            stats["identical"] += 1
            stats["blocks"] += st[2]
            stats["blocks_found_by_search"] += st[2] - st[3]
        else:
            stats["different"] += 1
            print(json.dumps({"different": i}), flush=True)
    stats["seconds"] = round(time.time() - t0, 1)
    stats["what"] = ("random valid PNG files of every colour type / bit depth, Adam7 or not, random palettes with or without tRNS, "
                     "gray / RGB tRNS keys, suggested palettes, sizes 1..199 x 1..119, filters per file / cycled / adaptive, zlib "
                     "levels 0-9, 5 strategies, windows 512 B - 32 KiB, random IDAT splits, through p2p_png_decode_host_ex(formats=1) "
                     "vs cv2.imdecode; different and declined must be 0") if formats else ("random valid PNG files (4 colour types, sizes 1..159 x 1..259, filters per file / per row / adaptive, zlib levels 0-9, "
                     "5 strategies, windows 512 B - 32 KiB, memLevel 1-9, random IDAT splits, sync / full flushes) through "
                     "p2p_png_decode_host vs cv2.imdecode; different and declined must be 0")
    print(json.dumps(stats))
    return 1 if stats["different"] or stats["declined"] else 0


if __name__ == "__main__":
    sys.exit(main())
