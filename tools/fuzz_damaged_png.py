"""Damaged PNG files against the library's host model of the device decoder (the same __host__ __device__ routines as the
kernels, run serially - no GPU needed): a file must be decoded exactly like cv2.imdecode (libpng + zlib) or declined, never
differently.  Damage: bit flips / byte overwrites / deletions / insertions anywhere in the file (chunk CRCs left alone), and
the same inside the deflate data with the chunk CRC recomputed (so that only the inflate's own checks and the Adler-32 stand
between the damage and the pixels).

    python tools/fuzz_damaged_png.py [n_files] > profiles/r2_fuzz_damaged_png.jsonl
    python tools/fuzz_damaged_png.py --formats extended [n_files] > profiles/r3_fuzz_damaged_png_ext.jsonl

--formats extended: the decoder's wider subset (P2P_OPT_PNG_FORMATS = 1) on damaged 16-bit, palette (with tRNS), 1/2/4-bit
gray and Adam7 files; a damaged chunk may also be one of PLTE / tRNS.
"""
import ctypes as C
import json
import sys
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402
from oracle import png_decode_model as M  # noqa: E402


def main():
    import cv2

    args = sys.argv[1:]
    formats = 0
    if "--formats" in args:
        k = args.index("--formats")
        formats = {"default": 0, "extended": 1}[args[k + 1]]
        del args[k:k + 2]
    n_files = int(args[0]) if args else 4000
    g.build()
    lib = g.load_package()._lib.load()

    def host_decode(data):
        w, h = C.c_int(), C.c_int()
        if lib.p2p_png_probe_ex(data, len(data), formats, C.byref(w), C.byref(h)):
            return None
        out = np.zeros((h.value, w.value, 3), np.uint8)
        rc = lib.p2p_png_decode_host_ex(data, len(data), formats, out.ctypes.data, out.strides[0], h.value, None)
        return out if rc == 0 else None

    rng = np.random.default_rng(2026 + formats)
    bases = []
    if formats:
        sys.path.insert(0, str(ROOT / "tests"))
        from png_formats import make

        for k, (ct, d, lace) in enumerate([(0, 16, 1), (2, 16, 0), (3, 4, 1), (3, 8, 0), (0, 1, 0), (0, 2, 1), (4, 16, 0), (6, 16, 1),
                                           (2, 8, 1), (3, 2, 0)]):
            trns = bytes(range(3)) if ct == 3 else None
            bases.append(make(ct, d, lace, 150, 96, k, level=6, idat=[3000], trns=trns))
            bases.append(make(ct, d, lace, 150, 96, k + 1, level=1, strategy=zlib.Z_RLE))
    else:
        for k, (ctype, ch) in enumerate([(2, 3), (6, 4), (0, 1), (4, 2)]):
            img = M.test_image(96, 150, ch, k)
            bases.append(M.write_png(img, ctype, level=6, idat=[3000]))
            bases.append(M.write_png(img, ctype, level=1, strategy=zlib.Z_RLE, filters=[1] * 96))
            bases.append(M.write_png(img, ctype, level=9, flush_every=4000))
    stats = {"files": 0, "declined": 0, "decoded_identically": 0, "cv2_none_among_declined": 0, "violations": 0}
    by_kind = {}
    t0 = time.time()
    for i in range(n_files):
        base = bases[i % len(bases)]
        kind = ["flip", "byte", "delete", "insert", "z_flip", "z_byte", "z_truncate", "z_swap"][int(rng.integers(0, 8))]
        if kind.startswith("z_"):
            ch = M.chunks(base)
            z = bytearray(b"".join(b for t, b, _, _ in ch if t == b"IDAT"))
            at = int(rng.integers(2, len(z)))
            if kind == "z_flip":
                z[at] ^= 1 << int(rng.integers(0, 8))
            elif kind == "z_byte":
                z[at] = int(rng.integers(0, 256))
            elif kind == "z_truncate":
                del z[at:]
            else:
                j = int(rng.integers(2, len(z)))
                z[at], z[j] = z[j], z[at]
            rest = b"".join(M.chunk(t, b) for t, b, _, _ in ch[1:] if t not in (b"IDAT", b"IEND"))   # PLTE / tRNS
            data = M.SIG + M.chunk(b"IHDR", ch[0][1]) + rest + M.chunk(b"IDAT", bytes(z)) + M.chunk(b"IEND", b"")
        else:
            d = bytearray(base)
            at = int(rng.integers(8, len(d)))
            if kind == "flip":
                d[at] ^= 1 << int(rng.integers(0, 8))
            elif kind == "byte":
                d[at] = int(rng.integers(0, 256))
            elif kind == "delete":
                del d[at:at + int(rng.integers(1, 9))]
            else:
                d[at:at] = bytes(rng.integers(0, 256, int(rng.integers(1, 9)), dtype=np.uint8))
            data = bytes(d)
        got = host_decode(data)
        ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
        stats["files"] += 1
        k = by_kind.setdefault(kind, {"files": 0, "declined": 0, "decoded_identically": 0})
        k["files"] += 1
        if got is None:
            stats["declined"] += 1
            k["declined"] += 1
            stats["cv2_none_among_declined"] += ref is None
        elif ref is not None and ref.shape == got.shape and np.array_equal(ref, got):
            stats["decoded_identically"] += 1
            k["decoded_identically"] += 1
        else:
            stats["violations"] += 1
            print(json.dumps({"violation": kind, "file_index": i}), flush=True)
    stats["seconds"] = round(time.time() - t0, 1)
    stats["by_kind"] = by_kind
    stats["formats"] = ["default", "extended"][formats]
    stats["what"] = ("damaged PNG files through p2p_png_decode_host_ex (the device decoder's routines run serially) vs cv2.imdecode: "
                     "decoded identically or declined; violations must be 0")
    print(json.dumps(stats))
    return 1 if stats["violations"] else 0


if __name__ == "__main__":
    sys.exit(main())
