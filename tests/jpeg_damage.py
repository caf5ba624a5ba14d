"""Damaged JPEG files for the decoder tests: seeded bit flips, overwritten, deleted and inserted bytes in the headers
or in the entropy-coded scan of files written by cv2.  The rule under test: the device decoder either declines such a
file (status -6, the caller falls back to cv2.imread as the reference does for every file) or returns exactly the
pixels cv2.imdecode returns; a file cv2 cannot read at all must be declined."""
import cv2
import numpy as np

from tools import synth_inputs as synth

SAMPLING = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]


def damaged_files(seed: int, count: int, max_wh=(120, 90), gray_every: int = 0, progressive_every: int = 0, writer=None):
    """Yields (label, bytes).  ``gray_every`` = k: every k-th file is a grayscale JPEG; ``progressive_every`` = k: every
    k-th file (offset by one) is a progressive JPEG.  ``writer``: None = cv2's default (Annex K) tables, "optimize" = cv2's
    IMWRITE_JPEG_OPTIMIZE tables, or a tests/jpeg_writer.py table policy (the cv2 file re-encoded with it before the
    damage; no progressive files then)."""
    rng = np.random.default_rng(seed)
    for i in range(count):
        w, h = int(rng.integers(16, max_wh[0])), int(rng.integers(16, max_wh[1]))
        img = synth.smooth(w, h, i) if i % 2 else synth.noise(w, h, i)
        if gray_every and i % gray_every == 0:
            img = np.ascontiguousarray(img[..., 0])
        rst, q = int(rng.integers(0, 4)), int(rng.integers(5, 100))
        samp = SAMPLING[int(rng.integers(0, 3))]
        prog = 1 if progressive_every and i % progressive_every == (1 if progressive_every > 1 else 0) else 0
        if writer not in (None, "optimize"):
            prog = 0
        data = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst,
                                          cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp, cv2.IMWRITE_JPEG_PROGRESSIVE, prog,
                                          cv2.IMWRITE_JPEG_OPTIMIZE, int(writer == "optimize")])[1].tobytes()
        if writer not in (None, "optimize"):
            import jpeg_writer

            data = jpeg_writer.write(data, tables=writer)
        data = bytearray(data)
        sos = data.find(b"\xff\xda")
        lo, hi = ((2, sos + 14), (sos + 14, len(data) - 2), (2, len(data) - 2))[int(rng.integers(0, 3))]
        mode = int(rng.integers(0, 3))
        if mode == 0:
            for _ in range(int(rng.integers(1, 4))):
                data[int(rng.integers(lo, hi))] ^= 1 << int(rng.integers(0, 8))
        elif mode == 1:
            data[int(rng.integers(lo, hi))] = int(rng.integers(0, 256))
        elif rng.integers(0, 2):
            del data[int(rng.integers(lo, hi))]
        else:
            data.insert(int(rng.integers(lo, hi)), int(rng.integers(0, 256)))
        yield f"{i}:{w}x{h} q{q} rst{rst} mode{mode}{' progressive' if prog else ''}{' ' + writer if writer else ''} [{lo},{hi})", bytes(data)


def colour_space_variants(img):
    """(label, file bytes, YCbCr?) - one 4:4:4 file with its JFIF / Adobe markers rearranged: libjpeg guesses the colour space
    from them (jdapimin.c default_decompress_parms): JFIF -> YCbCr; else Adobe transform 0 -> RGB, other -> YCbCr; else by
    component ids."""
    base = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444])[1].tobytes()
    assert base[2:4] == b"\xff\xe0"
    n0 = (base[4] << 8) | base[5]
    jfif, rest = base[2:4 + n0], base[4 + n0:]

    def adobe(transform, size=12):
        body = (b"Adobe" + b"\x00\x64" + b"\x00\x00" + b"\x00\x00" + bytes([transform]))[:size]
        return b"\xff\xee" + (len(body) + 2).to_bytes(2, "big") + body

    soi = base[:2]
    sof = rest.find(b"\xff\xc0")
    rgb_ids = bytearray(rest)
    for k, cid in enumerate(b"RGB"):                     # component ids in SOF0 and SOS
        rgb_ids[sof + 4 + 6 + 3 * k] = cid
    sos = bytes(rgb_ids).find(b"\xff\xda")
    for k, cid in enumerate(b"RGB"):
        rgb_ids[sos + 5 + 2 * k] = cid
    rgb_ids = bytes(rgb_ids)
    yield "jfif", base, True
    yield "jfif+adobe1", soi + jfif + adobe(1) + rest, True
    yield "jfif+adobe0", soi + jfif + adobe(0) + rest, True
    yield "adobe1", soi + adobe(1) + rest, True
    yield "adobe2", soi + adobe(2) + rest, True
    yield "adobe0", soi + adobe(0) + rest, False
    yield "short adobe segment", soi + adobe(0, size=7) + rest, True
    yield "no marker", soi + rest, True
    yield "no marker, ids RGB", soi + rgb_ids, False
    yield "jfif, ids RGB", soi + jfif + rgb_ids, True
    yield "adobe1, ids RGB", soi + adobe(1) + rgb_ids, True
