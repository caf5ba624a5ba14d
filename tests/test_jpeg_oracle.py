"""The JPEG oracle (oracle/jpeg_model.py: integer restatement of libjpeg-turbo at OpenCV's defaults) pinned byte for
byte against the real encoder behind the reference's ``cv2.imwrite`` (ref :277)."""
import cv2
import numpy as np
import pytest

from oracle import jpeg_model as jm
from oracle import synth


def images():
    rng = np.random.default_rng(7)
    for (h, w) in [(1, 1), (8, 8), (16, 16), (17, 33), (37, 53), (40, 56), (136, 240)]:
        yield f"noise{w}x{h}", rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        yy, xx = np.mgrid[0:h, 0:w]
        yield f"smooth{w}x{h}", np.stack([(127 + 120 * np.sin(xx / 7.0 + c) * np.cos(yy / 5.0)).astype(np.uint8)
                                          for c in range(3)], -1)
    yield "flat", np.full((24, 40, 3), 255, np.uint8)
    yield "black", np.zeros((9, 70, 3), np.uint8)
    yield "pano", synth.smooth(256, 128, 1)


@pytest.mark.parametrize("name,img", list(images()), ids=[n for n, _ in images()])
def test_oracle_equals_cv2_imencode(name, img):
    ref = cv2.imencode(".jpg", img)[1].tobytes()
    assert jm.encode(img) == ref


@pytest.mark.parametrize("quality", [1, 30, 50, 75, 95, 100])
def test_oracle_quality_scaling(quality):
    img = synth.smooth(96, 64, 2)
    ref = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, quality])[1].tobytes()
    assert jm.encode(img, quality) == ref


def test_oracle_file_equals_imwrite(tmp_path):
    img = synth.noise(64, 48, 3)
    path = tmp_path / "x.jpg"
    cv2.imwrite(str(path), img)   # the call at ref :277
    assert path.read_bytes() == jm.encode(img)


# ---- the decode side: oracle/jpeg_decode_model.py against cv2.imdecode (what cv2.imread does at ref :244) ----------
SAMPLING = {"420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444}


def jpeg_files():
    rng = np.random.default_rng(11)
    for (h, w) in [(1, 1), (2, 3), (3, 4), (17, 33), (40, 56), (47, 95)]:
        for sname, sv in SAMPLING.items():
            for q, rst in ((100, 0), (95, 0), (75, 3), (20, 1)):
                img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if q != 20 else \
                    (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
                data = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst,
                                                  cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sv])[1].tobytes()
                yield f"{w}x{h}_{sname}_q{q}_rst{rst}", data


@pytest.mark.parametrize("name,data", list(jpeg_files()), ids=[n for n, _ in jpeg_files()])
def test_decoder_oracle_equals_cv2_imdecode(name, data):
    from oracle import jpeg_decode_model as jd

    ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
    assert np.array_equal(jd.decode(data), ref)


def test_host_huffman_stage_equals_oracle(pkg):
    """The C++ entropy decoder inside the library (no GPU needed) against the oracle's coefficient planes."""
    import ctypes as C

    from oracle import jpeg_decode_model as jd

    lib = pkg._lib.load()
    for name, data in jpeg_files():
        lay = (C.c_int32 * 10)()
        assert lib.p2p_jpeg_coefficients(data, len(data), None, 0, lay) == 0, name
        n = sum(lay[4 + 2 * k] * lay[5 + 2 * k] * 64 for k in range(3))
        coef = np.zeros(n, np.int16)
        assert lib.p2p_jpeg_coefficients(data, len(data), coef.ctypes.data, n, lay) == 0, name
        planes, _ = jd.entropy_decode(jd.parse(data))
        assert np.array_equal(coef, np.concatenate([p.reshape(-1) for p in planes]).astype(np.int16)), name


def _coefficients(lib, data):
    import ctypes as C

    lay = (C.c_int32 * 10)()
    if lib.p2p_jpeg_coefficients(data, len(data), None, 0, lay) != 0:
        return None
    coef = np.zeros(sum(lay[4 + 2 * k] * lay[5 + 2 * k] * 64 for k in range(3)), np.int16)
    return coef if lib.p2p_jpeg_coefficients(data, len(data), coef.ctypes.data, coef.size, lay) == 0 else None


def progressive_cases():
    rng = np.random.default_rng(21)
    for (h, w) in [(1, 1), (8, 8), (17, 33), (47, 95), (128, 200), (333, 500)]:
        for sname, sv in SAMPLING.items():
            for q, rst in ((95, 0), (75, 0), (50, 5), (100, 1)):
                kind = (h * 7 + w + q) % 3
                img = (rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if kind == 0 else synth.smooth(w, h, q) if kind == 1
                       else np.clip(synth.smooth(w, h, q).astype(int) + rng.integers(-20, 21, (h, w, 3)), 0, 255).astype(np.uint8))
                yield f"{w}x{h}_{sname}_q{q}_rst{rst}", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst,
                                                              cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sv]


def test_progressive_files_give_the_baseline_coefficients(pkg):
    """Progressive files (SOF2: DC / AC, first / refinement scans, end-of-band runs, restart intervals; decoded by the
    library's host decoder, no GPU needed): the quantised coefficients are the ones the baseline file of the same image
    holds - the two differ only in their entropy coding - and cv2 decodes both files to the same pixels, which the oracle's
    IDCT / upsampling / colour model reproduces from these coefficients."""
    from oracle import jpeg_decode_model as jd

    lib = pkg._lib.load()
    n = 0
    for name, img, params in progressive_cases():
        base = cv2.imencode(".jpg", img, params)[1].tobytes()
        prog = cv2.imencode(".jpg", img, params + [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
        assert b"\xff\xc2" in prog[:800], name
        want, got = _coefficients(lib, base), _coefficients(lib, prog)
        assert want is not None and got is not None, name
        assert np.array_equal(got, want), name
        ref = cv2.imdecode(np.frombuffer(prog, np.uint8), cv2.IMREAD_COLOR)
        assert np.array_equal(ref, cv2.imdecode(np.frombuffer(base, np.uint8), cv2.IMREAD_COLOR)), name
        if img.shape[0] <= 128:   # (the NumPy model is slow)
            p = jd.parse(base)
            planes, _ = jd.entropy_decode(p)
            shapes = [pl.shape for pl in planes]
            mine, o = [], 0
            for sh in shapes:
                k = int(np.prod(sh))
                mine.append(got[o:o + k].reshape(sh).astype(planes[0].dtype))
                o += k
            assert np.array_equal(jd.reconstruct(p, mine), ref), name
        n += 1
    # grayscale progressive files, and files the decoder must decline: a scan script that stops before full precision
    # (libjpeg then smooths blocks from their neighbours), a truncated file
    g = synth.smooth(100, 60, 3)[..., 1]
    gb = cv2.imencode(".jpg", g, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    gp = cv2.imencode(".jpg", g, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    assert np.array_equal(_coefficients(lib, gp), _coefficients(lib, gb))
    prog = cv2.imencode(".jpg", synth.smooth(200, 120, 5), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    assert _coefficients(lib, prog) is not None
    last_sos = prog.rfind(b"\xff\xda")
    assert _coefficients(lib, prog[:last_sos] + b"\xff\xd9") is None      # last refinement scan missing
    assert _coefficients(lib, prog[:len(prog) * 2 // 3]) is None            # truncated
    assert n >= 60


def test_unsupported_files_are_reported(pkg):
    import ctypes as C

    lib = pkg._lib.load()
    w, h = C.c_int(), C.c_int()
    img = synth.smooth(64, 48, 1)
    prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    gray = cv2.imencode(".jpg", img[..., 0])[1].tobytes()
    png = cv2.imencode(".png", img)[1].tobytes()
    ok = cv2.imencode(".jpg", img)[1].tobytes()
    cmyk = ok.replace(b"\xff\xc0\x00\x11\x08", b"\xff\xc0\x00\x14\x08", 1)   # a frame header announcing more data
    for data in (png, ok[:300], cmyk, b""):
        assert lib.p2p_jpeg_probe(data, len(data), C.byref(w), C.byref(h)) == -6
    assert lib.p2p_jpeg_probe(prog, len(prog), C.byref(w), C.byref(h)) == 0 and (w.value, h.value) == (64, 48)
    assert lib.p2p_jpeg_probe(gray, len(gray), C.byref(w), C.byref(h)) == 0 and (w.value, h.value) == (64, 48)
    assert lib.p2p_jpeg_probe(ok, len(ok), C.byref(w), C.byref(h)) == 0 and (w.value, h.value) == (64, 48)
    # a truncated scan must not be decoded with made-up bits: libjpeg has its own recovery, the file is left to it
    lay = (C.c_int32 * 10)()
    big = cv2.imencode(".jpg", synth.noise(64, 48, 2))[1].tobytes()
    assert lib.p2p_jpeg_coefficients(big, len(big), None, 0, lay) == 0
    coef = np.zeros(sum(lay[4 + 2 * k] * lay[5 + 2 * k] * 64 for k in range(3)), np.int16)
    assert lib.p2p_jpeg_coefficients(big, len(big), coef.ctypes.data, coef.size, lay) == 0
    cut = big[:len(big) // 2]
    assert lib.p2p_jpeg_coefficients(cut, len(cut), coef.ctypes.data, coef.size, lay) == -6
    cut_eoi = cut + b"\xff\xd9"
    assert lib.p2p_jpeg_coefficients(cut_eoi, len(cut_eoi), coef.ctypes.data, coef.size, lay) == -6
    # EXIF orientation 6 (rotated): cv2.imread would rotate the image, so the device decoder declines
    exif = (b"Exif\x00\x00MM\x00\x2a\x00\x00\x00\x08\x00\x01\x01\x12\x00\x03\x00\x00\x00\x01\x00\x06\x00\x00"
            b"\x00\x00\x00\x00")
    seg = b"\xff\xe1" + (len(exif) + 2).to_bytes(2, "big") + exif
    rotated = ok[:2] + seg + ok[2:]
    assert lib.p2p_jpeg_probe(rotated, len(rotated), C.byref(w), C.byref(h)) == -6


def _host_stage(lib, data):
    """(status, coefficient planes as the oracle lays them out) of the library's host entropy decoder."""
    import ctypes as C

    lay = (C.c_int32 * 10)()
    st = lib.p2p_jpeg_coefficients(data, len(data), None, 0, lay)
    if st:
        return st, None
    shapes = [(lay[5 + 2 * k], lay[4 + 2 * k], 64) for k in range(3)]
    coef = np.zeros(sum(a * b * c for a, b, c in shapes), np.int16)
    st = lib.p2p_jpeg_coefficients(data, len(data), coef.ctypes.data, coef.size, lay)
    if st:
        return st, None
    planes, off = [], 0
    for sh in shapes:
        n = sh[0] * sh[1] * 64
        planes.append(coef[off:off + n].astype(np.int64).reshape(sh))
        off += n
    return 0, planes


def test_damaged_files_are_declined_or_decode_like_cv2(pkg, capfd):
    """Seeded damage in headers and scans (tests/jpeg_damage.py): the host stage declines, or its coefficients give
    cv2.imdecode's pixels; what cv2 cannot read is always declined.  (libjpeg has its own recovery heuristics - restart
    resynchronisation, zero feeding, 16-bit SIMD wrap-around on out-of-range blocks - which are left to it.)"""
    from jpeg_damage import damaged_files
    from oracle import jpeg_decode_model as jd

    lib = pkg._lib.load()
    # cv2's default tables, its optimised tables, and hand-built ones (16-bit codes only, a DC table of 28 entries whose
    # codes in use sit at index 16 and up, size-0 symbols other than 0x00 as end of block)
    for writer, seed, n in ((None, 2025, 400), ("optimize", 2026, 160), ("all_len(16)", 2027, 60), ("dc_dup", 2028, 60),
                            ("eob_alias", 2029, 60)):
        declined = same = 0
        for label, data in damaged_files(seed, n, gray_every=4, progressive_every=3, writer=writer):
            ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
            st, planes = _host_stage(lib, data)
            if st:
                assert st == -6, label
                declined += 1
                continue
            assert ref is not None, label
            assert np.array_equal(jd.reconstruct(jd.parse(data), planes), ref), label
            same += 1
        # (damage in 16-bit codes mostly makes codes that do not exist: few of those files stay decodable)
        assert declined > n // 8 and same > (50 if writer is None else 3), (writer, declined, same)
    capfd.readouterr()               # libjpeg's warnings about the damaged files


def test_known_damage_patterns_are_declined(pkg):
    import ctypes as C

    lib = pkg._lib.load()
    w, h = C.c_int(), C.c_int()

    def probe(d):
        return lib.p2p_jpeg_probe(bytes(d), len(d), C.byref(w), C.byref(h))

    img = synth.noise(64, 48, 3)
    ok = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_RST_INTERVAL, 1])[1].tobytes()
    assert probe(ok) == 0
    dht = ok.find(b"\xff\xc4")
    # a DC symbol > 15 (libjpeg: bogus Huffman table), an over-subscribed code length (would index past the lookup
    # table), the all-ones code in use
    bad = bytearray(ok); bad[dht + 5 + 16 + 3] = 0x23
    assert probe(bad) == -6
    bad = bytearray(ok); bad[dht + 5] = 200
    assert probe(bad) == -6
    bad = bytearray(ok); bad[dht + 5:dht + 5 + 16] = bytes([2] + [0] * 15); bad[dht + 2:dht + 4] = (2 + 17 + 2).to_bytes(2, "big")
    bad[dht + 5 + 16 + 2:dht + 5 + 16 + 12] = b""
    assert probe(bad) == -6
    # an unknown marker segment, a 16-bit quantisation table, a restart marker out of sequence
    bad = bytearray(ok); bad[3] = 0xF0
    assert probe(bad) == -6
    dqt = ok.find(b"\xff\xdb")
    bad = bytearray(ok); bad[dqt + 4] |= 0x10
    assert probe(bad) == -6
    sos = ok.find(b"\xff\xda")
    rst = ok.find(b"\xff\xd1", sos)
    bad = bytearray(ok); bad[rst + 1] = 0xD3
    lay = (C.c_int32 * 10)()
    assert lib.p2p_jpeg_coefficients(bytes(bad), len(bad), None, 0, lay) == 0
    coef = np.zeros(sum(lay[4 + 2 * k] * lay[5 + 2 * k] * 64 for k in range(3)), np.int16)
    assert lib.p2p_jpeg_coefficients(ok, len(ok), coef.ctypes.data, coef.size, lay) == 0
    assert lib.p2p_jpeg_coefficients(bytes(bad), len(bad), coef.ctypes.data, coef.size, lay) == -6


def test_host_decoder_under_address_sanitizer(tmp_path):
    """The header parser, the device table builder and the host Huffman decoder, built with ASan + UBSan
    (tools/asan_jpeg_host.cu), on seeded damaged files incl. garbage runs and truncations, with cv2's default, optimised and
    hand-built tables: no out-of-bounds access, no undefined behaviour."""
    import itertools
    import shutil
    import subprocess
    from pathlib import Path

    from jpeg_damage import damaged_files

    root = Path(__file__).resolve().parents[1]
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not on PATH")
    exe = tmp_path / "asan_jpeg_host"
    build = subprocess.run(["nvcc", "-O1", "-g", "-Xcompiler", "-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer",
                            "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(root / "tools" / "asan_jpeg_host.cu"),
                            "-lasan", "-lubsan"], capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + build.stderr[-300:])
    rng = np.random.default_rng(9)
    names = []
    files = itertools.chain(damaged_files(301, 600, gray_every=3, progressive_every=4),
                            damaged_files(302, 150, gray_every=3, progressive_every=4, writer="optimize"),
                            damaged_files(303, 60, gray_every=3, writer="all_len(16)"),
                            damaged_files(304, 60, gray_every=3, writer="dc_dup"),
                            damaged_files(305, 60, gray_every=3, writer="fast_ac_edge"))
    for k, (label, data) in enumerate(files):
        d = bytearray(data)
        if k % 3 == 0:                                     # heavier damage: garbage runs, truncation
            for _ in range(int(rng.integers(1, 6))):
                a, n = int(rng.integers(2, len(d))), int(rng.integers(1, 24))
                d[a:a + n] = bytes(rng.integers(0, 256, n, dtype=np.uint8))
            if rng.integers(0, 3) == 0:
                d = d[:int(rng.integers(2, len(d)))]
        f = tmp_path / f"{k:04d}.jpg"
        f.write_bytes(bytes(d))
        names.append(str(f))
    run = subprocess.run([str(exe)] + names, capture_output=True, text=True, env={"ASAN_OPTIONS": "detect_leaks=0"})
    assert run.returncode == 0 and "runtime error" not in run.stderr and "ERROR" not in run.stderr, run.stderr[-2000:]
    assert run.stdout.startswith("decoded ")


def test_colour_space_rule_follows_libjpeg(pkg):
    """Adobe-marked files (Photoshop / Lightroom), files without any marker, RGB component ids: decoded when libjpeg
    takes them for YCbCr (same pixels as cv2), declined when it takes them for RGB - oracle, probe and host stage."""
    import ctypes as C

    from jpeg_damage import colour_space_variants
    from oracle import jpeg_decode_model as jd

    lib = pkg._lib.load()
    w, h = C.c_int(), C.c_int()
    img = synth.smooth(96, 64, 3)
    base_pixels = None
    for label, data, ycc in colour_space_variants(img):
        ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
        assert ref is not None, label
        if base_pixels is None:
            base_pixels = ref
        assert np.array_equal(ref, base_pixels) == ycc, label          # cv2 itself follows the rule
        assert (lib.p2p_jpeg_probe(data, len(data), C.byref(w), C.byref(h)) == 0) == ycc, label
        if ycc:
            assert np.array_equal(jd.decode(data), ref), label
            st, planes = _host_stage(lib, data)
            assert st == 0 and np.array_equal(jd.reconstruct(jd.parse(data), planes), ref), label
        else:
            with pytest.raises(jd.Unsupported):
                jd.decode(data)


def gray_files():
    rng = np.random.default_rng(23)
    for k, (h, w) in enumerate([(1, 1), (7, 9), (8, 8), (17, 33), (40, 56), (47, 95), (64, 200)]):
        for q, rst in ((95, 0), (60, 2), (15, 1)):
            g = synth.noise(w, h, k)[..., 0] if q != 60 else synth.smooth(w, h, k)[..., 1]
            yield f"{w}x{h}_q{q}_rst{rst}", cv2.imencode(".jpg", g, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst])[1].tobytes()


@pytest.mark.parametrize("name,data", list(gray_files()), ids=[n for n, _ in gray_files()])
def test_grayscale_files_decode_like_cv2_imread(pkg, name, data):
    """cv2.imread(path) of a grayscale JPEG returns B = G = R = Y (libjpeg's gray -> RGB conversion); a single-component
    scan has one block per MCU.  Oracle against cv2, host stage against the oracle (luma plane; the chroma planes the
    device pipeline keeps for such files are all zero)."""
    from oracle import jpeg_decode_model as jd

    ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
    assert ref.shape[2] == 3 and np.array_equal(ref[..., 0], ref[..., 1]) and np.array_equal(ref[..., 0], ref[..., 2])
    assert np.array_equal(jd.decode(data), ref)
    st, planes = _host_stage(pkg._lib.load(), data)
    oracle_planes, _ = jd.entropy_decode(jd.parse(data))
    assert st == 0 and np.array_equal(planes[0], oracle_planes[0]) and not planes[1].any() and not planes[2].any()


def test_block_norm_bound_never_declines_valid_extreme_files(pkg):
    """The damaged-data bound (dequantised block norm <= 2048) against the harshest valid content: checkerboards, 1-pixel
    stripes, binary noise, hard edges at qualities 1 .. 100 (all-255 quantisation tables at quality 1), colour and
    grayscale, 4:4:4 / 4:2:2 / 4:2:0 - every file must pass the host stage (measured maximum: 1249, a checkerboard at
    quality 1)."""
    import ctypes as C

    lib = pkg._lib.load()
    rng = np.random.default_rng(0)
    w, h = 67, 45
    yy, xx = np.mgrid[0:h, 0:w]
    pats = {
        "checker": np.repeat((((xx + yy) & 1) * 255)[..., None], 3, 2),
        "vstripes": np.repeat(((xx & 1) * 255)[..., None], 3, 2),
        "hstripes": np.repeat(((yy & 1) * 255)[..., None], 3, 2),
        "binary": rng.integers(0, 2, (h, w, 3)) * 255,
        "blocks4": np.repeat(np.repeat(rng.integers(0, 2, (h // 4 + 1, w // 4 + 1, 3)) * 255, 4, 0), 4, 1)[:h, :w],
        "colour_checker": np.stack([((xx + yy) & 1) * 255, ((xx // 2 + yy) & 1) * 255, ((xx + yy // 2) & 1) * 255], -1),
        "half": np.concatenate([np.zeros((h, w // 2, 3)), np.full((h, w - w // 2, 3), 255)], 1),
    }
    for q in (1, 2, 3, 5, 10, 50, 100):
        for samp in SAMPLING.values():
            for name, img in pats.items():
                img = np.ascontiguousarray(img, dtype=np.uint8)
                for src in (img, np.ascontiguousarray(img[..., 0])):
                    data = cv2.imencode(".jpg", src, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp])[1].tobytes()
                    st, _ = _host_stage(lib, data)
                    assert st == 0, (q, samp, name, src.ndim)
