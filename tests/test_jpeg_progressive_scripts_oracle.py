"""Progressive (SOF2) files with scan scripts cv2 does not write, through the library's host stage (no GPU needed).

tests/jpeg_writer.py ``write_progressive`` restates libjpeg's jcphuff.c; it is first checked against libjpeg itself (byte
for byte cv2's progressive file with libjpeg's script), then used to re-encode the coefficients of baseline files with
the scripts of mozjpeg, Photoshop, ``jpegtran -scans`` and edge cases: separate and partial DC scans, several
refinement levels, one-coefficient bands, end-of-band runs across rows and restart intervals, tables and restart
intervals changed between scans, fill bytes.  Every such file must decode to exactly the source's coefficients, and the
files libjpeg would not decode as given must be declined."""
import ctypes as C

import cv2
import numpy as np
import pytest

import jpeg_writer as jw
from oracle import synth

SAMPLING = {"420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "gray": None}
SIZES = [(1, 1), (17, 33), (47, 95), (333, 500)]

# Valid files the decoder declines on purpose, with the reason; any other valid file that is declined fails the tests.
CONSERVATIVE = {
    "over_cap": "more than 64 scans: the scan list is capped (no encoder writes that many; cv2 decodes the file)",
}

DECLINED = -6   # p2p_jpeg_coefficients: the file is outside what the device decoder takes


def _image(kind, w, h, seed):
    if kind == "noise":
        return synth.noise(w, h, seed)
    return synth.smooth(w, h, seed)


def _baseline(sname, w, h, kind, q=90, seed=3):
    img = _image(kind, w, h, seed + w)
    params = [cv2.IMWRITE_JPEG_QUALITY, q]
    if sname == "gray":
        img = np.ascontiguousarray(img[..., 1])
    else:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
    return img, params, cv2.imencode(".jpg", img, params)[1].tobytes()


def status(lib, data):
    """(status of p2p_jpeg_coefficients, coefficient planes as read_coefficients lays them out)"""
    lay = (C.c_int32 * 10)()
    st = lib.p2p_jpeg_coefficients(data, len(data), None, 0, lay)
    if st:
        return st, None
    shapes = [(lay[5 + 2 * k], lay[4 + 2 * k], 64) for k in range(3)]
    coef = np.zeros(sum(a * b * c for a, b, c in shapes), np.int16)
    st = lib.p2p_jpeg_coefficients(data, len(data), coef.ctypes.data, coef.size, lay)
    planes, off = [], 0
    for sh in shapes:
        n = sh[0] * sh[1] * 64
        planes.append(coef[off:off + n].reshape(sh))
        off += n
    return st, planes


def expected_planes(source, scans):
    """the coefficients a progressive file of ``scans`` carries: the source's, except the luma blocks of the MCU padding
    (below / right of ceil(H / 8) x ceil(W / 8) in 4:2:0 / 4:2:2), which only interleaved DC scans code - a DC scan of
    luma alone leaves them zero, as in libjpeg's coefficient buffer"""
    p, planes = source
    out = [pl.copy() for pl in planes]
    comps, hmax, vmax = jw._frame_geometry(p)
    if len(comps) == 1 or hmax * vmax == 1:
        return out
    W, H = p["frame"]["W"], p["frame"]["H"]
    Y = out[0]
    pad = np.ones(Y.shape[:2], bool)
    pad[:-(-H // 8), :-(-W // 8)] = False
    assert not Y[pad][:, 1:].any()          # (AC of the encoder's padding blocks is zero)
    dc, val = planes[0][..., 0], np.zeros(Y.shape[:2], np.int64)
    for sc, Ss, Se, Ah, Al in scans:
        if Ss == 0 and 0 in sc and len(sc) > 1:
            val = (dc >> Al) << Al if Ah == 0 else val | (dc & (1 << Al))
    Y[..., 0][pad] = val[pad]
    return out


def imdecode(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


def assert_same_pixels_silently(capfd, data, ref, label):
    """cv2 decodes ``data`` to ``ref`` and libjpeg has nothing to say about it (no "Corrupt JPEG data" warning)"""
    capfd.readouterr()
    assert np.array_equal(imdecode(data), ref), label
    err = capfd.readouterr().err
    assert "Corrupt JPEG" not in err and "JPEG" not in err, (label, err)


# ---- the writer against libjpeg ------------------------------------------------------------------------------------
def identity_cases():
    for sname in SAMPLING:
        for (w, h), kind, q, rst in (((17, 33), "noise", 95, 0), ((333, 500), "smooth", 75, 0), ((47, 95), "noise", 50, 3),
                                     ((333, 500), "noise", 100, 1), ((1, 1), "smooth", 90, 2)):
            yield f"{sname} {w}x{h} {kind} q{q} rst{rst}", sname, w, h, kind, q, rst


@pytest.mark.parametrize("label,sname,w,h,kind,q,rst", list(identity_cases()), ids=[c[0] for c in identity_cases()])
def test_simple_script_is_byte_for_byte_cv2s_progressive_file(label, sname, w, h, kind, q, rst):
    """libjpeg's jpeg_simple_progression with its per-scan optimal tables: the writer's file is the one cv2 writes (the
    coefficients come from the NumPy oracle, not from the library)"""
    img, params, _ = _baseline(sname, w, h, kind, q)
    params += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    base = cv2.imencode(".jpg", img, params)[1].tobytes()
    prog = cv2.imencode(".jpg", img, params + [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    assert jw.write_progressive(base, "simple") == prog


def test_writer_forces_out_long_runs_like_libjpeg(pkg):
    """The end-of-band run cut at 0x7FFF blocks (a smooth 1700 x 1700 gray image: 45,000 blocks whose high band is all
    zero) and at the correction-bit buffer's limit (binary noise in 4-pixel cells at quality 100: refinement bands full of
    correction bits and no new coefficient): byte for byte cv2's file"""
    lib = pkg._lib.load()
    rng = np.random.default_rng(1)
    cells = (rng.integers(0, 2, (64, 64)) * 255).astype(np.uint8).repeat(4, 0).repeat(4, 1)
    for img, q in ((synth.smooth(1700, 1700, 1)[..., 0].copy(), 50), (cells, 100)):
        base = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes()
        prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
        assert jw.write_progressive(base, "simple", source=jw.read_coefficients(base, lib)) == prog
    # the first file does reach the cut: its 6-63 band (Al 2) holds a run of exactly 0x7FFF blocks
    p = jw.read_coefficients(cv2.imencode(".jpg", synth.smooth(1700, 1700, 1)[..., 0].copy(),
                                          [cv2.IMWRITE_JPEG_QUALITY, 50])[1].tobytes(), lib)
    P = jw._Pieces()
    Z = p[1][0][:213, :213].reshape(-1, 64)[:, jw.ZIGZAG].astype(np.int64)
    has_sym, trailing, be, parts = jw._ac_pieces(P, Z, 6, 63, 0, 2, 0)
    assert trailing.sum() >= jw.MAX_EOBRUN
    P2 = jw._Pieces()
    jw._eob_runs(P2, has_sym, trailing, be, parts, np.zeros(len(Z), np.int64), 0)
    runs = P2.parts[1]
    assert ((1 << runs[7]) + runs[6] == jw.MAX_EOBRUN).any()


# ---- every script ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sname", list(SAMPLING))
@pytest.mark.parametrize("name", jw.SCRIPTS)
def test_scripts_decode_to_the_source_coefficients(pkg, capfd, name, sname):
    """Every script x sampling x size (partial MCUs at every edge) x noise / smooth content x restart interval on / off:
    cv2 reads the file silently to the baseline file's pixels, and the host stage gives exactly the coefficients the file
    carries - or declines it, for the reasons listed in CONSERVATIVE only."""
    lib = pkg._lib.load()
    n = 0
    for w, h in SIZES:
        for kind, rst in (("noise", 0), ("smooth", 0), ("noise", 2), ("smooth", 7)):
            if w * h > 10 ** 5 and (kind, rst) in (("noise", 0), ("smooth", 7)):
                continue   # (the module's time: two combinations at 333 x 500)
            _, _, base = _baseline(sname, w, h, kind)
            source = jw.read_coefficients(base, lib)
            data = jw.write_progressive(base, name, restart=rst, source=source)
            label = (name, sname, w, h, kind, rst)
            assert_same_pixels_silently(capfd, data, imdecode(base), label)
            st, planes = status(lib, data)
            if name in CONSERVATIVE:
                assert st == DECLINED, label
                continue
            assert st == 0, label
            want = expected_planes(source, jw.named(name, len(source[1]))["script"])
            for k, (got, exp) in enumerate(zip(planes, want)):
                assert np.array_equal(got, exp), (label, k)
            n += 1
    assert n >= 12 or name in CONSERVATIVE


def test_every_script_is_what_its_name_says():
    """the scripts hold the scan shapes they are named for (so that the decode tests above reach those branches)"""
    S = {n: jw.script(n) for n in jw.SCRIPTS}
    dc = lambda s: [x for x in s if x[1] == 0]
    assert S["simple"][0] == ((0, 1, 2), 0, 0, 0, 1) and len(S["simple"]) == 10
    assert all(len(x[0]) == 1 for x in dc(S["mozjpeg_like"])) and len(dc(S["mozjpeg_like"])) == 6
    assert all(x[3] == x[4] == 0 for x in S["spectral_only"])
    assert {(x[3], x[4]) for x in S["deep_sa"]} == {(0, 3), (3, 2), (2, 1), (1, 0)}
    assert sum(x[1] == x[2] != 0 for x in S["single_coef"]) >= 20 and len(S["single_coef"]) <= 63
    assert dc(S["dc_subset"])[:2] == [((0,), 0, 0, 0, 1), ((1, 2), 0, 0, 0, 1)]
    cf = S["chroma_first"]
    assert cf[1] == ((0, 1, 2), 0, 0, 1, 0) and max(k for k, x in enumerate(cf) if x[0] != (0,)) < min(
        k for k, x in enumerate(cf) if x[0] == (0,) and x[1])
    assert len(S["over_cap"]) > 64 and len(jw.script("over_cap", 1)) > 64
    rst = jw.named("rst_everywhere")["restart"]
    assert 1 in rst and 13 in rst and 0 in rst and len(set(rst)) > 2
    churn = jw.named("table_churn")
    assert {2, 3} <= {s for sl in churn["slots"] for s in sl} and churn["decoy"]


# ---- layouts and fill bytes ------------------------------------------------------------------------------------------
def test_fill_bytes_between_scans_are_skipped(pkg, capfd):
    """0xFF fill bytes in front of any marker behind a scan (the next DHT, SOS or EOI) and in front of restart markers:
    libjpeg skips them silently (jdmarker.c next_marker), so the file decodes to the same coefficients"""
    lib = pkg._lib.load()
    for sname, rst in (("420", 0), ("444", 5), ("gray", 1)):
        img, params, base = _baseline(sname, 200, 120, "smooth", seed=5)
        prog = cv2.imencode(".jpg", img, params + [cv2.IMWRITE_JPEG_PROGRESSIVE, 1, cv2.IMWRITE_JPEG_RST_INTERVAL, rst])[1].tobytes()
        ref = imdecode(prog)
        st, want = status(lib, prog)
        assert st == 0
        first = prog.find(b"\xff\xda")
        marks = [first + 2 + k for k in range(len(prog) - first - 3) if prog[first + 2 + k] == 0xFF and
                 prog[first + 3 + k] in (0xC4, 0xDA, 0xD9, 0xDD) or
                 (prog[first + 2 + k] == 0xFF and 0xD0 <= prog[first + 3 + k] <= 0xD7)]
        assert len(marks) >= 10
        for k, at in enumerate(marks):
            for fill in (b"\xff", b"\xff\xff\xff"):
                data = prog[:at] + fill + prog[at:]
                assert_same_pixels_silently(capfd, data, ref, (sname, at, len(fill)))
                st, got = status(lib, data)
                assert st == 0, (sname, at, hex(prog[at + 1]), len(fill))
                assert all(np.array_equal(a, b) for a, b in zip(got, want))
        data = prog
        for at in marks[::-1]:                       # every one at once
            data = data[:at] + b"\xff\xff" + data[at:]
        assert status(lib, data)[0] == 0


@pytest.mark.parametrize("sname", ["420", "gray"])
def test_layouts_with_progressive_scripts(pkg, capfd, sname):
    """every segment layout of the writer (COM segments between the scans, fill bytes before every marker, DRI before
    DQT, one-segment tables, tables behind SOF) with the scripts that change tables and restart intervals"""
    lib = pkg._lib.load()
    _, _, base = _baseline(sname, 47, 95, "noise")
    source = jw.read_coefficients(base, lib)
    ref = imdecode(base)
    for name in ("simple", "mozjpeg_like", "rst_everywhere", "table_churn", "deep_sa"):
        for layout in [(lay,) for lay in jw.LAYOUTS] + [jw.LAYOUTS]:
            for rst in (0, 3):
                data = jw.write_progressive(base, name, restart=rst, layout=layout, source=source)
                assert_same_pixels_silently(capfd, data, ref, (name, layout, rst))
                st, planes = status(lib, data)
                assert st == 0, (name, layout, rst)
                want = expected_planes(source, jw.named(name, len(source[1]))["script"])
                assert all(np.array_equal(a, b) for a, b in zip(planes, want)), (name, layout, rst)


# ---- files that must be declined -------------------------------------------------------------------------------------
def declined_cases(ncomp):
    Y, ALL = (0,), (0, 1, 2)[:ncomp]
    simple = jw.script("simple", ncomp)
    chroma = [((1,), 1, 63, 0, 0), ((2,), 1, 63, 0, 0)] if ncomp == 3 else []
    yield "precision left incomplete (last AC refinement missing)", simple[:-1]
    yield "precision left incomplete (DC refinement missing)", [s for s in simple if not (s[1] == 0 and s[3])]
    yield "Ah is not the previous Al", [(ALL, 0, 0, 0, 0), (Y, 1, 63, 0, 2), (Y, 1, 63, 1, 0)] + chroma
    yield "AC before DC", [(Y, 1, 63, 0, 0), (ALL, 0, 0, 0, 0)] + chroma
    yield "a band refined twice at the same level", [(ALL, 0, 0, 0, 0), (Y, 1, 63, 0, 1), (Y, 1, 63, 1, 0),
                                                     (Y, 1, 63, 1, 0)] + chroma
    if ncomp == 3:
        yield "components out of frame order", [((1, 0, 2), 0, 0, 0, 0), (Y, 1, 63, 0, 0)] + chroma
    yield "over_cap", jw.script("over_cap", ncomp)


@pytest.mark.parametrize("sname", ["420", "444", "gray"])
def test_files_outside_the_accepted_progression_are_declined(pkg, sname):
    """scan scripts libjpeg warns about or cannot bring to full precision without smoothing (jdcoefct.c
    decompress_smooth_data), and the conservative declines: -6 each, so the front end falls back to cv2.imread"""
    lib = pkg._lib.load()
    _, _, base = _baseline(sname, 47, 95, "noise")
    source = jw.read_coefficients(base, lib)
    names = []
    for label, scans in declined_cases(1 if sname == "gray" else 3):
        for rst in (0, 4):
            data = jw.write_progressive(base, scans, restart=rst, source=source)
            assert status(lib, data)[0] == DECLINED, (label, rst)
        names.append(label)
    assert set(CONSERVATIVE) <= set(names)


def test_unused_invalid_table_does_not_decline_but_a_used_one_does(pkg, capfd):
    """jdhuff.c checks a Huffman table when a scan uses it: a DHT with DC symbols above 15 (or an over-subscribed code
    length) left in a slot no scan uses before it is redefined is fine; the same table in use declines the file"""
    lib = pkg._lib.load()
    _, _, base = _baseline("420", 47, 95, "noise")
    source = jw.read_coefficients(base, lib)
    good = jw.write_progressive(base, "simple", source=source)
    st, want = status(lib, good)
    assert st == 0
    at = good.find(b"\xff\xda")
    bad_dc = bytes([0x03]) + bytes([0] * 7 + [255] + [0] * 8) + bytes(range(255))   # DC slot 3: symbols above 15
    over = bytes([0x12, 5] + [0] * 15) + bytes(range(5))       # AC slot 2: five codes of length 1
    for seg in (bad_dc, over):
        data = good[:at] + jw.segment(0xC4, seg) + good[at:]
        assert_same_pixels_silently(capfd, data, imdecode(good), seg[:2])
        st, got = status(lib, data)
        assert st == 0 and all(np.array_equal(a, b) for a, b in zip(got, want))
    # in use: the first scan's DC table for luma is the bad one
    sos = good[at:at + 14]
    used = good[:at] + jw.segment(0xC4, bad_dc) + sos[:6] + bytes([0x30]) + sos[7:] + good[at + 14:]
    assert status(lib, used)[0] == DECLINED


# ---- the host decoder under AddressSanitizer / UBSan -----------------------------------------------------------------
def test_progressive_scripts_under_address_sanitizer(pkg, tmp_path):
    """tools/asan_jpeg_host.cu over a file per script and sampling, and damaged copies of each (bit flips in the scans,
    garbage runs, truncation, a scan header's Ss / Se / Ah / Al or table id overwritten): no out-of-bounds access, no
    undefined behaviour, and the intact files decode"""
    import shutil
    import subprocess
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not on PATH")
    exe = tmp_path / "asan_jpeg_host"
    build = subprocess.run(["nvcc", "-O1", "-g", "-Xcompiler", "-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer",
                            "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(root / "tools" / "asan_jpeg_host.cu"),
                            "-lasan", "-lubsan"], capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + build.stderr[-300:])
    lib = pkg._lib.load()
    rng = np.random.default_rng(17)
    intact, damaged = [], []
    for sname in ("420", "422", "gray"):
        _, _, base = _baseline(sname, 47, 95, "noise")
        source = jw.read_coefficients(base, lib)
        for name in jw.SCRIPTS:
            data = jw.write_progressive(base, name, restart=int(rng.integers(0, 3)), source=source,
                                        layout=("fill_bytes",) if rng.integers(0, 2) else ())
            if name not in CONSERVATIVE:
                intact.append(data)
            sos = [k for k in range(len(data) - 1) if data[k] == 0xFF and data[k + 1] == 0xDA]
            for r in range(8):
                d = bytearray(data)
                if r < 3:
                    for _ in range(int(rng.integers(1, 4))):
                        a = int(rng.integers(sos[0], len(d)))
                        d[a] ^= 1 << int(rng.integers(0, 8))
                elif r < 5:
                    a, n = int(rng.integers(sos[0], len(d))), int(rng.integers(1, 24))
                    d[a:a + n] = bytes(rng.integers(0, 256, n, dtype=np.uint8))
                elif r == 5:
                    d = d[:int(rng.integers(sos[0], len(d)))]
                else:
                    s = sos[int(rng.integers(0, len(sos)))]
                    ns = d[s + 4]
                    # r == 6: Ss, Se or Ah / Al; r == 7: a component's table ids
                    field = s + 5 + 2 * ns + int(rng.integers(0, 3)) if r == 6 else s + 6 + 2 * int(rng.integers(0, ns))
                    d[field] = int(rng.integers(0, 256))
                damaged.append(bytes(d))
    names = []
    for k, data in enumerate(intact + damaged):
        f = tmp_path / f"{k:04d}.jpg"
        f.write_bytes(data)
        names.append(str(f))
    run = subprocess.run([str(exe)] + names[:len(intact)], capture_output=True, text=True, env={"ASAN_OPTIONS": "detect_leaks=0"})
    assert run.returncode == 0 and "runtime error" not in run.stderr and "ERROR" not in run.stderr, run.stderr[-2000:]
    assert run.stdout.strip() == f"decoded {len(intact)} declined 0", run.stdout
    run = subprocess.run([str(exe)] + names[len(intact):], capture_output=True, text=True, env={"ASAN_OPTIONS": "detect_leaks=0"})
    assert run.returncode == 0 and "runtime error" not in run.stderr and "ERROR" not in run.stderr, run.stderr[-2000:]
    assert run.stdout.startswith("decoded ")
