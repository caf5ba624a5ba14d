"""The PNG decoder's wider subset on the device (P2P_OPT_PNG_FORMATS = 1: 1/2/4/16-bit gray, 16-bit RGB / gray + alpha /
RGBA, palette images, Adam7): the pixels equal ``cv2.imdecode``'s, uploads project like uploads of cv2's pixels, the files
the subset declines leave no state behind, and the front end with ``set_png_formats(True)`` writes the cv2 path's files."""
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import pytest

import png_formats_model as X
from oracle import synth
from png_formats import damaged, declines, make, matrix

pytestmark = pytest.mark.gpu


def cv2_decode(data: bytes):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


@pytest.fixture(scope="module")
def pw(pkg):
    """A context with the wider subset switched on."""
    p = pkg.Projector(0, n_slots=8)
    p.set_option(pkg._lib.OPT_PNG_FORMATS, 1)
    yield p
    p.close()


def test_device_matrix_equals_cv2(pw):
    for name, f in matrix():
        assert np.array_equal(pw.decode_png(f), cv2_decode(f)), name


def test_upload_and_projection(pkg, pw):
    """upload_png: download_pano equals cv2's pixels, and the views equal those of an upload of cv2's pixels."""
    for name, f in [("16-bit RGB", make(2, 16, 0, 257, 129, 0)), ("palette 4 bit, Adam7", make(3, 4, 1, 257, 129, 1)),
                    ("gray 2 bit", make(0, 2, 0, 257, 129, 2)), ("RGBA 16 bit, Adam7", make(6, 16, 1, 257, 129, 3))]:
        ref = cv2_decode(f)
        H, W = ref.shape[:2]
        consts = [pkg.pitch_constants(64, 90, p) for p in (60, 120)]
        shifts = [0, W // 4]   # column rolls (integer yaws)
        with pw.slots(2) as (a, b):
            assert pw.upload_png(a, f) == (W, H)
            assert np.array_equal(pw.download_pano(a, W, H), ref), name
            pw.upload(b, ref)
            va = pw.project(a, shifts, consts, 64, 48)
            vb = pw.project(b, shifts, consts, 64, 48)
            pw.sync()
        assert np.array_equal(va, vb), name


def test_full_size_files(pkg, pw):
    """An 8192 x 4096 16-bit RGB file written by cv2.imwrite and a 4096 x 2048 Adam7 file: decoded and projected."""
    base = synth.smooth(8192, 4096, 3)
    f16 = cv2.imencode(".png", base.astype(np.uint16) * 257 + np.arange(8192, dtype=np.uint16)[None, :, None] % 251)[1].tobytes()
    small = base[::2, ::2]
    laced = X.write_png(np.ascontiguousarray(small[:, :, ::-1]), 2, interlace=1, level=6)
    for name, f in [("16-bit RGB 8192 x 4096", f16), ("Adam7 4096 x 2048", laced)]:
        ref = cv2_decode(f)
        H, W = ref.shape[:2]
        assert np.array_equal(pw.decode_png(f), ref), name
        consts = [pkg.pitch_constants(400, 90, 90)]
        shifts = [0, W // 3]
        with pw.slots(2) as (a, b):
            pw.upload_png(a, f)
            pw.upload(b, ref)
            va = pw.project(a, shifts, consts, 400, 300)
            vb = pw.project(b, shifts, consts, 400, 300)
            pw.sync()
        assert np.array_equal(va, vb), name


def test_declines_leave_no_state_behind(pkg, pw):
    good = make(3, 8, 1, 257, 129, 5)
    ref = cv2_decode(good)
    for name, f in list(declines().items()) + [(f"damaged {k}", d) for k, d in enumerate(damaged(24, 3))]:
        try:
            out = pw.decode_png(f)
        except pkg.P2PError as e:
            assert e.code == -6, name
        else:
            assert name.startswith("damaged") and np.array_equal(out, cv2_decode(f)), name
        assert np.array_equal(pw.decode_png(good), ref), name


def test_option_toggled_between_calls(pkg):
    p = pkg.Projector(0, n_slots=1)
    try:
        f = make(0, 16, 1, 100, 60, 4)
        with pytest.raises(pkg.P2PError) as e:
            p.decode_png(f)
        assert e.value.code == -6
        with p.slots(1) as (s,):
            with pytest.raises(pkg.P2PError):
                p.upload_png(s, f)
        p.set_option(pkg._lib.OPT_PNG_FORMATS, 1)
        assert p.get_option(pkg._lib.OPT_PNG_FORMATS) == 1
        assert np.array_equal(p.decode_png(f), cv2_decode(f))
        p.set_option(pkg._lib.OPT_PNG_FORMATS, 0)
        with pytest.raises(pkg.P2PError):
            p.decode_png(f)
    finally:
        p.close()


def test_eight_threads_decode_new_formats_at_once(pw):
    files = [make(ct, d, k % 2, 200 + 9 * k, 120 + 5 * k, k) for k, (ct, d) in enumerate([(0, 16), (2, 16), (3, 1), (3, 8), (0, 2),
                                                                                         (6, 16), (4, 16), (2, 8)])]
    refs = [cv2_decode(f) for f in files]

    def work(k):
        return all(np.array_equal(pw.decode_png(files[k]), refs[k]) for _ in range(3))

    with ThreadPoolExecutor(8) as ex:
        assert all(ex.map(work, range(8)))


def test_front_end_new_formats_equal_imread_path(pkg, tmp_path):
    """main over 16-bit / palette / interlaced / damaged files with set_png_formats(True): the same PNG and JPEG files as
    the cv2 path."""
    src = tmp_path / "in"
    src.mkdir()
    pano = synth.smooth(1024, 512, 22)
    cv2.imwrite(str(src / "a.png"), pano.astype(np.uint16) * 257)
    (src / "b.png").write_bytes(make(3, 8, 0, 1024, 512, 7))
    (src / "c.png").write_bytes(X.write_png(np.ascontiguousarray(pano[:, :, ::-1]), 2, interlace=1))
    (src / "d.png").write_bytes(make(0, 4, 1, 1024, 512, 8))
    dmg = bytearray((src / "c.png").read_bytes())
    dmg[len(dmg) // 2] ^= 0x10
    (src / "e.png").write_bytes(bytes(dmg))
    W, H, fov, yaws, pitches = 200, 120, 100, [0, 90, 30], [60, 120]
    out_png, out_jpg = tmp_path / "png", tmp_path / "jpg"
    pkg.set_png_formats(True)
    try:
        pkg.main(str(src), str(out_png), yaws, pitches, W, H, num_workers=3, output_format="png", fov_deg=fov)
        pkg.main(str(src), str(out_jpg), yaws, pitches, W, H, num_workers=3, output_format="jpg", fov_deg=fov)
    finally:
        pkg.set_png_formats(False)
    for stem in "abcde":
        img = cv2.imread(str(src / f"{stem}.png"))
        for y in yaws:
            for p in pitches:
                fp, fj = out_png / f"{stem}_{W}x{H}_yaw_{y}_pitch_{p}.png", out_jpg / f"{stem}_{W}x{H}_yaw_{y}_pitch_{p}.jpg"
                if img is None:
                    assert not fp.exists() and not fj.exists(), stem
                    continue
                view = pkg.process_yaw_and_pitchs(img, y, [p], W, H, fov)[0]
                assert np.array_equal(cv2.imread(str(fp)), view), (stem, y, p)
                assert fj.read_bytes() == cv2.imencode(".jpg", view)[1].tobytes(), (stem, y, p)
