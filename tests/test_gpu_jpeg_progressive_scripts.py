"""The device JPEG decoder on progressive files with scan scripts cv2 does not write (tests/jpeg_writer.py
``write_progressive``): every script through decode_jpeg, upload_jpeg + download_pano and the front door, 8192 x 4096
panoramas whose scans feed all four host decode chains (DC, and the AC scans of each component), and the files the
decoder declines, which the front door hands to cv2.imread.  Pixels against cv2 every time."""
import cv2
import numpy as np
import pytest

import jpeg_writer as jw
from oracle import synth
from test_jpeg_progressive_scripts_oracle import CONSERVATIVE, declined_cases

pytestmark = pytest.mark.gpu


def imdecode(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


def _textured(w, h, seed):
    img = synth.smooth(w, h, seed)
    rng = np.random.default_rng(seed)
    return np.clip(img.astype(np.int16) + rng.integers(-12, 13, img.shape, dtype=np.int16), 0, 255).astype(np.uint8)


def _front_door(pkg, tmp_path, data, name):
    """panorama_to_plane on the file, against the view of the cv2.imread pixels (or, for a file libjpeg refuses too - scan
    components out of frame order -, the reference's "Failed to decode image")"""
    W, H, fov = 240, 136, 110
    path = tmp_path / f"{name}.jpg"
    path.write_bytes(data)
    img = cv2.imread(str(path))
    if img is None:
        with pytest.raises(ValueError, match="Failed to decode image"):
            pkg.panorama_to_plane(path, fov, (W, H), 90, 60)
        return False
    view = pkg.panorama_to_plane(path, fov, (W, H), 90, 60)
    assert np.array_equal(view, pkg.process_yaw_and_pitchs(img, 90, [60], W, H, fov)[0]), name
    return True


@pytest.mark.parametrize("name", jw.SCRIPTS)
def test_scripts_decode_like_cv2(pkg, proj, tmp_path, name):
    lib = pkg._lib.load()
    for sname, samp, (w, h), rst in (("420", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, (1000, 333), 0),
                                     ("422", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, (333, 201), 3),
                                     ("444", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, (47, 95), 1),
                                     ("gray", None, (1000, 333), 5)):
        img = _textured(w, h, w + h)
        params = [cv2.IMWRITE_JPEG_QUALITY, 92]
        if samp is None:
            img = np.ascontiguousarray(img[..., 1])
        else:
            params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp]
        base = cv2.imencode(".jpg", img, params)[1].tobytes()
        data = jw.write_progressive(base, name, restart=rst, source=jw.read_coefficients(base, lib))
        ref = imdecode(data)
        assert np.array_equal(ref, imdecode(base)), (name, sname)
        label = f"{name}_{sname}"
        if name in CONSERVATIVE:
            with pytest.raises(pkg._lib.P2PError) as e:
                proj.decode_jpeg(data)
            assert e.value.code == -6
        else:
            assert np.array_equal(proj.decode_jpeg(data), ref), label
            with proj.slots(1) as (s,):
                assert proj.upload_jpeg(s, data) == (w, h)
                assert np.array_equal(proj.download_pano(s, w, h), ref), label
        assert _front_door(pkg, tmp_path, data, label)


@pytest.mark.parametrize("name", ["mozjpeg_like", "deep_sa"])
def test_8k_progressive_panoramas(pkg, proj, name):
    """8192 x 4096, 4:2:0: separate DC scans per component (mozjpeg_like) and three refinement levels (deep_sa), so every
    decode chain runs over full-size planes; decode_jpeg and upload_jpeg + download_pano give cv2's pixels"""
    Wp, Hp = 8192, 4096
    lib = pkg._lib.load()
    base = cv2.imencode(".jpg", _textured(Wp, Hp, 31), [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    data = jw.write_progressive(base, name, source=jw.read_coefficients(base, lib))
    ref = imdecode(data)
    assert np.array_equal(ref, imdecode(base))
    assert np.array_equal(proj.decode_jpeg(data), ref)
    with proj.slots(1) as (s,):
        assert proj.upload_jpeg(s, data) == (Wp, Hp)
        assert np.array_equal(proj.download_pano(s, Wp, Hp), ref)


@pytest.mark.parametrize("sname", ["420", "gray"])
def test_declined_files_take_the_cv2_fallback(pkg, proj, tmp_path, sname):
    """files outside the accepted progression: decode_jpeg reports -6, and the front door gives the cv2.imread views (every
    file but the one with scan components out of frame order, which libjpeg refuses as well, is one cv2 reads)"""
    lib = pkg._lib.load()
    img = _textured(640, 320, 4)
    params = [cv2.IMWRITE_JPEG_QUALITY, 90]
    if sname == "gray":
        img = np.ascontiguousarray(img[..., 1])
    else:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420]
    base = cv2.imencode(".jpg", img, params)[1].tobytes()
    source = jw.read_coefficients(base, lib)
    unreadable = []
    for k, (label, scans) in enumerate(declined_cases(1 if sname == "gray" else 3)):
        data = jw.write_progressive(base, scans, source=source)
        with pytest.raises(pkg._lib.P2PError) as e:
            proj.decode_jpeg(data)
        assert e.value.code == -6, label
        if not _front_door(pkg, tmp_path, data, f"declined_{sname}_{k}"):
            unreadable.append(label)
    assert unreadable == ([] if sname == "gray" else ["components out of frame order"])
