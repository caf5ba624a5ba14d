"""The PNG decoder's wider subset (P2P_OPT_PNG_FORMATS = 1: 1/2/4/16-bit gray, 16-bit RGB / gray + alpha / RGBA, palette
images, Adam7) on the CPU: the reference (``tests/png_formats_model.py``) and the library's host model of the device decoder
(``p2p_png_decode_host_ex``, the kernels' own routines run serially) against ``cv2.imdecode``; with ``formats = 0`` the same
files are declined exactly as before; the files the wider subset must still decline; routing of the front end."""
import ctypes as C

import cv2
import numpy as np
import pytest

import png_formats_model as X
from oracle import png_decode_model as M
from png_formats import FORMATS, damaged, declines, make, matrix

MATRIX = matrix()


def cv2_decode(data: bytes):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


@pytest.fixture(scope="module")
def lib(pkg):
    return pkg._lib.load()


def host_decode(lib, data: bytes, formats: int):
    w, h = C.c_int(), C.c_int()
    rc = lib.p2p_png_probe_ex(data, len(data), formats, C.byref(w), C.byref(h))
    if rc:
        return rc, None
    out = np.zeros((h.value, w.value, 3), np.uint8)
    rc = lib.p2p_png_decode_host_ex(data, len(data), formats, out.ctypes.data, out.strides[0], h.value, None)
    return rc, (out if rc == 0 else None)


@pytest.mark.parametrize("ct,depth", FORMATS, ids=[f"type{c}_{d}bit" for c, d in FORMATS])
def test_matrix_oracle_and_host_model_equal_cv2(lib, ct, depth):
    """Every size x interlace of the format (filters 0-4 / adaptive / per row, noise / smooth / mixed content), PLTE shorter
    than 2^depth, tRNS (gray, RGB, shorter than PLTE), a suggested PLTE, gAMA / sBIT / bKGD / iCCP."""
    files = [(n, f) for n, f in MATRIX if n.startswith(f"ct{ct}_d{depth}_")]
    assert len(files) >= 2 * 6 + 2
    for name, f in files:
        ref = cv2_decode(f)
        assert ref is not None, name
        assert X.in_subset(f) is not None, name
        assert np.array_equal(X.decode(f), ref), name
        rc, out = host_decode(lib, f, 1)
        assert rc == 0 and np.array_equal(out, ref), name


def test_option_off_declines_the_new_formats_as_before(lib):
    """formats = 0: p2p_png_probe_ex / p2p_png_decode_host_ex decline exactly the files p2p_png_probe declines, and decode
    the 8-bit non-interlaced ones as before."""
    n_new = 0
    for name, f in MATRIX:
        w, h = C.c_int(), C.c_int()
        old = lib.p2p_png_probe(f, len(f), C.byref(w), C.byref(h))
        rc, out = host_decode(lib, f, 0)
        assert (old == 0) == (rc == 0) and (old == 0) == (M.in_subset(f) is not None), name
        if rc == 0:
            assert np.array_equal(out, cv2_decode(f)), name
        else:
            assert rc == -6 and old == -6, name
            n_new += 1
    assert n_new > 200


def test_formats_argument_is_checked(lib):
    f = MATRIX[0][1]
    w, h = C.c_int(), C.c_int()
    assert lib.p2p_png_probe_ex(f, len(f), 2, C.byref(w), C.byref(h)) == -1
    assert lib.p2p_png_probe_ex(f, len(f), -1, C.byref(w), C.byref(h)) == -1


@pytest.mark.parametrize("name", list(declines()))
def test_declined_with_the_wider_subset(lib, name):
    f = declines()[name]
    rc, out = host_decode(lib, f, 1)
    assert rc == -6 and out is None


def test_damaged_new_format_files_decode_like_libpng_or_not_at_all(lib):
    """Seeded bit flips / truncations of 16-bit, palette, 2-bit gray and Adam7 files: decoded like cv2 or declined."""
    declined = decoded = 0
    for f in damaged(240, 7):
        rc, out = host_decode(lib, f, 1)
        if rc == 0:
            ref = cv2_decode(f)
            assert ref is not None and np.array_equal(out, ref)
            decoded += 1
        else:
            assert rc == -6
            declined += 1
    assert declined > 200


def test_open_image_routes_by_the_switch(pkg, tmp_path):
    """_open_image: with set_png_formats(True) a 16-bit / palette / interlaced file stays bytes for the device decoder; with it
    off (the default) cv2.imread reads it.  No GPU needed: only the chunk walk runs."""
    from importlib import import_module

    front = import_module(pkg.__name__ + ".panorama_to_plane_pitch")
    files = {"16bit.png": make(2, 16, 0, 33, 17, 1), "palette.png": make(3, 4, 0, 33, 17, 2), "laced.png": make(2, 8, 1, 33, 17, 3)}
    for name, data in files.items():
        (tmp_path / name).write_bytes(data)
    assert front._png_formats == 0
    for name in files:
        got = front._open_image(tmp_path / name)
        assert isinstance(got, np.ndarray) and np.array_equal(got, cv2.imread(str(tmp_path / name))), name
    front._png_formats = 1   # (set_png_formats also sets the option of every projector already made: none without a GPU)
    try:
        for name in files:
            got = front._open_image(tmp_path / name)
            assert isinstance(got, front._JpegSource) and (got.Wp, got.Hp) == (33, 17), name
    finally:
        front._png_formats = 0
    assert front.build_parser().parse_args(["--input_path", "x", "--png_all_formats"]).png_all_formats


def test_host_model_under_address_sanitizer_new_formats(tmp_path):
    """tools/asan_png_host.cu --formats 1 (ASan + UBSan) over damaged new-format files and the declined ones."""
    import shutil
    import subprocess
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not on PATH")
    exe = tmp_path / "asan_png_host"
    build = subprocess.run(["nvcc", "-O1", "-g", "-Xcompiler", "-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer",
                            "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(root / "tools" / "asan_png_host.cu"),
                            "-lasan", "-lubsan"], capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + build.stderr[-300:])
    names = []
    for k, f in enumerate(damaged(300, 23) + list(declines().values()) + [f for _, f in MATRIX[::5]]):
        p = tmp_path / f"{k:04d}.png"
        p.write_bytes(f)
        names.append(str(p))
    run = subprocess.run([str(exe), "--formats", "1"] + names, capture_output=True, text=True, env={"ASAN_OPTIONS": "detect_leaks=0"})
    assert run.returncode == 0 and "runtime error" not in run.stderr and "ERROR" not in run.stderr, run.stderr[-2000:]
    assert run.stdout.startswith("decoded ")
    assert int(run.stdout.split()[1]) >= len(MATRIX[::5])
