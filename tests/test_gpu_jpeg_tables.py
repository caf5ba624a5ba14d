"""The device JPEG decoder on Huffman tables and layouts cv2 does not write by default: cv2's optimised tables
(IMWRITE_JPEG_OPTIMIZE, as stitchers, ``cjpeg -optimize`` and PIL ``optimize=True`` write them), luma / chroma qualities
that differ, and every policy and layout of tests/jpeg_writer.py - 16-bit codes, DC tables of more than 16 entries,
end-of-block aliases, table ids 2 / 3, fill bytes.  Every file through every P2P_OPT_GPU_HUFFMAN mode, against cv2."""
import cv2
import numpy as np
import pytest

import jpeg_writer as jw
from oracle import synth

pytestmark = pytest.mark.gpu

SAMPLING = {"420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444}


def _image(kind, w, h, seed):
    if kind == "noise":
        return synth.noise(w, h, seed)
    if kind == "sat":
        return (np.random.default_rng(seed).integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    img = synth.smooth(w, h, seed)
    if kind == "textured":
        rng = np.random.default_rng(seed)
        img = np.clip(img.astype(np.int16) + rng.integers(-12, 13, img.shape, dtype=np.int16), 0, 255).astype(np.uint8)
    return img


def imdecode(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


def decode_every_mode(pkg, proj, data, ref, label):
    """decode_jpeg with the device Huffman stage (optimistic 1, plain rounds 2, host-checked 3) and the host stage (0):
    cv2's pixels every time, and in modes 1 to 3 the device stage finished the file (the count of device-decoded files
    advances by exactly one: a fallback to the host decoder takes its count back)."""
    L = pkg._lib
    try:
        for mode in (1, 2, 3, 0):
            proj.set_option(L.OPT_GPU_HUFFMAN, mode)
            n0 = proj.get_option(L.OPT_GPU_HUFFMAN_COUNT)
            got = proj.decode_jpeg(data)
            assert np.array_equal(got, ref), (label, mode)
            assert proj.get_option(L.OPT_GPU_HUFFMAN_COUNT) == n0 + (1 if mode else 0), (label, mode, "device stage did not finish")
    finally:
        proj.set_option(L.OPT_GPU_HUFFMAN, 1)


def optimised_cases():
    # (saturated binary noise stays at low quality: at quality 100 almost every coefficient is non-zero, blocks carry no
    # end of block that re-aligns a decoder started at a wrong zigzag index, the synchronisation rounds do not reach their
    # fixed point within kMaxSyncRounds and the host decoder takes the file by design, whatever the tables)
    combos = [(20, "sat", 0), (75, "textured", 7), (95, "noise", 1), (100, "smooth", 0)]
    for i, (w, h) in enumerate([(1, 1), (17, 33), (240, 136), (1000, 333), (2048, 1024)]):
        for j, sname in enumerate(("420", "422", "444", "gray")):
            picks = (combos[3], combos[1]) if w * h > 10 ** 6 else (combos[(i + j) % 4], combos[(i + j + 2) % 4])
            for q, kind, rst in picks:
                yield f"{w}x{h} {sname} q{q} {kind} rst{rst}", w, h, sname, q, kind, rst


@pytest.mark.parametrize("label,w,h,sname,q,kind,rst", list(optimised_cases()), ids=[c[0] for c in optimised_cases()])
def test_optimised_files_decode_like_cv2(pkg, proj, label, w, h, sname, q, kind, rst):
    img = _image(kind, w, h, w + q)
    params = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if sname == "gray":
        img = np.ascontiguousarray(img[..., 1])
    else:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
    default = cv2.imencode(".jpg", img, params)[1].tobytes()
    data = cv2.imencode(".jpg", img, params + [cv2.IMWRITE_JPEG_OPTIMIZE, 1])[1].tobytes()
    ref = imdecode(data)
    assert np.array_equal(ref, imdecode(default))          # same coefficients, other tables
    decode_every_mode(pkg, proj, data, ref, label)
    assert np.array_equal(proj.decode_jpeg(default), ref)


def test_luma_and_chroma_qualities_that_differ(pkg, proj):
    img = _image("textured", 1000, 333, 5)
    for lq, cq, opt in ((95, 30, 0), (20, 100, 1), (100, 60, 1)):
        data = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_LUMA_QUALITY, lq, cv2.IMWRITE_JPEG_CHROMA_QUALITY, cq,
                                          cv2.IMWRITE_JPEG_OPTIMIZE, opt])[1].tobytes()
        decode_every_mode(pkg, proj, data, imdecode(data), (lq, cq, opt))


def writer_sources():
    for kind in ("smooth", "noise"):
        for (w, h), sname in (((240, 136), "420"), ((1000, 333), "444"), ((1000, 333), "420"), ((240, 136), "gray")):
            if kind == "noise" and w == 1000 and sname == "420":
                continue
            yield f"{kind} {w}x{h} {sname}", kind, w, h, sname


@pytest.mark.parametrize("label,kind,w,h,sname", list(writer_sources()), ids=[c[0] for c in writer_sources()])
def test_writer_tables_and_layouts_decode_like_cv2(pkg, proj, label, kind, w, h, sname):
    """Every jpeg_writer policy and layout: same pixels as the source file, through every mode."""
    lib = pkg._lib.load()
    img = _image(kind, w, h, 7)
    params = [cv2.IMWRITE_JPEG_QUALITY, 92]
    if sname == "gray":
        img = np.ascontiguousarray(img[..., 0])
    else:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
    src = cv2.imencode(".jpg", img, params)[1].tobytes()
    ref = imdecode(src)
    source = jw.read_coefficients(src, lib)
    for name, kw in jw.variants(1 if sname == "gray" else 3):
        data = jw.write(src, source=source, **kw)
        assert np.array_equal(imdecode(data), ref), name
        decode_every_mode(pkg, proj, data, ref, f"{label} {name}")


# ---- panorama scale ---------------------------------------------------------------------------------------------------
def test_optimised_and_16_bit_panoramas_project_like_imread(pkg, proj):
    """An 8192 x 4096 panorama with cv2's optimised tables, and the same coefficients with every symbol a 16-bit code
    (every code word through the slow path): upload_jpeg + project give the views of the cv2.imread pixels."""
    Wp, Hp, W, H, fov = 8192, 4096, 320, 200, 110
    lib = pkg._lib.load()
    data = cv2.imencode(".jpg", _image("textured", Wp, Hp, 12), [cv2.IMWRITE_JPEG_OPTIMIZE, 1])[1].tobytes()
    ref = imdecode(data)
    long_codes = jw.write(data, tables="all_len(16)", source=jw.read_coefficients(data, lib))
    assert np.array_equal(imdecode(long_codes), ref)
    shifts = [pkg.yaw_table(Wp, y)[2] for y in (0, 90, 180, 270)]
    consts = [pkg.pitch_constants(W, fov, p) for p in (30, 90, 150)]
    L = pkg._lib
    with proj.slots(1) as (s,):
        proj.upload(s, ref)
        want = proj.project(s, shifts, consts, W, H)
        proj.sync(s)
        for f in (data, long_codes):
            n0 = proj.get_option(L.OPT_GPU_HUFFMAN_COUNT)
            assert proj.upload_jpeg(s, f) == (Wp, Hp)
            got = proj.project(s, shifts, consts, W, H)
            proj.sync(s)
            assert proj.get_option(L.OPT_GPU_HUFFMAN_COUNT) == n0 + 1
            assert np.array_equal(got, want)
        assert np.array_equal(proj.download_pano(s, Wp, Hp), ref)


def test_largest_optimised_panorama(pkg, proj):
    data = cv2.imencode(".jpg", synth.smooth(16384, 8192, 8), [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_OPTIMIZE, 1])[1].tobytes()
    n0 = proj.get_option(pkg._lib.OPT_GPU_HUFFMAN_COUNT)
    assert np.array_equal(proj.decode_jpeg(data), imdecode(data))
    assert proj.get_option(pkg._lib.OPT_GPU_HUFFMAN_COUNT) == n0 + 1


def test_front_end_optimised_and_long_dc_table_files_equal_imread_path(pkg, tmp_path):
    """The directory pipeline over an optimised file and a file whose DC table has 28 entries (codes in use at index
    16 and up): the files written equal what the cv2.imread pixels give."""
    src = tmp_path / "in"
    src.mkdir()
    pano = _image("textured", 2048, 1024, 21)
    opt = cv2.imencode(".jpg", pano, [cv2.IMWRITE_JPEG_OPTIMIZE, 1])[1].tobytes()
    (src / "opt.jpg").write_bytes(opt)
    base = cv2.imencode(".jpg", pano[:, ::-1].copy(), [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    (src / "dcdup.jpg").write_bytes(jw.write(base, tables="dc_dup", source=jw.read_coefficients(base, pkg._lib.load())))
    W, H, fov, yaws, pitches = 200, 120, 100, [0, 90, 30], [60, 120]
    out = tmp_path / "out"
    pkg.main(str(src), str(out), yaws, pitches, W, H, num_workers=2, output_format="png", fov_deg=fov)
    for name in ("opt", "dcdup"):
        img = cv2.imread(str(src / f"{name}.jpg"))
        for y in yaws:
            views = pkg.process_yaw_and_pitchs(img, y, pitches, W, H, fov)
            for p, view in zip(pitches, views):
                assert np.array_equal(cv2.imread(str(out / f"{name}_{W}x{H}_yaw_{y}_pitch_{p}.png")), view), (name, y, p)
