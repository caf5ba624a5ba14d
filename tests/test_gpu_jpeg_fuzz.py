"""Seeded random differential tests of the device JPEG encoder / decoder against cv2 (libjpeg-turbo), plus the
largest BASELINE shapes (4K views, a 16K panorama)."""
import cv2
import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu

SAMPLING = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]


def random_image(rng, w, h):
    kind = rng.integers(0, 5)
    if kind == 0:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:
        return (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    if kind == 2:
        return np.full((h, w, 3), rng.integers(0, 256, 3), np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([(127 + 120 * np.sin(xx / rng.uniform(2, 30) + c) * np.cos(yy / rng.uniform(2, 30))) for c in range(3)], -1)
    if kind == 4:
        img = img + rng.integers(-20, 21, img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


def test_encoder_fuzz(proj):
    rng = np.random.default_rng(2024)
    for i in range(48):
        w, h = int(rng.integers(1, 320)), int(rng.integers(1, 240))
        q = int(rng.integers(1, 101))
        img = random_image(rng, w, h)
        ref = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes()
        assert proj.encode_jpeg(img, quality=q)[0] == ref, (i, w, h, q)


def test_decoder_fuzz(proj):
    rng = np.random.default_rng(4202)
    for i in range(48):
        w, h = int(rng.integers(1, 320)), int(rng.integers(1, 240))
        q = int(rng.integers(5, 101))
        rst = int(rng.integers(0, 6))
        samp = SAMPLING[int(rng.integers(0, 3))]
        img = random_image(rng, w, h)
        data = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst,
                                          cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp])[1].tobytes()
        ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
        assert np.array_equal(proj.decode_jpeg(data), ref), (i, w, h, q, rst, samp)


def test_largest_shapes(proj):
    view = synth.smooth(3840, 2160, 5)                                  # a C4 view
    assert proj.encode_jpeg(view)[0] == cv2.imencode(".jpg", view)[1].tobytes()
    assert proj.encode_png(view)[0] == cv2.imencode(".png", view)[1].tobytes()
    pano = synth.smooth(16384, 8192, 6)                                 # the C4 panorama as a JPEG file
    data = cv2.imencode(".jpg", pano, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
    got = proj.decode_jpeg(data)
    assert np.array_equal(got, ref)


def test_damaged_files_are_declined_or_decode_like_cv2(pkg, proj, capfd):
    """tests/jpeg_damage.py through the whole device decoder, with the Huffman stage on the device and on the host: a
    damaged file is declined (-6: the front end then uses cv2.imread, like the reference) or decodes to cv2's pixels;
    a file cv2 cannot read is always declined.  Larger images than the CPU test so that scans span many subsequences;
    files with cv2's default and with its optimised Huffman tables."""
    from jpeg_damage import damaged_files

    L = pkg._lib
    counts = {}
    for writer, seed, n in ((None, 77, 300), ("optimize", 78, 150)):
        for device_stage in (1, 0):
            proj.set_option(L.OPT_GPU_HUFFMAN, device_stage)
            declined = same = 0
            try:
                for label, data in damaged_files(seed, n, max_wh=(400, 300), gray_every=5, progressive_every=4, writer=writer):
                    ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
                    try:
                        got = proj.decode_jpeg(data)
                    except pkg.P2PError as e:
                        assert e.code == -6, (label, e)
                        declined += 1
                        continue
                    assert ref is not None, label
                    assert np.array_equal(got, ref), (label, device_stage)
                    same += 1
            finally:
                proj.set_option(L.OPT_GPU_HUFFMAN, 1)
            counts[(writer, device_stage)] = (declined, same)
            assert declined > n // 10 and same > n // 10, counts
    capfd.readouterr()
    # the decoder still works after all that
    img = synth.smooth(320, 200, 3)
    data = cv2.imencode(".jpg", img)[1].tobytes()
    assert np.array_equal(proj.decode_jpeg(data), cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR))


def test_many_threads_mixed_files(pkg):
    """Eight host threads, one slot each, decoding a mix of files at once through both entry points: smooth and textured
    files (the optimistic enqueue passes its device-side gate), white noise (needs ~80 synchronisation rounds: the gate stays
    closed and the host continues from the states reached), restart intervals (host destuffing), grayscale, progressive
    (host scans), a file with bytes behind its EOI (irregular for the device destuffing pass) and damaged files (declined).
    Every result is compared with cv2; sleeping host waits (P2P_OPT_HOST_WAIT) are switched on for half of the run."""
    from concurrent.futures import ThreadPoolExecutor

    from jpeg_damage import damaged_files

    L = pkg._lib
    rng = np.random.default_rng(4)
    smooth = synth.smooth(1024, 512, 2)
    textured = np.clip(smooth.astype(np.int16) + rng.integers(-14, 15, smooth.shape, dtype=np.int16), 0, 255).astype(np.uint8)
    enc = lambda img, *p: cv2.imencode(".jpg", img, list(p))[1].tobytes()   # noqa: E731
    files = [
        enc(smooth, cv2.IMWRITE_JPEG_QUALITY, 95),
        enc(textured, cv2.IMWRITE_JPEG_QUALITY, 90),
        enc(synth.noise(768, 384, 1), cv2.IMWRITE_JPEG_QUALITY, 95),
        enc(textured, cv2.IMWRITE_JPEG_QUALITY, 85, cv2.IMWRITE_JPEG_RST_INTERVAL, 7),
        enc(smooth[..., 1], cv2.IMWRITE_JPEG_QUALITY, 92),
        enc(textured[:333, :1000], cv2.IMWRITE_JPEG_QUALITY, 80, cv2.IMWRITE_JPEG_PROGRESSIVE, 1),
        enc(smooth, cv2.IMWRITE_JPEG_QUALITY, 75) + b"trailing bytes behind the EOI marker",
    ]
    files += [d for _, d in damaged_files(5, 6, max_wh=(300, 200))]
    refs = [cv2.imdecode(np.frombuffer(d, np.uint8), cv2.IMREAD_COLOR) for d in files]
    proj = pkg.Projector(0, n_slots=8)
    try:
        def one(k):
            i = k % len(files)
            data, ref = files[i], refs[i]
            try:
                if k % 2:
                    got = proj.decode_jpeg(data)
                else:
                    with proj.slots(1) as (s,):
                        w, h = proj.upload_jpeg(s, data)
                        got = proj.download_pano(s, w, h)
            except pkg.P2PError as e:
                assert e.code == -6, (i, e)
                return "declined"
            assert ref is not None and np.array_equal(got, ref), i
            return "same"

        for wait in (0, 1):
            proj.set_option(L.OPT_HOST_WAIT, wait)
            with ThreadPoolExecutor(8) as ex:
                res = list(ex.map(one, range(26 * 8)))
            assert res.count("same") >= 7 * 16 - 8, res
        n0 = proj.get_option(L.OPT_GPU_HUFFMAN_COUNT)
        assert n0 >= 2 * 26 * 4        # smooth, textured, noise, restart, gray, trailing: the device stage ran
    finally:
        proj.close()

