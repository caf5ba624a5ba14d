"""The PNG and JPEG encoders at the largest images they accept, and the first ones they refuse.

The PNG encoder takes W, H < 32767 and fewer than 2^31 filtered bytes N = H (1 + 3 W).  White noise is stored
uncompressed, so from N > 2^29 on its zlib stream passes 2^32 bits: 16384 x 11000 noise (N = 540,683,000) puts its later
blocks behind that point, where a 32-bit block offset would wrap.  The largest case, 32766 x 21846 (N = 2,147,439,954),
needs about 14 GB of device scratch and about 10 GB of host memory (the image, cv2's file, the device's file and the
page-locked file buffer).  Files are compared as arrays, without extra copies."""
import cv2
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def big(pkg):
    """A context of its own, closed at the end of the module: its scratch and file buffers are large."""
    p = pkg.Projector(0, n_slots=1)
    yield p
    p.close()


def _noise(W, H, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


def _same_as_cv2(got, img, ext=".png", params=()):
    ok, ref = cv2.imencode(ext, img, list(params))
    assert ok and got is not None
    return len(got) == ref.size and np.array_equal(np.frombuffer(got, np.uint8), ref.reshape(-1))


def test_png_noise_stream_past_2pow32_bits(big):
    W, H = 16384, 11000
    img = _noise(W, H, 1)
    got = big.encode_png(img)[0]
    assert len(got) * 8 > 2 ** 32
    assert _same_as_cv2(got, img)


@pytest.mark.parametrize("kind", ["noise", "ramp"])
def test_png_largest_n(big, kind):
    W, H = 32766, 21846
    assert H * (1 + 3 * W) == 2_147_439_954 < 2 ** 31 <= (H + 1) * (1 + 3 * W)
    if kind == "noise":
        img = _noise(W, H, 2)
    else:   # filtered bytes all 1: runs of 258 over the whole image, 8.3 M tokens, many tiles and blocks
        ramp = (np.arange(W) & 255).astype(np.uint8)
        img = np.ascontiguousarray(np.broadcast_to(ramp[None, :, None], (H, W, 3)))
    got = big.encode_png(img)[0]
    assert _same_as_cv2(got, img)


@pytest.mark.parametrize("W,H", [(32766, 1), (32766, 3), (1, 32766), (3, 32766)])
def test_png_longest_sides(big, W, H):
    img = _noise(W, H, W + H)
    assert _same_as_cv2(big.encode_png(img)[0], img)


@pytest.mark.parametrize("W,H", [(32766, 21847), (32767, 1), (1, 32767)])
def test_png_refuses_past_the_limit(pkg, big, W, H):
    img = np.zeros((H, W, 3), np.uint8)
    with pytest.raises(pkg.P2PError) as e:
        big.encode_png(img)
    assert e.value.code == -5


def test_jpeg_largest_square(big):
    """10288 x 10288 is the largest square the JPEG encoder takes (4:2:0: 2,480,694 blocks of at most 64 x 27 bits stay
    below 2^32 bits): saturated binary noise at quality 100, the most bits per block cv2 writes."""
    n = 10288
    img = (np.random.default_rng(3).integers(0, 2, (n, n, 3), dtype=np.uint8) * 255)
    assert _same_as_cv2(big.encode_jpeg(img, 100)[0], img, ".jpg", (cv2.IMWRITE_JPEG_QUALITY, 100))


@pytest.mark.parametrize("W,H", [(10289, 10289), (65536, 8)])
def test_jpeg_refuses_past_the_limit(pkg, big, W, H):
    with pytest.raises(pkg.P2PError) as e:
        big.encode_jpeg(np.zeros((H, W, 3), np.uint8))
    assert e.value.code == -5


def test_jpeg_widest(big):
    """65500 pixels: the widest JPEG cv2 (libjpeg-turbo) writes; the device encoder takes up to 65535."""
    img = _noise(65500, 16, 4)
    assert _same_as_cv2(big.encode_jpeg(img)[0], img, ".jpg")
