"""The device PNG encoder (csrc/p2p_png.cuh) on the designed streams of tests/png_streams.py: literal / length trees
deeper than 15 bits, bit-length trees deeper than 7, fixed-code blocks with every length code, the largest tree
descriptions, stored blocks at every bit residue, exact block fills and runs at the tokeniser's tile and look-ahead
edges.  tests/test_png_streams_oracle.py shows on the CPU that the corpus reaches these paths; here every file must be
the bytes cv2.imencode('.png') writes."""
import cv2
import numpy as np
import pytest

import png_streams as ps

pytestmark = pytest.mark.gpu

CORPUS = ps.corpus()


def ref_png(img):
    return cv2.imencode(".png", img)[1].tobytes()


@pytest.mark.parametrize("fam,name,W,F", CORPUS, ids=[f"{c[0]}-{c[1]}" for c in CORPUS])
def test_designed_stream_equals_cv2(proj, fam, name, W, F):
    img = ps.image_from_filtered(F, W)
    got = proj.encode_png(img)[0]
    assert got is not None and got == ref_png(img), (fam, name)


def test_designed_batch_with_different_block_counts(proj):
    """Same-size images in one call: one block (a single run), three blocks with an empty last one (16383 run-free
    bytes: 14 x 381 ... x 2), stored blocks (noise), and runs across every tile boundary."""
    W, H = 14, 2 * 381
    imgs = [ps.image_from_filtered(np.full(H * (1 + 3 * W), 1, np.uint8), W),
            ps.image_from_filtered(ps.background(H, W, 1), W),
            np.random.default_rng(2).integers(0, 256, (H, W, 3), dtype=np.uint8),
            ps.image_from_filtered(ps.with_runs(H, W, 3, [(k * ps.TILE - 1 - k, k * ps.TILE + 300) for k in range(1, 8)]), W)]
    files = proj.encode_png(np.stack(imgs))
    for i, (f, img) in enumerate(zip(files, imgs)):
        assert f == ref_png(img), i
