"""On the CPU: the images of tests/jpeg_symbols.py, encoded by cv2.imencode at their qualities, reach every named target
(every DC category and AC symbol of both Huffman tables with both signs, ZRL chains, coefficients at zig-zag 63, padding
that completes an 0xFF, 0xFF at every byte of a stuffing chunk, blocks at every bit of an emit word); the integer model
of the encoder writes the same bytes as cv2 for all of them; and the reciprocal quantisation of jpeg_dct_kernel is
exact over the FDCT's whole output range."""
import numpy as np
import pytest

import jpeg_symbols as js
from oracle import jpeg_model as jm

CORPUS = js.corpus()


@pytest.fixture(scope="module")
def stats():
    return {name: js.file_stats(js.cv2_jpeg(img, q)) for name, img, q in CORPUS}


def test_corpus_reaches_every_target(stats):
    got = set().union(*(js.reached(st) for st in stats.values()))
    missing = sorted(js.targets() - got)
    assert not missing, f"{len(missing)} targets not reached: {missing}"


def test_target_counts():
    """2 x 12 DC categories (11 with both signs + 0), 2 x 162 AC symbols (160 with both signs, ZRL, EOB), and the
    run / stuffing / bit-sink targets."""
    t = js.targets()
    assert sum(1 for x in t if x.startswith("dc") and "/cat" in x) == 2 * (1 + 11 * 2)
    assert sum(1 for x in t if x.startswith("ac") and "/r" in x and "s" in x.split("/")[1][1:]) == 2 * 160 * 2
    assert {"ac0/zrl", "ac0/eob", "ac1/zrl", "ac1/eob"} <= t


def test_symbol_counter_sees_what_the_builder_placed(stats):
    """The counter is not vacuous: a size-10 luma AC coefficient and DC category 11 are seen only in the images that
    were built for them, and the flat image has nothing but DC-only blocks."""
    assert not any(s == 10 for (_, s, _) in stats["flat-gray"]["ac"][0])
    assert stats["flat-gray"]["dc_only"][0] == 4 * 64 and stats["flat-gray"]["dc_only"][1] == 2 * 64
    assert any(s == 10 for (_, s, _) in stats["ac0-q100-0"]["ac"][0])
    assert any(c == 11 for (c, _) in stats["dc0-q100"]["dc"][0])


@pytest.mark.parametrize("name,img,quality", CORPUS, ids=[c[0] for c in CORPUS])
def test_model_equals_cv2(name, img, quality):
    assert jm.encode(img, quality) == js.cv2_jpeg(img, quality), name


@pytest.mark.parametrize("quality", [-1, 0, 101, 1000])
def test_cv2_clamps_quality_like_the_encoder(quality):
    """cv2 takes any quality and clamps it to 1 .. 100 as build_tables does (jm.quant_table restates the clamp)."""
    img = next(c[1] for c in CORPUS if c[0] == "ac0-q100-0")
    assert js.cv2_jpeg(img, quality) == jm.encode(img, quality)


def test_fdct_output_range():
    """Every |x| jpeg_fdct_islow can produce is below 2^14 (the sign patterns of the basis functions at full swing
    are the extremes of the linear transform): far inside the 2^18 of the quantiser's exactness claim."""
    P = np.where(js.BASIS > 0, 127, -128)
    X = jm.fdct_islow(np.concatenate([P, -P - 1]))
    assert np.abs(X).max() < 1 << 14


def test_reciprocal_quantisation_is_exact():
    """jpeg_dct_kernel: umulhi(|x| + d / 2, floor(2^32 / d) + 1) == (|x| + d / 2) / d for every divisor d = 8 q,
    q = 1 .. 255, and every numerator below 2^18 (|x| < 2^14 plus d / 2 < 2^10)."""
    n = np.arange(1 << 18, dtype=np.uint64)
    for q in range(1, 256):
        d = 8 * q
        rcp = np.uint64((1 << 32) // d + 1)
        got = (n * rcp) >> np.uint64(32)
        bad = np.flatnonzero(got != n // np.uint64(d))
        assert bad.size == 0, (q, int(n[bad[0]]))
