"""The device PNG decoder on designed deflate streams (tests/deflate_writer.py): header shapes zlib never writes, dynamic
blocks at every residue of a stream word, history across block and group starts and the 32 KiB edge, false candidates of
the block-start search, and the files declined on purpose at the present limits.

The expected outcome of every file comes from cv2: where ``cv2.imdecode`` returns None the device must decline (-6);
otherwise the device must return cv2's pixels - and must not decline - except for the named decline classes, which must
decline exactly.  ``P2P_OPT_PNG_HOST_BLOCKS`` must not move: a dynamic block the search misses is measured on the host
and still decodes, so only the counter shows the miss.  Files whose false candidates overflow the search's capacity may
decode or decline (which candidates are kept depends on the order of atomics) but never differ from cv2."""
import cv2
import numpy as np
import pytest

import deflate_writer as D

pytestmark = pytest.mark.gpu


def cv2_decode(data: bytes):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


@pytest.mark.parametrize("design", D.all_designs(), ids=lambda d: d.name)
def test_designed_streams_decode_like_cv2(pkg, proj, design):
    L = pkg._lib
    ref = cv2_decode(design.png)
    n0 = proj.get_option(L.OPT_PNG_HOST_BLOCKS)
    if ref is None or design.expect.startswith("decline:"):
        with pytest.raises(pkg.P2PError) as ei:
            proj.decode_png(design.png)
        assert ei.value.code == -6
        if ref is not None:   # (a damaged dynamic block fails the search's header test: the walk measures it, and counts it)
            assert proj.get_option(L.OPT_PNG_HOST_BLOCKS) == n0
        return
    if design.expect == "overflow":
        try:
            got = proj.decode_png(design.png)
        except pkg.P2PError as e:
            assert e.code == -6
        else:
            assert np.array_equal(got, ref)
        return
    got = proj.decode_png(design.png)
    assert np.array_equal(got, ref)
    assert proj.get_option(L.OPT_PNG_HOST_BLOCKS) == n0, "a dynamic block was not found by the device search"


def test_designed_stream_with_all_formats(pkg, proj):
    """The extended formats share the inflate: one designed stream with P2P_OPT_PNG_FORMATS = 1."""
    L = pkg._lib
    d = next(d for d in D.corpus()["headers"] if d.name == "all_lengths_and_distances")
    proj.set_option(L.OPT_PNG_FORMATS, 1)
    try:
        assert np.array_equal(proj.decode_png(d.png), cv2_decode(d.png))
    finally:
        proj.set_option(L.OPT_PNG_FORMATS, 0)


def test_panorama_flushed_every_row_through_upload_and_projection(pkg, proj):
    """8192 x 4096 with a zlib partial flush per row: 4096 dynamic blocks and 4096 empty fixed blocks (walked on the host),
    history chains through every group of the tail pass.  upload_png + project against the cv2.imread path."""
    L = pkg._lib
    pano, png = D.panorama_flushed_per_row()
    ref = cv2_decode(png)
    assert np.array_equal(ref, pano)
    Wp, Hp, W, H, fov = 8192, 4096, 320, 200, 100
    shifts = [pkg.yaw_table(Wp, y)[2] for y in (0, 90, 180, 270)]
    consts = [pkg.pitch_constants(W, fov, p) for p in (45, 90, 135)]
    n0 = proj.get_option(L.OPT_PNG_HOST_BLOCKS)
    with proj.slots(1) as (s,):
        assert proj.upload_png(s, png) == (Wp, Hp)
        got = proj.project(s, shifts, consts, W, H)
        proj.sync(s)
        assert np.array_equal(proj.download_pano(s, Wp, Hp), pano)
        proj.upload(s, ref)
        want = proj.project(s, shifts, consts, W, H)
        proj.sync(s)
    assert np.array_equal(got, want)
    assert proj.get_option(L.OPT_PNG_HOST_BLOCKS) == n0


def test_directory_of_designed_files_through_main(pkg, tmp_path):
    """Designed files (rows of 4095 gray pixels and more) through the directory pipeline: the same views as the cv2.imread
    path."""
    src, out = tmp_path / "in", tmp_path / "out"
    src.mkdir()
    dims = {d.name: (int.from_bytes(d.png[16:20], "big"), int.from_bytes(d.png[20:24], "big")) for d in D.all_designs()}
    picks = [d for d in D.all_designs() if d.expect == "decode" and min(dims[d.name]) >= 8][:6]
    assert len(picks) >= 4
    for d in picks:
        (src / f"{d.name}.png").write_bytes(d.png)
    W, H, fov, yaws, pitches = 96, 64, 90, [0, 180], [90]
    pkg.main(str(src), str(out), yaws, pitches, W, H, num_workers=2, output_format="png", fov_deg=fov)
    for d in picks:
        img = cv2.imread(str(src / f"{d.name}.png"))
        for y in yaws:
            view = pkg.process_yaw_and_pitchs(img, y, pitches, W, H, fov)[0]
            assert np.array_equal(cv2.imread(str(out / f"{d.name}_{W}x{H}_yaw_{y}_pitch_90.png")), view), (d.name, y)
