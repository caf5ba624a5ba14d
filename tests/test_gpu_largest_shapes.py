"""The largest panoramas and outputs the library accepts.

* Panorama widths above 16384 up to the limit of 32766: the texture sampler picks its 2 x 2 footprint from
  normalised coordinates, ((ix + 1) * f32(1 / Wp)) + f32(shift / Wp) with one rounded FADD, and the rounding margin of
  that addition shrinks as Wp grows.  Pole faces sweep every azimuth and the seam; fractional yaws go through the
  16-bit column table of the one-pass kernel; p2p_process_image uploads only the rows the views read.
* Outputs past 32-bit byte offsets: a view above 2 GiB (the row-segment kernel, whose offsets inside a view are
  32-bit), a batch above 4 GiB (the host leaves the row-segment kernel for the generic one) and (ny - 1) * yaw_stride
  on both sides of 2^32 (the generic kernel lowers its yaws per launch).

Large buffers stay on the device and are compared with torch.equal; oracle rows are computed on the host.
"""
import numpy as np
import pytest

from oracle import fixedpoint as fp
from oracle import ref_port, svml_model

GiB = 1 << 30


def _noise(Wp, Hp, seed):
    return np.random.default_rng(seed).integers(0, 256, (Hp, Wp, 3), dtype=np.uint8)


def _check_noise(got, want, *info):
    """Bit-identical where this host's NumPy uses SVML; otherwise the gate of tests/test_gpu_fuzz.py."""
    if svml_model.host_numpy_uses_svml():
        assert np.array_equal(got, want), info
    else:
        assert float((got == want).all(axis=-1).mean()) >= 0.93, info


def test_scalar_model_rows_subset():
    """The row subset of the scalar coordinate model is the same rows of the whole map."""
    W, H, fov, pitch, Wp, Hp = 96, 70, 100, 33, 1000, 500
    U, V = fp.pitch_coords_scalar_model(W, H, fov, pitch, Wp, Hp)
    rows = [0, 1, 34, 35, 69]
    Ur, Vr = fp.pitch_coords_scalar_model(W, H, fov, pitch, Wp, Hp, rows=rows)
    assert np.array_equal(Ur, U[rows], equal_nan=True) and np.array_equal(Vr, V[rows], equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("Wp", [16385, 24576, 32766])
def test_widest_panoramas(pkg, proj, Wp):
    Hp = Wp // 2
    pano = _noise(Wp, Hp, Wp)
    F = 2048
    poles = [pkg.pitch_constants(F, 90, p) for p in (0, 180)]
    Ws, Hs, fov_s = 2048, 1024, 100
    side = [pkg.pitch_constants(Ws, fov_s, 90)]
    rolls = [1, Wp - 3]
    frac_yaw = 33.3
    table = pkg.yaw_table(Wp, frac_yaw)
    assert table[2] is None, "the yaw is meant to be fractional"
    with proj.slots(1) as (s,):
        proj.upload(s, pano)
        proj.sync(s)
        got_poles = proj.project(s, [0], poles, F, F)
        got_side = proj.project(s, rolls, side, Ws, Hs)
        got_frac = proj.project_tables(s, [table], side, Ws, Hs)
        proj.sync(s)
        # pole faces: every azimuth, the seam included
        for j, p in enumerate((0, 180)):
            _check_noise(got_poles[0, j], fp.project_view_single_pass(pano, 0, p, F, F, 90), Wp, "pole", p)
        # side view: two integer column rolls of one coordinate map
        U, V = ref_port.pitch_mapping(Ws, Hs, fov_s, 90, Wp, Hp)
        for k, shift in enumerate(rolls):
            _check_noise(got_side[k, 0], fp.sample_view(pano, U, V, yaw_shift=shift), Wp, "roll", shift)
        # fractional yaw: the reference's yaw pass, materialised for the panorama rows the view reads only
        lo, hi = proj.view_row_range(side, Ws, Hs, Wp, Hp)
        ix, fx = fp.yaw_column_table(Wp, frac_yaw)
        rot = np.zeros_like(pano)
        for r in range(lo, min(hi + 2, Hp), 256):
            r1 = min(r + 256, hi + 2, Hp)
            rot[r:r1] = fp.apply_yaw_table(pano[r:r1], ix, fx)
        _check_noise(got_frac[0, 0], fp.sample_view(rot, U, V, yaw_shift=0), Wp, "fractional yaw")
        del rot
        # the same views through p2p_process_image, which uploads only the rows they read
        out = np.empty((1, 2, F, F, 3), np.uint8)
        proj.process_image(s, pano, [0], poles, F, F, out)
        proj.sync(s)
        assert np.array_equal(out, got_poles), (Wp, "process_image poles")
        out = np.empty((2, 1, Hs, Ws, 3), np.uint8)
        proj.process_image(s, pano, rolls, side, Ws, Hs, out)
        proj.sync(s)
        assert np.array_equal(out, got_side), (Wp, "process_image rolls")


def _device_out(torch, n_bytes):
    return torch.empty(n_bytes, dtype=torch.uint8, device="cuda:0")


@pytest.mark.gpu
def test_view_above_2gib(pkg, proj):
    """One 27000 x 27000 view (2.04 GiB, W % 8 == 0: the row-segment kernel): equal to the per-pixel kernel, whose
    offsets are 64-bit; oracle rows straddling byte offset 2^31; a p2p_project_view_list row band past 2^31 bytes equal
    to the same rows of the full view."""
    torch = pytest.importorskip("torch")
    L = pkg._lib
    Wp, Hp, W, H, fov, pitch, shift = 8192, 4096, 27000, 27000, 90, 60, 1234
    assert W * H * 3 > 2 * GiB and W % 8 == 0
    pano = _noise(Wp, Hp, 27)
    consts = [pkg.pitch_constants(W, fov, pitch)]
    row_bytes = W * 3
    v31 = (1 << 31) // row_bytes            # the row holding byte 2^31
    with proj.slots(1) as (s,):
        proj.upload(s, pano)
        proj.sync(s)
        rows = _device_out(torch, H * row_bytes)
        proj.project(s, [shift], consts, W, H, out_device_ptr=rows.data_ptr())
        proj.sync(s)
        other = _device_out(torch, H * row_bytes)
        mirror = proj.get_option(L.OPT_MIRROR)
        try:
            proj.set_option(L.OPT_MIRROR, 0)
            proj.project(s, [shift], consts, W, H, out_device_ptr=other.data_ptr())
            proj.sync(s)
        finally:
            proj.set_option(L.OPT_MIRROR, mirror)
        assert torch.equal(rows, other), "row-segment kernel differs from the per-pixel kernel"
        # oracle rows around byte offset 2^31
        sel = list(range(v31 - 2, v31 + 3))
        U, V = fp.pitch_coords_scalar_model(W, H, fov, pitch, Wp, Hp, rows=sel)
        want = fp.sample_view(pano, U, V, yaw_shift=shift)
        got = rows[sel[0] * row_bytes:(sel[-1] + 1) * row_bytes].cpu().numpy().reshape(len(sel), W, 3)
        _check_noise(got, want, "rows", sel)
        # a row band past 2^31 bytes through the flat view list
        other.zero_()
        torch.cuda.synchronize()   # the library's streams do not wait for torch's
        band = (v31 - 10, v31 + 50)
        proj.project_list(s, [shift], consts, W, H, rows=band, out_device_ptr=other.data_ptr())
        proj.sync(s)
        b0, b1 = band[0] * row_bytes, band[1] * row_bytes
        assert torch.equal(other[b0:b1], rows[b0:b1]), "view-list band differs from the full view"
        assert not other[:b0].any() and not other[b1:].any(), "view-list band wrote outside its rows"
        del rows, other
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_batch_above_4gib(pkg, proj):
    """4 yaws x 3 pitches of 11008 x 10880 (4.02 GiB): the host takes the generic kernel; every view equals the same
    view rendered alone, which takes the row-segment kernel."""
    torch = pytest.importorskip("torch")
    Wp, Hp, W, H, fov = 8192, 4096, 11008, 10880, 100
    view = W * H * 3
    assert 12 * view > 4 * GiB and view < GiB
    pano = _noise(Wp, Hp, 44)
    shifts = [0, 1000, 4096, 8191]
    consts = [pkg.pitch_constants(W, fov, p) for p in (30, 90, 150)]
    with proj.slots(1) as (s,):
        proj.upload(s, pano)
        proj.sync(s)
        batch = _device_out(torch, 12 * view)
        proj.project(s, shifts, consts, W, H, out_device_ptr=batch.data_ptr())
        proj.sync(s)
        one = _device_out(torch, view)
        for k, sh in enumerate(shifts):
            for j, c in enumerate(consts):
                proj.project(s, [sh], [c], W, H, out_device_ptr=one.data_ptr())
                proj.sync(s)
                i = k * 3 + j
                assert torch.equal(batch[i * view:(i + 1) * view], one), (sh, j)
        del batch, one
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("side", ["below", "above"])
def test_yaw_stride_at_2pow32(pkg, proj, side):
    """4 yaws of one pitch with 3 * view bytes just below / just above 2^32: below, the generic kernel takes all four
    yaws in one launch (32-bit k * yaw_stride); above, the host lowers the yaws per launch.  Both equal one-yaw
    launches."""
    torch = pytest.importorskip("torch")
    L = pkg._lib
    Wp, Hp, W, fov = 4096, 2048, 21840, 120
    H = ((1 << 32) - 1) // (3 * W * 3) + (1 if side == "above" else 0)
    view = W * H * 3
    assert (3 * view < (1 << 32)) == (side == "below") and 2 * view < (1 << 32)
    pano = _noise(Wp, Hp, 32)
    shifts = [0, 7, 2048, 4095]
    consts = [pkg.pitch_constants(W, fov, 75)]
    with proj.slots(1) as (s,):
        proj.upload(s, pano)
        proj.sync(s)
        got = _device_out(torch, 4 * view)
        n0 = proj.launches
        proj.project(s, shifts, consts, W, H, out_device_ptr=got.data_ptr())
        proj.sync(s)
        n_launch = proj.launches - n0
        want = _device_out(torch, 4 * view)
        ny = proj.get_option(L.OPT_YAWS_PER_THREAD)
        try:
            proj.set_option(L.OPT_YAWS_PER_THREAD, 1)
            n0 = proj.launches
            proj.project(s, shifts, consts, W, H, out_device_ptr=want.data_ptr())
            proj.sync(s)
            assert proj.launches - n0 == 4
        finally:
            proj.set_option(L.OPT_YAWS_PER_THREAD, ny)
        assert n_launch == (1 if side == "below" else 2), n_launch
        assert torch.equal(got, want), side
        del got, want
        torch.cuda.empty_cache()
