"""Every device path on adversarial memory: results must depend on the inputs only.

Each case runs one entry point five times and asks for the same result every time:
  - in fresh contexts whose every allocation is filled with 0x00, 0xFF and 0xA5 first (P2P_OPT_POISON);
  - on a slot that first ran the same entry point on a larger, different input and was then poisoned
    (p2p_debug_poison: everything the slot does not hold, at full capacity);
  - on the same kind of slot without the explicit poison (stale but plausible data).
The result must also equal the independent reference (oracle.fixedpoint, scipy, cv2), and the device paths must not
quietly fall back: the counters of the device JPEG Huffman stage, of the PNG blocks the device search missed and of the
kernel launches move by the same amount in every run (launches: apart from the memoised tap-row range of a geometry the
priming call already saw).  A read of memory the call did not write shows up as a difference between the runs.
"""
import ctypes as C

import cv2
import numpy as np
import pytest

import deflate_writer as D
import jpeg_writer as jw
import png_formats
from oracle import exact_bilinear as eb
from oracle import fixedpoint as fp
from oracle import svml_model, synth

pytestmark = pytest.mark.gpu

BYTES = (0x00, 0xFF, 0xA5)
STRICT = svml_model.host_numpy_uses_svml()   # else NumPy's own arccos differs from the reference in the last ulp here


# ------------------------------------------------------------------------------------------
# the contract
# ------------------------------------------------------------------------------------------
def _counters(p, L):
    return (p.get_option(L.OPT_GPU_HUFFMAN_COUNT), p.get_option(L.OPT_PNG_HOST_BLOCKS), p.launches)


def _assert_same(a, b, what):
    if isinstance(a, (list, tuple)):
        assert len(a) == len(b), what
        for i, (x, y) in enumerate(zip(a, b)):
            _assert_same(x, y, f"{what}[{i}]")
    elif isinstance(a, np.ndarray):
        assert a.shape == b.shape and np.array_equal(a, b), f"{what}: {int((a != b).sum())} bytes differ"
    else:
        assert a == b, what


def contract(pkg, run, prime, options=(), n_slots=2, prime_fresh=False):
    """``run(p)`` -> result on a context ``p`` (slot 0, others as it likes); ``prime(p)``: the same entry point on a larger,
    different input (``prime_fresh``: the fresh contexts run it too, on their poisoned allocations).  Asserts the five runs
    agree (results and counters) and returns the result with the counter deltas of a fresh context."""
    L = pkg._lib
    results, deltas = [], []

    def one(byte, primed, poisoned):
        p = pkg.Projector(0, n_slots)
        try:
            if byte is not None:
                p.set_option(L.OPT_POISON, byte)
            for k, v in options:
                p.set_option(k, v)
            if primed:
                prime(p)
                p.sync()
                if poisoned:
                    for s in range(n_slots):
                        p.poison(s, 0xA5)
            c0 = _counters(p, L)
            r = run(p)
            p.sync()
            deltas.append(tuple(b - a for a, b in zip(c0, _counters(p, L))))
            results.append(r)
        finally:
            p.close()

    for b in BYTES:
        one(b, prime_fresh, False)
    one(None, True, True)
    one(None, True, False)
    labels = [f"fresh 0x{b:02X}" for b in BYTES] + ["reused + poisoned", "reused stale"]
    for i in range(1, len(results)):
        _assert_same(results[i], results[0], f"{labels[i]} vs {labels[0]}")
    for i in range(1, len(deltas)):
        assert deltas[i][:2] == deltas[0][:2], ("device decoder counters differ", labels[i], deltas)
    assert len({d[2] for d in deltas[:3]}) == 1, ("launches differ between fresh contexts", deltas)
    assert deltas[3][2] == deltas[4][2] <= deltas[0][2], ("launches of a reused slot", deltas)
    return results[0], deltas[0]


def _poison_of(p, L):
    return p.get_option(L.OPT_POISON)


def _second_context(pkg, p):
    """A second context poisoned like ``p`` (fresh runs) or with 0xA5 (reuse runs)."""
    q = pkg.Projector(0, 1)
    b = _poison_of(p, pkg._lib)
    q.set_option(pkg._lib.OPT_POISON, b if b >= 0 else 0xA5)
    return q


# ------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------
def _rolls(pkg, Wp, yaws=(0, 90, 180, 270, 45, 135, 225, 315)):
    return [(y, pkg.yaw_table(Wp, y)[2]) for y in yaws if pkg.yaw_table(Wp, y)[2] is not None]


def _check_view(got, want, *info):
    if STRICT:
        assert np.array_equal(got, want), info
    else:
        assert (got == want).all(axis=-1).mean() >= 0.93, info


def _check_views(out, pano, views, W, H, fov):
    for i, (yaw, pitch) in enumerate(views):
        _check_view(out[i], fp.project_view_single_pass(pano, yaw, pitch, W, H, fov), yaw, pitch)


def _flat(pkg, Wp, W, fov, views):
    return [pkg.yaw_table(Wp, y)[2] for y, _ in views], [pkg.pitch_constants(W, fov, p) for _, p in views]


def _torch():
    torch = pytest.importorskip("torch")
    return torch


# ------------------------------------------------------------------------------------------
# panorama writers
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sampler", [1, 0])
@pytest.mark.parametrize("Wp", [1000, 1003, 8, 12])
def test_host_upload(pkg, Wp, sampler):
    """p2p_upload_pano at widths that are and are not multiples of 4, down to 8 columns; the views cross the seam and
    reach both poles, so the wrap column and the clamp row are read (the LDG sampler reads the linear copy)."""
    L = pkg._lib
    Hp = 61 if Wp > 12 else 6
    W, H, fov = (40, 24, 100) if Wp > 12 else (16, 8, 120)
    pano = synth.noise(Wp, Hp, Wp)
    views = [(y, p) for y, _ in _rolls(pkg, Wp)[:3] for p in (0, 90, 180)]
    shifts, consts = _flat(pkg, Wp, W, fov, views)

    def run(p):
        p.upload(0, pano)
        out = p.project_list(0, shifts, consts, W, H)
        p.sync(0)
        return [p.download_pano(0, Wp, Hp), out]

    def prime(p):
        big = synth.noise(Wp + 37, Hp + 20, 1)
        p.upload(0, big)
        p.project_list(0, [0, 5], [pkg.pitch_constants(W + 8, fov, 30)] * 2, W + 8, H + 3)
        p.upload(1, big)

    (dl, out), _ = contract(pkg, run, prime, [(L.OPT_SAMPLER, sampler)])
    assert np.array_equal(dl, pano)
    _check_views(out, pano, views, W, H, fov)


def test_device_upload_strided_unaligned(pkg):
    """p2p_upload_pano_device with row_stride > 3 Wp and source pointers 1..3 bytes past an aligned address."""
    torch = _torch()
    Wp, Hp, W, H, fov = 1003, 71, 48, 32, 110
    stride = 3 * Wp + 13
    pano = synth.noise(Wp, Hp, 4)
    views = [(0, 0), (0, 90), (180, 180)] if pkg.yaw_table(Wp, 180)[2] is not None else [(0, 0), (0, 90), (0, 180)]
    shifts, consts = _flat(pkg, Wp, W, fov, views)
    host = np.zeros((Hp, stride), np.uint8)
    host[:, :3 * Wp] = pano.reshape(Hp, -1)
    buf = torch.zeros(Hp * stride + 8, dtype=torch.uint8, device="cuda:0")

    def run(p):
        got = []
        for off in (1, 2, 3):
            buf[off:off + Hp * stride].copy_(torch.from_numpy(host.reshape(-1)))
            torch.cuda.synchronize()
            p.upload_device(0, buf.data_ptr() + off, Wp, Hp, stride)
            out = p.project_list(0, shifts, consts, W, H)
            p.sync(0)
            got += [p.download_pano(0, Wp, Hp), out]
        return got

    def prime(p):
        p.upload(0, synth.noise(Wp + 100, Hp + 40, 9))

    got, _ = contract(pkg, run, prime)
    for k in range(3):
        assert np.array_equal(got[2 * k], pano)
        _check_views(got[2 * k + 1], pano, views, W, H, fov)


def test_rows_from_pieces_and_copies(pkg):
    """A panorama assembled by p2p_upload_pano_rows from three pieces, replicated into a poisoned second context whole
    (p2p_copy_pano) and in pieces (p2p_copy_pano_rows)."""
    Wp, Hp, W, H, fov = 1000, 90, 40, 32, 100
    pano = synth.noise(Wp, Hp, 5)
    views = [(0, 0), (90, 90), (180, 180), (270, 120)]
    shifts, consts = _flat(pkg, Wp, W, fov, views)

    def run(p):
        for a, b in ((30, 61), (0, 30), (61, Hp)):
            p.upload_rows(0, pano, a, b)
        got = [p.project_list(0, shifts, consts, W, H)]
        p.sync(0)
        got.append(p.download_pano(0, Wp, Hp))
        q = _second_context(pkg, p)
        try:
            q.copy_pano_from(0, p, 0)
            got.append(q.project_list(0, shifts, consts, W, H))
            q.sync(0)
            q.upload(0, synth.noise(Wp + 5, Hp, 1))   # another panorama size: the pieces below start a new one
            q.sync(0)
            q.poison(0, 0x5A)
            for a, b in ((45, Hp + 1), (0, 45)):
                q.copy_pano_rows_from(0, p, 0, a, b)
            got.append(q.project_list(0, shifts, consts, W, H))
            q.sync(0)
            got.append(q.download_pano(0, Wp, Hp))
        finally:
            q.close()
        return got

    def prime(p):
        p.upload(0, synth.noise(Wp + 24, Hp + 50, 2))

    got, _ = contract(pkg, run, prime)
    for k in (0, 2, 3):
        _check_views(got[k], pano, views, W, H, fov)
    assert np.array_equal(got[1], pano) and np.array_equal(got[4], pano)


def test_rotate(pkg):
    """p2p_rotate_pano (the materialised yaw pass of a fractional yaw) into a poisoned slot, read back and projected."""
    Wp, Hp, W, H, fov = 1000, 80, 40, 32, 100
    pano = synth.noise(Wp, Hp, 6)
    ix, fx, shift = pkg.yaw_table(Wp, 33.3)
    assert shift is None
    rotated = fp.apply_yaw_table(pano, *fp.yaw_column_table(Wp, 33.3))
    pitches = (0, 90, 180)
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]

    def run(p):
        p.upload(0, pano)
        p.rotate(0, 1, ix, fx)
        out = p.project_list(1, [0] * len(pitches), consts, W, H)
        p.sync(1)
        return [p.download_pano(1, Wp, Hp), out]

    def prime(p):
        big = synth.noise(Wp + 40, Hp + 30, 3)
        p.upload(0, big)
        t = pkg.yaw_table(Wp + 40, 71.7)
        p.rotate(0, 1, t[0], t[1])

    (dl, out), _ = contract(pkg, run, prime)
    assert np.array_equal(dl, rotated)
    for j, pt in enumerate(pitches):
        _check_view(out[j], fp.project_view_single_pass(pano, 33.3, pt, W, H, fov), pt)


@pytest.mark.parametrize("pitches", [(90,), (0,), (180,), (30, 60)])
def test_partial_slot_renders_its_own_views_again(pkg, pitches):
    """A slot filled by p2p_process_image holds only the rows its views touch.  Poisoned around those rows, it must
    render the same views again, through the product entry and the list entry: a row range one row short reads poison."""
    Wp, Hp, W, H, fov = 1024, 512, 96, 64, 90
    pano = synth.noise(Wp, Hp, 7)
    yaws = [0, 90, 180, 270]
    shifts = [pkg.yaw_table(Wp, y)[2] for y in yaws]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]
    flat = [(y, pt) for y in yaws for pt in pitches]
    fs, fc = _flat(pkg, Wp, W, fov, flat)

    def run(p):
        out = np.empty((len(yaws), len(pitches), H, W, 3), np.uint8)
        p.process_image(0, pano, shifts, consts, W, H, out)
        p.sync(0)
        p.poison(0, 0x5A)
        again = p.project(0, shifts, consts, W, H)
        p.sync(0)
        p.poison(0, 0xC3)
        listed = p.project_list(0, fs, fc, W, H)
        p.sync(0)
        return [out, again, listed]

    def prime(p):
        out = np.empty((4, len(pitches), H, W, 3), np.uint8)
        p.process_image(0, synth.noise(Wp, Hp, 8), shifts, consts, W, H, out)

    (out, again, listed), _ = contract(pkg, run, prime)
    assert np.array_equal(again, out)
    assert np.array_equal(listed, out.reshape(-1, H, W, 3))
    _check_views(out.reshape(-1, H, W, 3), pano, flat, W, H, fov)


# ------------------------------------------------------------------------------------------
# projection routes
# ------------------------------------------------------------------------------------------
def test_quarter_turn_groups_fold_between_poisons(pkg):
    """Row-segment kernel (W % 8 == 0): the second render of a quarter-turn group folds the panorama; the slot is
    poisoned between the two renders."""
    Wp, Hp, W, H, fov = 1024, 256, 64, 48, 100
    pano = synth.noise(Wp, Hp, 9)
    views = [(y, pt) for pt in (0, 60, 180) for y in (0, 90, 180, 270)]
    shifts, consts = _flat(pkg, Wp, W, fov, views)

    def run(p):
        p.upload(0, pano)
        first = p.project_list(0, shifts, consts, W, H)
        p.sync(0)
        p.poison(0, 0x3C)
        second = p.project_list(0, shifts, consts, W, H)
        p.sync(0)
        p.poison(0, 0xC3)
        third = p.project_list(0, shifts, consts, W, H)
        p.sync(0)
        return [first, second, third]

    def prime(p):
        big = synth.noise(Wp + 256, Hp + 64, 1)
        p.upload(0, big)
        s2, c2 = _flat(pkg, Wp + 256, W, fov, [(y, 45) for y in (0, 90, 180, 270)])
        for _ in range(2):
            p.project_list(0, s2, c2, W, H)

    (a, b, c), _ = contract(pkg, run, prime)
    assert np.array_equal(a, b) and np.array_equal(a, c)
    _check_views(a, pano, views, W, H, fov)


@pytest.mark.parametrize("W", [64, 60, 58])
def test_table_groups_and_frac_kernel(pkg, W):
    """Fractional yaws through a view list: row-segment TAB groups (W % 8 == 0) or project_frac_kernel (W % 8 != 0,
    byte stores for W % 4 != 0), mixed with integer rolls."""
    Wp, Hp, H, fov = 1000, 200, 40, 100
    pano = synth.noise(Wp, Hp, 10)
    yaws = [12.5, 0, 201.3, 90, 12.5]
    pitches = [0, 90, 150, 90, 90]
    tables = [pkg.yaw_table(Wp, y) for y in yaws]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]

    def run(p):
        p.upload(0, pano)
        out = p.project_list_tables(0, tables, consts, W, H)
        p.sync(0)
        return out

    def prime(p):
        p.upload(0, synth.noise(Wp + 48, Hp + 24, 2))
        t = [pkg.yaw_table(Wp + 48, y) for y in (7.7, 99.1)]
        p.project_list_tables(0, t, [pkg.pitch_constants(W + 4, fov, 45)] * 2, W + 4, H + 9)

    out, _ = contract(pkg, run, prime)
    for i, (y, pt) in enumerate(zip(yaws, pitches)):
        _check_view(out[i], fp.project_view_single_pass(pano, y, pt, W, H, fov), y, pt)


ROUTES = [  # (label, options, W): every generic kernel variant of launch_project
    ("mirror1 s1", dict(MIRROR=1), 64),
    ("mirror1 s0", dict(MIRROR=1, SAMPLER=0), 64),
    ("mirror0 s1 ny1", dict(MIRROR=0, YAWS_PER_THREAD=1), 64),
    ("mirror0 s1 ny2", dict(MIRROR=0, YAWS_PER_THREAD=2), 64),
    ("mirror0 s0 ny3", dict(MIRROR=0, SAMPLER=0, YAWS_PER_THREAD=3), 64),
    ("mirror0 s0 ny4 warp8", dict(MIRROR=0, SAMPLER=0, WARP_W=8), 64),
    ("mirror0 s1 warp8", dict(MIRROR=0, WARP_W=8), 64),
    ("byte stores s1", dict(), 62),
    ("byte stores s0", dict(SAMPLER=0), 61),
]


@pytest.mark.parametrize("label,opts,W", ROUTES, ids=[r[0] for r in ROUTES])
def test_generic_routes(pkg, label, opts, W):
    L = pkg._lib
    Wp, Hp, H, fov = 1024, 256, 40, 110
    pano = synth.noise(Wp, Hp, 11)
    yaws, pitches = [0, 90, 180, 270, 45], [0, 75, 180]
    shifts = [pkg.yaw_table(Wp, y)[2] for y in yaws]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]
    options = [(getattr(L, "OPT_" + k), v) for k, v in opts.items()]

    def run(p):
        p.upload(0, pano)
        out = p.project(0, shifts, consts, W, H)
        p.sync(0)
        return out

    def prime(p):
        p.upload(0, synth.noise(Wp + 64, Hp + 32, 3))
        p.project(0, [3, 77], [pkg.pitch_constants(W + 8, fov, 20)], W + 8, H + 5)

    out, _ = contract(pkg, run, prime, options)
    for k, y in enumerate(yaws):
        for j, pt in enumerate(pitches):
            _check_view(out[k, j], fp.project_view_single_pass(pano, y, pt, W, H, fov), label, y, pt)


@pytest.mark.parametrize("nb", [2, 4])
def test_images_per_launch(pkg, nb):
    """p2p_project_batch with 2 and 4 resident panoramas per launch, into device outputs."""
    torch = _torch()
    L = pkg._lib
    Wp, Hp, W, H, fov = 1024, 128, 64, 40, 100
    panos = [synth.noise(Wp, Hp, 20 + i) for i in range(nb)]
    yaws, pitches = [0, 90, 180], [0, 90]
    shifts = [pkg.yaw_table(Wp, y)[2] for y in yaws]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]
    n_bytes = len(yaws) * len(pitches) * H * W * 3

    def run(p):
        outs = [torch.empty(n_bytes, dtype=torch.uint8, device="cuda:0") for _ in range(nb)]
        for i in range(nb):
            p.upload(i, panos[i])
        p.sync()
        p.batch_call(list(range(nb)), shifts, consts, W, H, [o.data_ptr() for o in outs])()
        p.sync()
        return [o.cpu().numpy().reshape(len(yaws), len(pitches), H, W, 3) for o in outs]

    def prime(p):
        for i in range(nb):
            p.upload(i, synth.noise(Wp + 128, Hp + 64, i))

    got, _ = contract(pkg, run, prime, [(L.OPT_IMAGES_PER_LAUNCH, nb), (L.OPT_MIRROR, 0)], n_slots=nb)
    for i in range(nb):
        for k, y in enumerate(yaws):
            for j, pt in enumerate(pitches):
                _check_view(got[i][k, j], fp.project_view_single_pass(panos[i], y, pt, W, H, fov), i, y, pt)


@pytest.mark.parametrize("seam", [0, 1])
def test_exact_mode(pkg, seam):
    """The exact-bilinear mode reads the linear panorama, wrap column included when the seam is interpolated."""
    pytest.importorskip("scipy")
    L = pkg._lib
    Wp, Hp, W, H, fov = 1024, 256, 60, 40, 100
    pano = synth.smooth(Wp, Hp, 12)
    yaws, pitches = [0, 90, 270], [0, 90, 180]
    shifts = [pkg.yaw_table(Wp, y)[2] for y in yaws]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]

    def run(p):
        p.upload(0, pano)
        out = p.project(0, shifts, consts, W, H)
        p.sync(0)
        return out

    def prime(p):
        p.upload(0, synth.noise(Wp + 64, Hp + 64, 4))
        p.project(0, [1], [pkg.pitch_constants(W, fov, 45)], W, H)

    out, _ = contract(pkg, run, prime, [(L.OPT_INTERP, 1), (L.OPT_SEAM_WRAP, seam)])
    for k, y in enumerate(yaws):
        for j, pt in enumerate(pitches):
            want = eb.project_view_exact(pano, y, pt, W, H, fov, seam_wrap=bool(seam))
            assert np.abs(out[k, j].astype(np.int16) - want.astype(np.int16)).max() <= 1, (y, pt)


BANDS = [  # (label, options, W): the row-segment kernel and the geometries it does not take
    ("rows kernel", {}, 64),
    ("W % 8", {}, 60),
    ("LDG sampler", dict(SAMPLER=0), 64),
    ("mirror 1", dict(MIRROR=1), 64),
    ("exact mode", dict(INTERP=1), 64),
    ("table views W % 8", {}, 60),
]


@pytest.mark.parametrize("label,opts,W", BANDS, ids=[b[0] for b in BANDS])
@pytest.mark.parametrize("on_device", [0, 1])
def test_row_bands_leave_other_rows_alone(pkg, label, opts, W, on_device):
    """p2p_project_view_list_tables writes rows row_begin .. row_end - 1 of every view and nothing else, into host and
    device outputs alike (p2p.h): the outputs are filled with a sentinel first, pole pitches included."""
    torch = _torch() if on_device else None
    L = pkg._lib
    Wp, Hp, H, fov = 1024, 256, 41, 100
    pano = synth.noise(Wp, Hp, 13)
    yaws = [0, 90, 180] if not label.startswith("table") else [0, 33.3, 180]
    pitches = [0, 90, 180]
    tables = [pkg.yaw_table(Wp, y) for y in yaws]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]
    bands = [(0, 13), (13, 30), (30, H), (7, 8)]
    options = [(getattr(L, "OPT_" + k), v) for k, v in opts.items()]
    n = len(yaws)

    def run(p):
        p.upload(0, pano)
        got = []
        for r0, r1 in bands:
            if on_device:
                out = torch.full((n * H * W * 3,), 0x77, dtype=torch.uint8, device="cuda:0")
                torch.cuda.synchronize()
                p.project_list_tables(0, tables, consts, W, H, rows=(r0, r1), out_device_ptr=out.data_ptr())
                p.sync(0)
                got.append(out.cpu().numpy().reshape(n, H, W, 3))
            else:
                out = np.full((n, H, W, 3), 0x77, np.uint8)
                p.project_list_tables(0, tables, consts, W, H, rows=(r0, r1), out=out)
                p.sync(0)
                got.append(out)
        return got

    def prime(p):
        p.upload(0, synth.noise(Wp, Hp, 14))
        p.project_list_tables(0, tables, consts, W, H)

    got, _ = contract(pkg, run, prime, options)
    for i, (y, pt) in enumerate(zip(yaws, pitches)):
        if opts.get("INTERP"):
            want = eb.project_view_exact(pano, y, pt, W, H, fov)
        else:
            want = fp.project_view_single_pass(pano, y, pt, W, H, fov)
        for (r0, r1), out in zip(bands, got):
            assert (out[i, :r0] == 0x77).all() and (out[i, r1:] == 0x77).all(), (label, (r0, r1), "rows outside the band")
            if opts.get("INTERP"):
                assert np.abs(out[i, r0:r1].astype(np.int16) - want[r0:r1].astype(np.int16)).max() <= 1
            else:
                _check_view(out[i, r0:r1], want[r0:r1], label, y, pt, r0, r1)


# ------------------------------------------------------------------------------------------
# encoders
# ------------------------------------------------------------------------------------------
def _sat(n, H, W, seed):
    return (np.random.default_rng(seed).integers(0, 2, (n, H, W, 3)) * 255).astype(np.uint8)


@pytest.mark.parametrize("q", [1, 95, 100])
def test_jpeg_encoder(pkg, q):
    """p2p_encode_jpeg at 1 x 1, 17 x 33 and W % 4 != 0, from host memory and from device memory 1..3 bytes past an
    aligned address, after a batch of 8 saturated-noise images: cv2.imencode's bytes."""
    torch = _torch()
    imgs = [synth.noise(1, 1, 1)[None], synth.noise(17, 33, 2)[None], np.stack([synth.noise(30, 21, 3 + i) for i in range(3)])]

    def run(p):
        got = []
        for im in imgs:
            got.append(p.encode_jpeg(im, q, slot=0))
            n, H, W, _ = im.shape
            for off in (1, 2, 3):
                d = torch.zeros(im.size + 8, dtype=torch.uint8, device="cuda:0")
                d[off:off + im.size].copy_(torch.from_numpy(im.reshape(-1)))
                torch.cuda.synchronize()
                got.append(p._files_call(p.lib.p2p_encode_jpeg, 0, (C.c_void_p(d.data_ptr() + off), 1, n, W, H, q), n,
                                         W * H * 3 + 4096))
        return got

    def prime(p):
        p.encode_jpeg(_sat(8, 77, 93, 5), q, slot=0)

    got, _ = contract(pkg, run, prime)
    for k, im in enumerate(imgs):
        want = [cv2.imencode(".jpg", x, [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes() for x in im]
        for r in got[4 * k:4 * k + 4]:
            assert r == want


def _png_corpus_subset():
    import png_streams as S
    seen, out = set(), []
    for family, name, W, F in S.corpus():
        if family not in seen:
            seen.add(family)
            out.append((f"{family}/{name}", S.image_from_filtered(F, W)))
    return out


def test_png_encoder(pkg):
    """p2p_encode_png on one designed stream of every family, stored-block sizes (noise) and small images, after a
    large noise image: cv2.imencode's bytes."""
    cases = _png_corpus_subset()
    cases += [("noise 200x150", synth.noise(200, 150, 1)), ("noise 1x1", synth.noise(1, 1, 2)),
              ("noise 1x97", synth.noise(1, 97, 3)), ("smooth 75x33", synth.smooth(75, 33, 4))]

    def run(p):
        return [p.encode_png(img, slot=0) for _, img in cases]

    def prime(p):
        p.encode_png(synth.noise(1500, 900, 5), slot=0)

    got, _ = contract(pkg, run, prime)
    for (label, img), files in zip(cases, got):
        assert files[0] == cv2.imencode(".png", img)[1].tobytes(), label


# ------------------------------------------------------------------------------------------
# JPEG decoder
# ------------------------------------------------------------------------------------------
SAMPLING = {"420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444}


def _jpeg(img, sname, q=90, rst=0, extra=()):
    params = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, *extra]
    if sname == "gray":
        img = np.ascontiguousarray(img[..., 1])
    else:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
    return cv2.imencode(".jpg", img, params)[1].tobytes()


def _imdecode(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


def _decode_run(pkg, files, W=40, H=24, fov=120):
    """run(p): every file through p2p_decode_jpeg / _png, then through the upload entry and views read with the LDG
    sampler (the linear panorama with its wrap column) across the seam and at both poles."""
    L = pkg._lib

    def run(p):
        got = []
        for data in files:
            got.append(p.decode_encoded(data, slot=0))
            Wp, Hp = p.upload_encoded(0, data)
            views = [(0, 0), (0, 180)] + [(y, 90) for y, _ in _rolls(pkg, Wp)[:4]]
            shifts, consts = _flat(pkg, Wp, W, fov, views)
            p.set_option(L.OPT_SAMPLER, 0)
            got.append(p.project_list(0, shifts, consts, W, H))
            p.sync(0)
            p.set_option(L.OPT_SAMPLER, 1)
            got.append(p.download_pano(0, Wp, Hp))
        return got

    def check(got):
        for k, data in enumerate(files):
            ref = _imdecode(data)
            assert np.array_equal(got[3 * k], ref), k
            assert np.array_equal(got[3 * k + 2], ref), k
            Hp, Wp = ref.shape[:2]
            views = [(0, 0), (0, 180)] + [(y, 90) for y, _ in _rolls(pkg, Wp)[:4]]
            _check_views(got[3 * k + 1], ref, views, W, H, fov)

    return run, check


def _textured(w, h, seed):
    return cv2.GaussianBlur(synth.noise(w, h, seed), (0, 0), 1.5)


@pytest.mark.parametrize("huffman", [1, 0])
@pytest.mark.parametrize("rst", [0, 3])
@pytest.mark.parametrize("sname", ["420", "422", "444", "gray"])
def test_jpeg_decoder_sampling(pkg, sname, rst, huffman):
    """Odd sizes of every sampling, with and without restart intervals, device Huffman stage on and off; the slot first
    decoded a larger file of the same sampling."""
    L = pkg._lib
    files = [_jpeg(_textured(w, h, w), sname, rst=rst) for w, h in ((97, 61), (33, 17), (256, 130))]
    run, check = _decode_run(pkg, files)

    def prime(p):
        big = _jpeg(_textured(701, 333, 1), sname, q=97, rst=rst)
        p.upload_jpeg(0, big)
        p.decode_jpeg(big, slot=0)

    got, delta = contract(pkg, run, prime, [(L.OPT_GPU_HUFFMAN, huffman)])
    check(got)
    assert delta[0] == (2 * len(files) if huffman else 0), "a baseline file was declined by the device Huffman stage"


def test_jpeg_decoder_writer_tables_and_progressive(pkg):
    """Optimised tables, DC tables longer than the Annex K ones, every table policy through one file each, and two
    progressive scripts."""
    L = pkg._lib
    lib = L.load()
    base = _jpeg(_textured(120, 72, 3), "420", q=92)
    files = [_jpeg(_textured(120, 72, 3), "420", q=92, extra=(cv2.IMWRITE_JPEG_OPTIMIZE, 1))]
    for label, kw in jw.variants():
        if label in ("optimal", "all_len(16)", "dc_dup rst 1", "eob_alias rst 3", "per component"):
            files.append(jw.write(base, lib=lib, **kw))
    baseline = len(files)
    for script in ("simple", "spectral_only"):
        files.append(jw.write_progressive(base, script, source=jw.read_coefficients(base, lib)))
    run, check = _decode_run(pkg, files)

    def prime(p):
        big = _jpeg(_textured(640, 320, 4), "444", q=98, rst=5)
        p.upload_jpeg(0, big)

    got, delta = contract(pkg, run, prime)
    check(got)
    assert delta[0] == 2 * baseline, "a baseline file was declined by the device Huffman stage"


def test_jpeg_decoder_long_then_short_scan(pkg):
    """A short scan behind a long one on the same slot: the tail of the destuffed stream and the subsequence arrays
    still hold the long scan's data."""
    L = pkg._lib
    files = [_jpeg(_textured(64, 40, 5), "420", q=75), _jpeg(synth.noise(48, 16, 6), "444", q=95)]
    run, check = _decode_run(pkg, files)

    def prime(p):
        for q in (100, 95):
            big = _jpeg(synth.noise(900, 450, 7), "444", q=q)
            p.decode_jpeg(big, slot=0)

    got, delta = contract(pkg, run, prime)
    check(got)
    assert delta[0] == 2 * len(files)


def test_jpeg_decoder_more_rounds_than_queued(pkg):
    """Files whose Huffman stage needs more synchronisation rounds than the default mode queues before its verdict: the
    stage continues with host-checked rounds, and their block-count check must not see the verdict of the queued one."""
    img = synth.smooth(1000, 333, 7)
    rng = np.random.default_rng(7)
    textured = np.clip(img.astype(np.int16) + rng.integers(-12, 13, img.shape, dtype=np.int16), 0, 255).astype(np.uint8)
    files = [cv2.imencode(".jpg", textured, [cv2.IMWRITE_JPEG_LUMA_QUALITY, lq, cv2.IMWRITE_JPEG_CHROMA_QUALITY, cq,
                                             cv2.IMWRITE_JPEG_OPTIMIZE, opt])[1].tobytes()
             for lq, cq, opt in ((95, 30, 0), (20, 100, 1), (100, 60, 1))]
    files.append(jw.write(_jpeg(img, "444", q=92), tables="all_len(16)", lib=pkg._lib.load()))
    run, check = _decode_run(pkg, files)

    def prime(p):
        p.upload_jpeg(0, _jpeg(synth.noise(1200, 500, 8), "420", q=95))

    got, delta = contract(pkg, run, prime)
    check(got)
    assert delta[0] == 2 * len(files), "a baseline file was declined by the device Huffman stage"


def _damaged_jpeg(seed, restart):
    """a file whose scan is cut short in the middle (EOI follows)"""
    data = _jpeg(_textured(320, 160, seed), "420", q=90, rst=restart)
    mid = (data.find(b"\xff\xda") + len(data)) // 2
    return data[:mid] + b"\xff\xd9"


def test_jpeg_decoder_valid_file_after_a_damaged_one(pkg):
    """A damaged file (declined) and then a valid one on the same slot: the valid file must be decoded on the device,
    not declined because a flag of the damaged one survived."""
    L = pkg._lib
    files = [_jpeg(_textured(97, 61, 8), "420", q=90), _jpeg(_textured(64, 48, 9), "422", q=90, rst=2)]
    run, check = _decode_run(pkg, files)
    bad = [_damaged_jpeg(s, rst) for s in range(2) for rst in (0, 4)]

    def prime(p):
        for b in bad:
            try:
                p.upload_jpeg(0, b)
            except pkg.P2PError as e:
                assert e.code == -6
            try:
                p.decode_jpeg(b, slot=0)
            except pkg.P2PError as e:
                assert e.code == -6

    got, delta = contract(pkg, run, prime, prime_fresh=True)   # the fresh contexts meet the damaged files on poisoned flags
    check(got)
    assert delta[0] == 2 * len(files), "a valid file behind a damaged one was declined by the device Huffman stage"


# ------------------------------------------------------------------------------------------
# PNG decoder
# ------------------------------------------------------------------------------------------
def test_png_decoder_colour_types(pkg):
    """Every 8-bit colour type at odd sizes, after a larger file on the same slot."""
    img = synth.noise(97, 61, 1)
    smooth = synth.smooth(64, 33, 2)
    files = [cv2.imencode(".png", img[..., 1])[1].tobytes(),                               # gray
             cv2.imencode(".png", img)[1].tobytes(),                                       # RGB
             cv2.imencode(".png", np.dstack([smooth, smooth[..., :1]]))[1].tobytes(),      # RGBA
             cv2.imencode(".png", smooth)[1].tobytes()]
    from png_formats import make
    files.append(make(4, 8, 0, 41, 23, 0))                                                  # gray + alpha
    run, check = _decode_run(pkg, files)

    def prime(p):
        big = cv2.imencode(".png", synth.noise(1200, 600, 3))[1].tobytes()
        p.upload_png(0, big)
        p.decode_png(big, slot=0)

    got, delta = contract(pkg, run, prime)
    check(got)


def test_png_decoder_formats(pkg):
    """P2P_OPT_PNG_FORMATS = 1: palette, 16-bit, sub-byte gray and Adam7 files."""
    L = pkg._lib
    picks = [(3, 8, 0), (3, 2, 1), (2, 16, 0), (6, 16, 1), (0, 1, 0), (0, 4, 1), (2, 8, 1)]
    files = [png_formats.make(ct, d, lace, 37, 19, k) for k, (ct, d, lace) in enumerate(picks)]
    run, check = _decode_run(pkg, files)

    def prime(p):
        p.upload_png(0, png_formats.make(6, 16, 1, 301, 157, 3))

    got, delta = contract(pkg, run, prime, [(L.OPT_PNG_FORMATS, 1)])
    check(got)


def test_png_decoder_designed_streams(pkg):
    """Designed deflate streams whose matches reach back across blocks, then a declined file, then valid ones."""
    designs = [d for fam in ("history", "layout") for d in D.corpus()[fam] if d.expect == "decode"][:8]
    decline = next(d for d in D.corpus()["invalid"])
    files = [d.png for d in designs]
    run, check = _decode_run(pkg, files)

    def prime(p):
        p.upload_png(0, cv2.imencode(".png", synth.noise(800, 500, 4))[1].tobytes())
        with pytest.raises(pkg.P2PError):
            p.upload_png(0, decline.png)

    got, delta = contract(pkg, run, prime)
    check(got)


# ------------------------------------------------------------------------------------------
# files flows
# ------------------------------------------------------------------------------------------
def _ref_views(pkg, pano, yaws, pitches, W, H, fov):
    """[yaw][pitch] views: the oracle's where this host's NumPy matches the reference bit for bit, else a plain render
    of a fresh context (the projection itself is pinned to the oracle by the tests above)."""
    if STRICT:
        return [[fp.project_view_single_pass(pano, y, pt, W, H, fov) for pt in pitches] for y in yaws]
    p = pkg.Projector(0, 1)
    try:
        out = p.project_image(pano, yaws, pitches, W, H, fov)
    finally:
        p.close()
    return [[out[k, j] for j in range(len(pitches))] for k in range(len(yaws))]


def _files_flows(pkg, Wp, Hp, W, H, fov, data, q=95):
    """run(p): the files entries from host rows and from a slot the device decoder filled."""
    ref_pano = _imdecode(data)
    rolls = [(y, s) for y, s in _rolls(pkg, Wp, (0, 90, 180, 270))]
    pitches = [0, 90, 180]
    frac = [10.5, 200.25]
    shifts = [s for _, s in rolls]
    consts = [pkg.pitch_constants(W, fov, pt) for pt in pitches]
    lview = [(y, pt) for y in [rolls[0][0], *frac] for pt in (90, 30)]
    ltables = [pkg.yaw_table(Wp, y) for y, _ in lview]
    lconsts = [pkg.pitch_constants(W, fov, pt) for _, pt in lview]

    def run(p):
        got = []
        got.append(p.process_image_jpeg(0, ref_pano, shifts, consts, W, H, q))
        got.append(p.process_image_png(0, ref_pano, shifts, consts, W, H, want_pixels=False)[0])
        got.append(p.process_view_list_jpeg(0, ref_pano, ltables, lconsts, W, H, q))
        got.append(p.process_view_list_png(0, ref_pano, ltables, lconsts, W, H)[0])
        for entry in range(4):
            p.upload_encoded(0, data)
            if entry == 0:
                got.append(p.project_jpeg(0, shifts, consts, W, H, q))
            elif entry == 1:
                got.append(p.process_image_png(0, None, shifts, consts, W, H, want_pixels=False)[0])
            elif entry == 2:
                got.append(p.process_view_list_jpeg(0, None, ltables, lconsts, W, H, q))
            else:
                got.append(p.process_view_list_png(0, None, ltables, lconsts, W, H)[0])
        return got

    def check(got):
        prod = _ref_views(pkg, ref_pano, [y for y, _ in rolls], pitches, W, H, fov)
        prod = [v for row in prod for v in row]
        lst = [_ref_views(pkg, ref_pano, [y], [pt], W, H, fov)[0][0] for y, pt in lview]
        jpg = lambda vs: [cv2.imencode(".jpg", v, [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes() for v in vs]
        png = lambda vs: [cv2.imencode(".png", v)[1].tobytes() for v in vs]
        want = [jpg(prod), png(prod), jpg(lst), png(lst)]
        for k in range(4):
            assert got[k] == want[k], ("host rows", k)
            assert got[4 + k] == want[k], ("decoded slot", k)

    return run, check


@pytest.mark.parametrize("fmt", ["jpg", "png"])
def test_files_flows(pkg, fmt):
    Wp, Hp, W, H, fov = 1024, 512, 64, 40, 100
    img = _textured(Wp, Hp, 15)
    data = cv2.imencode("." + fmt, img, [cv2.IMWRITE_JPEG_QUALITY, 93] if fmt == "jpg" else [])[1].tobytes()
    run, check = _files_flows(pkg, Wp, Hp, W, H, fov, data)

    def prime(p):
        big = _textured(1536, 768, 16)
        p.upload_encoded(0, cv2.imencode("." + fmt, big)[1].tobytes())
        p.process_image_jpeg(0, big, [0, 384], [pkg.pitch_constants(96, fov, 45)], 96, 80)
        p.process_image_png(0, big, [0, 384], [pkg.pitch_constants(96, fov, 45)], 96, 80)

    got, delta = contract(pkg, run, prime)
    check(got)
    if fmt == "jpg":
        assert delta[0] == 4, "the device Huffman stage declined the panorama"


@pytest.mark.parametrize("fmt", ["jpg", "png"])
def test_files_flows_8k(pkg, fmt):
    """One 8192 x 4096 panorama through the files flows."""
    Wp, Hp, W, H, fov = 8192, 4096, 256, 160, 90
    img = _textured(Wp, Hp, 17)
    data = cv2.imencode("." + fmt, img, [cv2.IMWRITE_JPEG_QUALITY, 90] if fmt == "jpg" else [])[1].tobytes()
    run, check = _files_flows(pkg, Wp, Hp, W, H, fov, data, q=90)

    def prime(p):
        p.upload_encoded(0, cv2.imencode("." + fmt, synth.noise(4096, 2048, 18))[1].tobytes())

    got, delta = contract(pkg, run, prime)
    check(got)
