"""GPU tests of the paired row-segment launches: p2p_project_batch renders the quarter-turn groups of two resident
panoramas on the same stream in one launch, the coordinates of every pixel pair shared between the two images, once both
panoramas read their yaw-folded planes (from their second quarter-turn render on); every other group is launched per
panorama.  Every batch is compared byte for byte with each slot rendered on its own (``project_list``: one slot per
launch) and, where host NumPy evaluates arccos / arctan2 like the kernel, with ``oracle.fixedpoint``.  The launch counter
shows which images shared a launch.
"""
import contextlib

import numpy as np
import pytest

from oracle import fixedpoint as fp
from oracle import ref_port, svml_model, synth

pytestmark = pytest.mark.gpu

W, H, FOV = 96, 64, 90
PITCHES = [30, 60, 90]
QUARTER = [0, 256, 512, 768]       # quarter turns of a 1024-wide panorama: the folded planes from the second render on
NEAR = [0, 256, 512, 772]          # 0 / 90 / 180 / ~271 degrees: the RGBA texture


@pytest.fixture(scope="module")
def proj8(pkg):
    p = pkg.Projector(0, n_slots=8)
    yield p
    p.close()


@contextlib.contextmanager
def _streams(proj, slots, n_streams):
    """slots[i] launches on the stream of slots[i % n_streams] for the duration; every slot gets its own stream back."""
    own = {s: proj.get_stream(s) for s in slots}
    try:
        for i, s in enumerate(slots):
            proj.set_stream(s, own[slots[i % n_streams]])
        yield
    finally:
        proj.sync(-1)
        for s in slots:
            proj.set_stream(s, own[s])


def _batch(pkg, proj, slots, shifts, pitches, W=W, H=H):
    """One p2p_project_batch call with device outputs -> [image][yaw][pitch][H][W][3] and the launches it took."""
    torch = pytest.importorskip("torch")
    consts = [pkg.pitch_constants(W, FOV, p) for p in pitches]
    d = torch.zeros((len(slots), len(shifts), len(pitches), H, W, 3), dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    n0 = proj.launches
    proj.batch_call(slots, shifts, consts, W, H, [d[i].data_ptr() for i in range(len(slots))], on_device=True)()
    proj.sync(-1)
    return d.cpu().numpy(), proj.launches - n0


def _solo(pkg, proj, s, shifts, pitches, W=W, H=H):
    """The batch's views of one slot as one flat view list of its own: view (yaw k, pitch j) at k * n_pitch + j."""
    consts = [pkg.pitch_constants(W, FOV, p) for p in pitches]
    out = np.zeros((len(shifts) * len(pitches), H, W, 3), np.uint8)
    proj.project_list(s, [sh for sh in shifts for _ in pitches], [c for _ in shifts for c in consts], W, H, out=out)
    proj.sync(s)
    return out.reshape(len(shifts), len(pitches), H, W, 3)


def _check_oracle(pano, shifts, pitches, got, W=W, H=H):
    if not svml_model.host_numpy_uses_svml():
        return   # the reference maps differ from the kernel's in the last ulp on this host; the per-slot check still holds
    Hp, Wp, _ = pano.shape
    for j, p in enumerate(pitches):
        U, V = ref_port.pitch_mapping(W, H, FOV, p, Wp, Hp)
        for k, sh in enumerate(shifts):
            assert np.array_equal(got[k, j], fp.sample_view(pano, U, V, yaw_shift=sh)), (Wp, sh, p)


def _fill(proj, slots, sizes, seed):
    panos = []
    for i, s in enumerate(slots):
        Wp, Hp = sizes[i % len(sizes)]
        panos.append(synth.noise(Wp, Hp, seed + i))
        proj.upload(s, panos[-1])
    proj.sync(-1)
    return panos


def _render_twice(pkg, proj, slots, shifts, pitches, W=W, H=H):
    """The batch rendered twice (a quarter-turn list: RGBA texture first; the second render folds the panoramas in the
    paired launch and reads the folded planes), then each image compared with its own single-slot render.  The single-slot
    renders come last: they would build the slots' folded planes themselves."""
    got, launches = [], []
    for _ in range(2):
        g, n = _batch(pkg, proj, slots, shifts, pitches, W, H)
        got.append(g)
        launches.append(n)
    assert np.array_equal(got[0], got[1])
    for i, s in enumerate(slots):
        assert np.array_equal(got[1][i], _solo(pkg, proj, s, shifts, pitches, W, H)), (i, s)
    return got[1], launches


@contextlib.contextmanager
def _seg_chunks(pkg, proj, value):
    """P2P_OPT_SEG_CHUNKS = value (None: the default) for the duration."""
    key = pkg._lib.OPT_SEG_CHUNKS
    old = proj.get_option(key)
    try:
        if value is not None:
            proj.set_option(key, value)
        yield
    finally:
        proj.set_option(key, old)


# (output width, chunks per warp segment): W = 96 at the default 4 chunks is one segment per row; W = 320 (6 chunks) and
# one chunk per segment put segment ends inside the row, where the per-image byte stores of the segment ends run
GEOMETRIES = [(96, None), (320, None), (96, 1)]


@pytest.mark.parametrize("n", [2, 3, 5])
@pytest.mark.parametrize("shifts", [QUARTER, NEAR], ids=["quarter", "near_quarter"])
@pytest.mark.parametrize("w, seg", GEOMETRIES, ids=["w96", "w320", "w96_seg1"])
def test_same_stream_batch_equals_single_slots(pkg, proj8, n, shifts, w, seg):
    """Once the panoramas read their folded planes, 2k images on one stream take k launches; an odd batch leaves its last
    image a launch of its own.  The first render (RGBA texture) and the near-quarter yaws take one launch per image."""
    slots = list(range(n))
    with _streams(proj8, slots, 1), _seg_chunks(pkg, proj8, seg):
        panos = _fill(proj8, slots, [(1024, 512)], 100 * n)
        got, launches = _render_twice(pkg, proj8, slots, shifts, PITCHES, w, H)
    assert launches == ([n, (n + 1) // 2] if shifts == QUARTER else [n, n])
    _check_oracle(panos[0], shifts, PITCHES, got[0], w, H)
    _check_oracle(panos[1], shifts, PITCHES, got[1], w, H)


def test_streams_pair_only_their_own_images(pkg, proj8):
    """Slot i on stream i % 2 (bench.py's layout): the pairs are (0, 2), (1, 3), (4, 6), (5, 7); two images on different
    streams never share a launch."""
    slots = list(range(8))
    with _streams(proj8, slots, 2):
        _fill(proj8, slots, [(1024, 512)], 7)
        _, launches = _render_twice(pkg, proj8, slots, QUARTER, PITCHES)
        assert launches == [8, 4]
        _, launches = _render_twice(pkg, proj8, slots[:2], QUARTER, PITCHES)
        assert launches == [2, 2]
    with _streams(proj8, slots, 8):   # every slot on its own stream
        _, launches = _render_twice(pkg, proj8, slots[:4], QUARTER, PITCHES)
        assert launches == [4, 4]


def test_mixed_panorama_sizes(pkg, proj8):
    """Only panoramas of one size pair: 1024- and 1000-wide images alternate in the batch, the pairs skip over each other.
    The rolls are quarter turns of the 1000-wide panoramas only."""
    slots = list(range(5))
    shifts = [0, 250, 500, 750]
    with _streams(proj8, slots, 1):
        panos = _fill(proj8, slots, [(1024, 512), (1000, 500)], 21)
        got, launches = _render_twice(pkg, proj8, slots, shifts, PITCHES)
    assert launches == [5, 4]   # then (0, 2) one launch each (not quarter turns of 1024), (1, 3) one, 4 one
    _check_oracle(panos[1], shifts, PITCHES, got[1])
    _check_oracle(panos[4], shifts, PITCHES, got[4])


@pytest.mark.parametrize("shifts, launches_per_pair", [
    ([0, 256, 512, 768, 100], 3),     # the quarter sets of the pair in one launch, the one-yaw groups in one per image
    ([0, 256, 772], 2),               # three yaws
    ([384, 0, 128, 512, 256, 640, 896, 768], 1),   # two quarter sets, permuted
    ([5], 2),
])
def test_mixed_yaw_lists(pkg, proj8, shifts, launches_per_pair):
    slots = list(range(4))
    with _streams(proj8, slots, 1):
        panos = _fill(proj8, slots, [(1024, 512)], 31)
        got, launches = _render_twice(pkg, proj8, slots, shifts, [0, 45, 90, 180])
    assert launches == [4, 2 * launches_per_pair]
    _check_oracle(panos[3], shifts, [0, 45, 90, 180], got[3])


def test_minimax_trig(pkg, proj8):
    L = pkg._lib
    slots = list(range(3))
    trig = proj8.get_option(L.OPT_TRIG)
    try:
        proj8.set_option(L.OPT_TRIG, 1)
        with _streams(proj8, slots, 1):
            _fill(proj8, slots, [(1024, 512)], 41)
            _, launches = _render_twice(pkg, proj8, slots, QUARTER, [0, 30, 90, 180])
            _, launches_near = _render_twice(pkg, proj8, slots, NEAR, [0, 30, 90, 180])
    finally:
        proj8.set_option(L.OPT_TRIG, trig)
    assert launches == [3, 2] and launches_near == [3, 3]


@pytest.mark.parametrize("refill", [0, 1])
def test_one_slot_of_a_pair_folded_the_other_new(pkg, proj8, refill):
    """A pair reads the folded planes only when both images have rendered a quarter-turn list before: a slot that has
    folded and a fresh one first render on their own (RGBA texture), then the paired launch folds the fresh one.  Then
    one slot of the folded pair is refilled: its old planes are stale, and the paired launch that folds it again must
    serve the new panorama to that image (no single-slot render in between builds the planes for it)."""
    slots = [0, 1]
    with _streams(proj8, slots, 1):
        _fill(proj8, slots, [(1024, 512)], 51)
        for _ in range(2):   # slot 0 alone: its planes are built
            _batch(pkg, proj8, [0], QUARTER, PITCHES)
        _, launches = _render_twice(pkg, proj8, slots, QUARTER, PITCHES)
        assert launches == [2, 1]
        before = _batch(pkg, proj8, slots, QUARTER, PITCHES)[0]
        b = synth.smooth(1024, 512, 52)
        proj8.upload(refill, b)
        proj8.sync(refill)
        got, launches = _render_twice(pkg, proj8, slots, QUARTER, PITCHES)
        assert launches == [2, 1]
    assert np.array_equal(got[1 - refill], before[1 - refill])
    assert not np.array_equal(got[refill], before[refill])
    _check_oracle(b, QUARTER, PITCHES, got[refill])


def test_partial_slots(pkg, proj8):
    """Slots filled by p2p_process_image hold only the rows of their own views: they pair when they cover the batch's
    views; a slot that does not cover them is left out of the pairs and reports the error on its own launch."""
    L = pkg._lib
    slots = list(range(4))
    panos = [synth.noise(1024, 512, 61 + i) for i in slots]
    partial = proj8.get_option(L.OPT_PARTIAL_UPLOAD)
    try:
        proj8.set_option(L.OPT_PARTIAL_UPLOAD, 1)
        with _streams(proj8, slots, 1):
            for i, s in enumerate(slots):
                ps = [0] if i == 1 else PITCHES    # slot 1 holds the rows of the horizon only
                out = np.zeros((4, len(ps), H, W, 3), np.uint8)
                proj8.process_image(s, panos[i], QUARTER, [pkg.pitch_constants(W, FOV, p) for p in ps], W, H, out)
            proj8.sync(-1)
            got, launches = _render_twice(pkg, proj8, [0, 2, 3], QUARTER, PITCHES)
            assert launches == [2, 2]
            torch = pytest.importorskip("torch")
            consts = [pkg.pitch_constants(W, FOV, p) for p in PITCHES]
            d = torch.zeros((4, 4, 3, H, W, 3), dtype=torch.uint8, device="cuda:0")
            torch.cuda.synchronize()
            n0 = proj8.launches
            with pytest.raises(pkg.P2PError, match="partial panorama"):
                proj8.batch_call(slots, QUARTER, consts, W, H, [d[i].data_ptr() for i in slots])()
            proj8.sync(-1)
            assert proj8.launches - n0 == 1     # slot 0 with slot 2, then slot 1 fails before any launch
            assert np.array_equal(d[0].cpu().numpy(), got[0]) and np.array_equal(d[2].cpu().numpy(), got[1])
    finally:
        proj8.set_option(L.OPT_PARTIAL_UPLOAD, partial)
    _check_oracle(panos[3], QUARTER, PITCHES, got[2])


@pytest.mark.parametrize("byte", [0x00, 0xFF, 0xA5])
@pytest.mark.parametrize("w", [96, 320])
def test_poisoned_scratch(pkg, byte, w):
    """Fresh contexts whose every allocation is filled with `byte` first (P2P_OPT_POISON), then the slots poisoned
    (everything a slot does not hold): the pairs give the single-slot bytes, on the RGBA texture and the folded planes."""
    L = pkg._lib
    p = pkg.Projector(0, n_slots=4)
    try:
        p.set_option(L.OPT_POISON, byte)
        slots = list(range(4))
        with _streams(p, slots, 1):
            panos = _fill(p, slots, [(1024, 512)], 71)
            for s in slots:
                p.poison(s, byte)
            got, launches = _render_twice(pkg, p, slots, QUARTER, PITCHES, w, H)
            _, launches_near = _render_twice(pkg, p, slots, NEAR, PITCHES, w, H)
    finally:
        p.close()
    assert launches == [4, 2] and launches_near == [4, 4]
    _check_oracle(panos[1], QUARTER, PITCHES, got[1], w, H)
