"""Which engine calls the front end makes for each kind of input, yaw list and output format, checked without a GPU.

A stand-in projector records every engine call with the arguments that select the work (slot, resident panorama or host
pixels, the views in order, the band, ``copy`` / ``want_pixels``) and returns files that name the view they encode, so a
file that lands under the wrong name shows.  The stand-in runs through the public entry points (``process_single_image``
and ``_project``) on one device and split over two:

* a JPEG or PNG source the device decoder takes stays resident in the slot; a decline (-6 / -3 / -5) from
  ``upload_encoded`` sends the file to ``_decode_source(..., device_declined=True)`` and the host pixels on;
* integer yaw rolls go to the product entries, any fractional yaw to the view-list entries;
* a PNG file the device encoder left out (``None``) makes the front end read the pixels back and ``cv2.imwrite`` them;
* an encoder that runs out of memory or limits (-3 / -5) falls back to the pixel route;
* file names are the reference's (ref :275).

``project_list`` and ``project_list_tables`` reach the same C routine (``p2p_project_view_list`` passes NULL tables to
``p2p_project_view_list_tables``), so the stand-in records both as one ``view_list`` call.
"""
from __future__ import annotations

import contextlib
import importlib

import numpy as np
import pytest

W, H = 8, 16
PITCHES = [60, 90]
YAWS = {"integer": [0, 90, 180], "fractional": [0, 10, 90]}   # 10 degrees of a 64-column panorama is not a column roll
READBACK = 7                                                   # the value of every pixel the stand-in reads back


def _yaw_key(t):
    return int(t[2]) if t[2] is not None else ("table", int(np.sum(t[0])), int(np.sum(t[1])))


def _content(view):
    return repr(view).encode()


class FakeProjector:
    """The engine calls the front end makes, recorded; files name their view."""

    n_slots = 4

    def __init__(self, dev, decline=None, encoder_error=None, png_none=None):
        self.dev, self.decline, self.encoder_error, self.png_none = dev, decline, encoder_error, png_none
        self.log, self.free, self.taken = [], [3, 2, 1, 0], []

    @contextlib.contextmanager
    def slots(self, n=1):
        got = tuple(self.free.pop() for _ in range(n))
        self.taken.append(("take", got))
        try:
            yield got
        finally:
            self.free.extend(reversed(got))
            self.taken.append(("give", got))

    def _files(self, views, png):
        if self.encoder_error is not None:
            raise FakeProjector.P2PError(self.encoder_error, "encoder scratch does not fit")
        files = [None if png and v == self.png_none else _content(v) for v in views]
        return (files, None) if png else files

    def upload_encoded(self, slot, data):
        self.log.append(("upload_encoded", slot))
        if self.decline is not None:
            raise FakeProjector.P2PError(self.decline, "declined")
        return 64, 32

    def decode_encoded(self, data, slot=None):
        raise AssertionError("the front end decodes on the device only through upload_encoded")

    def project_any(self, slot, tables, consts, W_, H_, out=None):
        self.log.append(("project_any", slot, [(_yaw_key(t), c) for t in tables for c in consts]))
        return np.zeros((len(tables), len(consts), H_, W_, 3), np.uint8)

    def project_image(self, pano, yaw_angles, pitch_angles, W_, H_, fov_deg=90, out=None, consts=None, tables=None):
        assert isinstance(pano, np.ndarray)
        self.log.append(("project_image", [(_yaw_key(t), c) for t in tables for c in consts]))
        return np.zeros((len(yaw_angles), len(pitch_angles), H_, W_, 3), np.uint8)

    def project(self, slot, shifts, consts, W_, H_, out=None, out_device_ptr=None):
        self.log.append(("project", slot, [(int(s), c) for s in shifts for c in consts]))
        return np.full((len(shifts), len(consts), H_, W_, 3), READBACK, np.uint8)

    def _view_list(self, slot, keys, consts, W_, H_, rows, out):
        rows = (0, H_) if rows is None else (int(rows[0]), int(rows[1]))
        self.log.append(("view_list", slot, list(zip(keys, consts)), rows))
        if out is None:
            out = np.empty((len(keys), H_, W_, 3), np.uint8)
        out[:, rows[0]:rows[1]] = READBACK
        return out

    def project_list(self, slot, shifts, consts, W_, H_, rows=None, out=None, out_device_ptr=None):
        return self._view_list(slot, [int(s) for s in shifts], consts, W_, H_, rows, out)

    def project_list_tables(self, slot, tables, consts, W_, H_, rows=None, out=None, out_device_ptr=None):
        return self._view_list(slot, [_yaw_key(t) for t in tables], consts, W_, H_, rows, out)

    @staticmethod
    def _pano(pano):
        assert pano is None or isinstance(pano, np.ndarray)
        return "resident" if pano is None else "pixels"

    def project_jpeg(self, slot, shifts, consts, W_, H_, quality=95, copy=True):
        views = [(int(s), c) for s in shifts for c in consts]
        self.log.append(("project_jpeg", slot, views, copy))
        return self._files(views, False)

    def process_image_jpeg(self, slot, pano, shifts, consts, W_, H_, quality=95, copy=True):
        views = [(int(s), c) for s in shifts for c in consts]
        self.log.append(("process_image_jpeg", slot, self._pano(pano), views, copy))
        return self._files(views, False)

    def process_image_png(self, slot, pano, shifts, consts, W_, H_, want_pixels=True, copy=True):
        views = [(int(s), c) for s in shifts for c in consts]
        self.log.append(("process_image_png", slot, self._pano(pano), views, want_pixels, copy))
        return self._files(views, True)

    def process_view_list_jpeg(self, slot, pano, tables, consts, W_, H_, quality=95, copy=True):
        views = [(_yaw_key(t), c) for t, c in zip(tables, consts)]
        self.log.append(("process_view_list_jpeg", slot, self._pano(pano), views, copy))
        return self._files(views, False)

    def process_view_list_png(self, slot, pano, tables, consts, W_, H_, want_pixels=False, copy=True):
        views = [(_yaw_key(t), c) for t, c in zip(tables, consts)]
        self.log.append(("process_view_list_png", slot, self._pano(pano), views, want_pixels, copy))
        return self._files(views, True)

    def sync(self, slot=-1):
        self.log.append(("sync", slot))

    def upload_rows(self, slot, pano, row_begin, row_end):
        self.log.append(("upload_rows", slot, row_begin, row_end))

    def copy_pano_rows_from(self, slot, src, src_slot, row_begin, row_end):
        self.log.append(("copy_pano_rows_from", slot, src.dev, src_slot, row_begin, row_end))

    def copy_pano_from(self, slot, src, src_slot):
        self.log.append(("copy_pano_from", slot, src.dev, src_slot))


@pytest.fixture
def front(pkg, monkeypatch):
    front = pkg.panorama_to_plane_pitch
    FakeProjector.P2PError = pkg.engine.P2PError
    monkeypatch.setattr(front, "_default_devices", None)
    return front


@pytest.fixture
def sources(tmp_path):
    """A PNG and a JPEG file the device decoders take, and a 16-bit PNG they do not (host pixels)."""
    import cv2

    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (32, 64, 3), np.uint8)
    paths = {"png": tmp_path / "pano_p.png", "jpg": tmp_path / "pano_j.jpg", "host": tmp_path / "pano_h.png"}
    cv2.imwrite(str(paths["png"]), img)
    cv2.imwrite(str(paths["jpg"]), img)
    cv2.imwrite(str(paths["host"]), img.astype(np.uint16) * 257)
    return paths


def _install(front, monkeypatch, n_dev=1, **kw):
    """Stand-ins for devices 0 .. n_dev - 1; ``_decode_source`` calls are recorded in the log of the projector they get."""
    fakes = {d: FakeProjector(d, **kw) for d in range(n_dev)}
    monkeypatch.setattr(front, "get_projector", lambda device=None: fakes[0 if device is None else int(device)])
    real = front._decode_source

    def decode_source(proj, src, slot=None, device_declined=False):
        if isinstance(src, front._JpegSource):
            proj.log.append(("decode_source", device_declined))
        return real(proj, src, slot=slot, device_declined=device_declined)

    monkeypatch.setattr(front, "_decode_source", decode_source)
    return fakes


def _geometry(front, yaws):
    consts = [front.get_pitch_mapping(W, H, p, 64, 32, 90) for p in PITCHES]
    keys = [_yaw_key(front.get_yaw_mapping(64, 32, y)) for y in yaws]
    return keys, consts


def _src_kind(src):
    return "host" if src == "host" else ("declined" if src.startswith("declined") else "resident")


def _open(src, sources):
    return sources["host"] if src == "host" else sources["jpg" if src == "jpg" else "png"]


def _names(stem, yaws, fmt):
    return sorted(f"{stem}_{W}x{H}_yaw_{y}_pitch_{p}.{fmt}" for y in yaws for p in PITCHES)


def _check_written(out_dir, stem, yaws, fmt, keys, consts, none_first=False):
    import cv2

    assert sorted(p.name for p in out_dir.iterdir()) == _names(stem, yaws, fmt)
    for k, y in enumerate(yaws):
        for j, p in enumerate(PITCHES):
            path = out_dir / f"{stem}_{W}x{H}_yaw_{y}_pitch_{p}.{fmt}"
            if none_first and (k, j) == (0, 0):    # the device left this file out: cv2.imwrite of the read-back pixels
                assert np.all(cv2.imread(str(path)) == READBACK), path.name
            else:
                assert path.read_bytes() == _content((keys[k], consts[j])), path.name


def _prefix(kind, slot=0):
    """The calls that put the panorama of a source into a slot, or decide it stays host pixels."""
    if kind == "host":
        return []
    return [("upload_encoded", slot)] + ([("decode_source", True)] if kind == "declined" else [])


def _view_list_entry(fmt):
    return "process_view_list_png" if fmt == "png" else "process_view_list_jpeg"


def _decline_code(src):
    return int(src[len("declined"):]) if src.startswith("declined") else None


def _run_single(front, tmp_path, sources, src, yaws, fmt, devices=None):
    out_dir = tmp_path / f"out_{fmt}"
    out_dir.mkdir()
    path = _open(src, sources)
    front.process_single_image(path, out_dir, yaws, PITCHES, W, H, num_workers=2, output_format=fmt, devices=devices)
    return out_dir, path.stem


def _assert_slots_returned(fake):
    assert sorted(fake.free) == [0, 1, 2, 3] and len(fake.taken) % 2 == 0, fake.taken


@pytest.mark.parametrize("src", ["png", "jpg", "declined-6", "declined-3", "declined-5", "host"])
@pytest.mark.parametrize("yaw_kind", ["integer", "fractional"])
@pytest.mark.parametrize("fmt", ["jpg", "png"])
def test_files_flow_calls_one_device(front, monkeypatch, tmp_path, sources, src, yaw_kind, fmt):
    """One device, encoded outputs: the product entries for integer rolls, the view-list entries otherwise, from the
    resident panorama or from host pixels; the slot stays leased until the files are written."""
    yaws = YAWS[yaw_kind]
    fakes = _install(front, monkeypatch, decline=_decline_code(src))
    out_dir, stem = _run_single(front, tmp_path, sources, src, yaws, fmt)
    keys, consts = _geometry(front, yaws)
    kind = _src_kind(src)
    pano = "resident" if kind == "resident" else "pixels"
    product = [(s, c) for s in keys for c in consts]
    if yaw_kind == "integer" and fmt == "jpg":
        call = ("project_jpeg", 0, product, False) if pano == "resident" else ("process_image_jpeg", 0, pano, product, False)
    elif yaw_kind == "integer":
        call = ("process_image_png", 0, pano, product, False, False)
    elif fmt == "jpg":
        call = ("process_view_list_jpeg", 0, pano, product, False)
    else:
        call = ("process_view_list_png", 0, pano, product, False, False)
    assert fakes[0].log == _prefix(kind) + [call]
    assert fakes[0].taken == [("take", (0,)), ("give", (0,))]
    _check_written(out_dir, stem, yaws, fmt, keys, consts)


@pytest.mark.parametrize("src", ["png", "declined-6", "host"])
@pytest.mark.parametrize("yaw_kind", ["integer", "fractional"])
def test_png_file_left_out_is_written_from_read_back_pixels(front, monkeypatch, tmp_path, sources, src, yaw_kind):
    """A None PNG file (``sizes[i] = 0`` of the ABI): the views are read back from the same slot and cv2 writes it."""
    yaws = YAWS[yaw_kind]
    keys, consts = _geometry(front, yaws)
    fakes = _install(front, monkeypatch, decline=_decline_code(src), png_none=(keys[0], consts[0]))
    out_dir, stem = _run_single(front, tmp_path, sources, src, yaws, "png")
    kind = _src_kind(src)
    pano = "resident" if kind == "resident" else "pixels"
    product = [(s, c) for s in keys for c in consts]
    if yaw_kind == "integer":
        tail = [("process_image_png", 0, pano, product, False, False), ("project", 0, product), ("sync", 0)]
    else:
        tail = [("process_view_list_png", 0, pano, product, False, False), ("view_list", 0, product, (0, H)), ("sync", 0)]
    assert fakes[0].log == _prefix(kind) + tail
    _assert_slots_returned(fakes[0])
    _check_written(out_dir, stem, yaws, "png", keys, consts, none_first=True)


@pytest.mark.parametrize("src", ["png", "declined-5", "host"])
@pytest.mark.parametrize("yaw_kind", ["integer", "fractional"])
@pytest.mark.parametrize("fmt", ["jpg", "png", "bmp"])
def test_pixel_route_calls(front, monkeypatch, tmp_path, sources, src, yaw_kind, fmt):
    """Outputs cv2 encodes (any other format, or an encoder that ran out of memory / limits): ``_project`` renders the views
    from the resident panorama (``project_any``) or from host pixels (``project_image``)."""
    import cv2

    yaws = YAWS[yaw_kind]
    fallback = fmt != "bmp"
    fakes = _install(front, monkeypatch, decline=_decline_code(src), encoder_error=-5 if fallback else None)
    out_dir, stem = _run_single(front, tmp_path, sources, src, yaws, fmt)
    keys, consts = _geometry(front, yaws)
    kind = _src_kind(src)
    product = [(s, c) for s in keys for c in consts]
    log = []
    if fallback:   # the encoder call raised: its slot is leased, the pixel route takes another one
        pano = "resident" if kind == "resident" else "pixels"
        if yaw_kind == "integer" and fmt == "jpg":
            enc = ("project_jpeg", 0, product, False) if pano == "resident" else ("process_image_jpeg", 0, pano, product, False)
        elif yaw_kind == "integer":
            enc = ("process_image_png", 0, pano, product, False, False)
        else:
            enc = (_view_list_entry(fmt), 0, pano, product, False) + ((False,) if fmt == "png" else ())
        log = _prefix(kind) + [enc]
    s = 1 if fallback else 0
    if kind == "resident":
        log += [("upload_encoded", s), ("project_any", s, product)]
    elif kind == "declined":
        log += [("upload_encoded", s), ("decode_source", True), ("project_image", product)]
    else:
        log += [("project_image", product)]
    assert fakes[0].log == log
    _assert_slots_returned(fakes[0])
    assert sorted(p.name for p in out_dir.iterdir()) == _names(stem, yaws, fmt)
    assert all(cv2.imread(str(p)) is not None for p in out_dir.iterdir())


def _split_prefix(kind, n=2):
    """Per device: the calls of ``_split_upload`` (decode on device 0 and replicate, or scatter the host rows)."""
    logs = {d: [] for d in range(n)}
    if kind in ("resident", "declined"):
        logs[0] += _prefix(kind)
    if kind == "resident":
        logs[1] += [("copy_pano_from", 0, 0, 0)]
    else:   # two devices: each uploads half of the rows and fetches the other half (the last piece carries row Hp)
        logs[0] += [("upload_rows", 0, 0, 16), ("copy_pano_rows_from", 0, 1, 0, 16, 33)]
        logs[1] += [("upload_rows", 0, 16, 32), ("copy_pano_rows_from", 0, 0, 0, 0, 16)]
    return logs


@pytest.mark.parametrize("src", ["png", "declined-3", "host"])
@pytest.mark.parametrize("yaw_kind", ["integer", "fractional"])
@pytest.mark.parametrize("fmt", ["jpg", "png", "bmp"])
def test_split_over_two_devices_calls(pkg, front, monkeypatch, tmp_path, sources, src, yaw_kind, fmt):
    """One image over two devices: encoded outputs split the pitch-major view list into runs (one product call per pitch
    for integer rolls, one view-list call for fractional yaws); pixel outputs split every view into row bands (one
    view-list call per device).  A None PNG file adds the pixel split."""
    shard = importlib.import_module("p2p_b200.shard")
    yaws = YAWS[yaw_kind]
    keys, consts = _geometry(front, yaws)
    fakes = _install(front, monkeypatch, n_dev=2, decline=_decline_code(src),
                     png_none=(keys[0], consts[0]) if fmt == "png" else None)
    out_dir, stem = _run_single(front, tmp_path, sources, src, yaws, fmt, devices=[0, 1])
    kind = _src_kind(src)
    n_y, n_p = len(yaws), len(PITCHES)
    flat = [(s, c) for s in keys for c in consts]
    want = _split_prefix(kind)
    if fmt != "bmp":
        for r in range(2):
            views = shard.shard_views(n_y, n_p, r, 2)
            if yaw_kind == "fractional":
                vl = [(keys[k], consts[j]) for k, j in views]
                want[r] += [(_view_list_entry(fmt), 0, "resident", vl) + ((False, True) if fmt == "png" else (True,))]
            for j, ks in (shard.group_by_pitch(views).items() if yaw_kind == "integer" else ()):
                pv = [(keys[k], consts[j]) for k in ks]
                want[r] += [("process_image_png", 0, "resident", pv, False, True) if fmt == "png"
                            else ("project_jpeg", 0, pv, True)]
            want[r] += [("sync", 0)]
    if fmt != "jpg":   # pixels: "bmp" outputs, or the read-back of the None PNG file
        again = _split_prefix(kind) if fmt == "png" else {0: [], 1: []}
        for r in range(2):
            want[r] += (again[r] if fmt == "png" else []) + [("view_list", 0, flat, shard.shard_rows(H, r, 2)), ("sync", 0)]
    for r in range(2):
        assert fakes[r].log == want[r], r
        _assert_slots_returned(fakes[r])
    if fmt == "bmp":
        assert sorted(p.name for p in out_dir.iterdir()) == _names(stem, yaws, fmt)
    else:
        _check_written(out_dir, stem, yaws, fmt, keys, consts, none_first=fmt == "png")


@pytest.mark.gpu
@pytest.mark.parametrize("W", [64, 60])   # W % 8 == 0: the row-segment kernel; W % 8 != 0: the generic kernels
def test_files_entries_launch_the_projection_and_the_encoder(proj, W):
    """Each files entry point makes the projection launches of the pixel entry point with the same views, plus the
    encoder's (JPEG 8, PNG 11): the product entries those of ``p2p_project_views`` / ``p2p_process_image`` (yaws batched),
    the view-list entries those of ``p2p_project_view_list_tables`` (one launch per view where the row-segment kernel does
    not take the geometry), from a resident panorama and from host pixels."""
    from p2p_b200 import engine

    Wp, Hp, Hv = 256, 128, 40
    pano = np.random.default_rng(3).integers(0, 256, (Hp, Wp, 3), np.uint8)
    consts = [engine.pitch_constants(W, 90, p) for p in (60, 90)]
    shifts = [0, 64, 128, 192]                                   # a quarter-turn group
    tables = [engine.yaw_table(Wp, y) for y in (0, 10, 90)]      # an integer roll, a column table, a quarter turn
    flat_t, flat_c = [t for t in tables for _ in consts], consts * len(tables)
    jpeg, png = 8, 11
    with proj.slots(1) as (s,):
        def launches(call, resident=True):
            # a fresh panorama before every call: the same fold state (Slot::quarter_seen) each time; the second call
            # finds the row range of the geometry memoised like every later one
            for _ in range(2):
                if resident:
                    proj.upload(s, pano)
                proj.sync(s)
                n0 = proj.launches
                call()
                proj.sync(s)
                n = proj.launches - n0
            return n

        out = np.empty((len(shifts), len(consts), Hv, W, 3), np.uint8)
        project = launches(lambda: proj.project(s, shifts, consts, W, Hv, out=out))
        process = launches(lambda: proj.process_image(s, pano, shifts, consts, W, Hv, out), resident=False)
        listed = launches(lambda: proj.project_list_tables(s, flat_t, flat_c, W, Hv))
        assert launches(lambda: proj.project_jpeg(s, shifts, consts, W, Hv)) == project + jpeg
        assert launches(lambda: proj.process_image_png(s, None, shifts, consts, W, Hv)) == project + png
        assert launches(lambda: proj.process_image_jpeg(s, pano, shifts, consts, W, Hv), resident=False) == process + jpeg
        assert launches(lambda: proj.process_image_png(s, pano, shifts, consts, W, Hv), resident=False) == process + png
        assert launches(lambda: proj.process_view_list_jpeg(s, None, flat_t, flat_c, W, Hv)) == listed + jpeg
        assert launches(lambda: proj.process_view_list_png(s, None, flat_t, flat_c, W, Hv)) == listed + png
        upload = 1   # the host-pixel view-list entries pack the rows the views touch: one launch
        assert launches(lambda: proj.process_view_list_jpeg(s, pano, flat_t, flat_c, W, Hv), resident=False) == \
            upload + listed + jpeg
        assert launches(lambda: proj.process_view_list_png(s, pano, flat_t, flat_c, W, Hv), resident=False) == \
            upload + listed + png
