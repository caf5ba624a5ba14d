"""Drop-in mirror of the reference's ``app/panorama_to_plane-pitch.py`` for its hot path.

Same entry points, argument meaning, return types, file naming and error behaviour - the
arithmetic runs on the B200 through ``libp2p_b200.so``:

* ``process_yaw_and_pitchs(pano_image, yaw_angle, pitch_angles, output_width, output_height,
  fov_deg=90) -> list[np.ndarray]``                                   (ref :181-221)
* ``process_single_image(...)`` / ``main(...)`` / ``check_pitch``      (ref :227-280, :286-356, :362-376)
* ``panorama_to_plane(path, FOV, output_size, yaw, pitch) -> np.ndarray`` - the 5-argument front
  door BASELINE.json names (the reference's README lineage; equals
  ``process_yaw_and_pitchs(cv2.imread(path), yaw, [pitch], W, H, FOV)[0]``)
* the CLI with the reference's flags (ref :382-457), plus ``--device``.

The reference's two memo tables survive with the same keys (ref :17-18, :42-73) but hold what
the GPU path needs: the quantised yaw *column table* instead of a full-size (U, V) map, and the
three f32 *pitch constants* instead of a full-size map (the map itself is evaluated per pixel
inside the kernel and never stored).

Views are encoded on the GPU - PNG (``csrc/p2p_png.cuh``) and JPEG (``csrc/p2p_jpeg.cuh``) - byte-identical to what
``cv2.imwrite`` (ref :277) writes at OpenCV's defaults, so only the files cross PCIe; ``.jpg`` and ``.png`` panoramas are decoded
on the GPU too (``csrc/p2p_jpegdec.cuh``, ``csrc/p2p_pngdec.cuh``: same pixels as ``cv2.imread``, ref :244).  cv2 remains for the
few files / views outside the device codecs' subsets (and for damaged files, which the device decoders decline).
"""
from __future__ import annotations

import argparse
import contextlib
import logging
import os
import threading
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

from . import engine as _engine

VERSION = "0.3.2"  # the reference version this mirrors (ref :20)

# caches, same keys as the reference
yaw_mapping_cache: dict = {}    # (pano_width, pano_height, yaw_angle) -> (ix, fx, shift)
pitch_mapping_cache: dict = {}  # (W, H, pitch, pano_width, pano_height, fov) -> (f, c, s)

_projectors: dict = {}
_projectors_lock = threading.Lock()
_default_device = 0
_default_devices: list | None = None   # several devices: every single image is split over them (set_devices)


def get_version():
    return VERSION


def set_device(device: int):
    """Select the CUDA device the module-level entry points use (default 0)."""
    global _default_device
    _default_device = int(device)


def set_devices(devices):
    """Split every image the module-level entry points process over these CUDA devices of one box (None / one device:
    off).  The panorama is uploaded (or decoded) once and replicated with peer copies; pixel outputs are split by output
    row bands, encoded outputs by whole views (SURVEY 8e; the reference's unit of parallelism is the yaw task of its
    thread pool, ref :251-265).  Results are identical to the single-device path."""
    global _default_devices
    devs = [int(d) for d in devices] if devices else None
    _default_devices = devs if devs and len(devs) > 1 else None
    if devs and len(devs) == 1:
        set_device(devs[0])


def set_png_formats(all_formats: bool):
    """PNG inputs the device decoder takes (default False: 8-bit gray / RGB / gray + alpha / RGBA, not interlaced; True:
    also 16-bit, palette, 1/2/4-bit gray and Adam7-interlaced files, ``P2P_OPT_PNG_FORMATS`` = 1).  Same pixels as
    ``cv2.imread`` either way; the files left out are read with cv2.imread."""
    global _png_formats
    with _projectors_lock:
        _png_formats = 1 if all_formats else 0
        for proj in _projectors.values():
            proj.set_option(_engine._lib.OPT_PNG_FORMATS, _png_formats)


_png_formats = 0
_host_checked = False


def get_projector(device: int | None = None) -> _engine.Projector:
    global _host_checked
    d = _default_device if device is None else int(device)
    with _projectors_lock:
        if not _host_checked:   # once per process: say so if this host does not meet the bit-exactness assumptions
            _host_checked = True
            _engine.warn_if_host_differs(logging.getLogger())
        if d not in _projectors:
            _projectors[d] = _engine.Projector(d, n_slots=16)  # device buffers are allocated per slot on first use
            if _png_formats:
                _projectors[d].set_option(_engine._lib.OPT_PNG_FORMATS, _png_formats)
        return _projectors[d]


def get_yaw_mapping(pano_width, pano_height, yaw_angle):
    """Ref ``get_yaw_mapping`` :42-52, holding the column table (rows of the map are identical)."""
    key = (pano_width, pano_height, yaw_angle)
    if key not in yaw_mapping_cache:
        logging.debug(f"[Yaw] Precomputing yaw mapping for yaw_angle: {yaw_angle} degrees")
        yaw_mapping_cache[key] = _engine.yaw_table(pano_width, yaw_angle)
    return yaw_mapping_cache[key]


def get_pitch_mapping(output_width, output_height, pitch_angle, pano_width, pano_height, fov_deg=90):
    """Ref ``get_pitch_mapping`` :55-73, holding the per-pitch constants."""
    key = (output_width, output_height, pitch_angle, pano_width, pano_height, fov_deg)
    if key not in pitch_mapping_cache:
        pitch_mapping_cache[key] = _engine.pitch_constants(output_width, fov_deg, pitch_angle)
    return pitch_mapping_cache[key]


# what makes the front end read a file with cv2.imread after all: the device decoder declined it (-6: outside its subset, or
# damaged), or it could not get the scratch memory / the size is beyond its limits (-3, -5: huge files, many images in flight)
_DECLINED = (-6, -3, -5)


class _JpegSource:
    """A JPEG or PNG panorama one of the device decoders handles, still as file bytes (the pixels will only exist on the GPU)."""

    __slots__ = ("data", "Wp", "Hp", "path")

    def __init__(self, data, dims, path):
        self.data, (self.Wp, self.Hp), self.path = data, dims, path


def _open_image(path):
    """``cv2.imread(path)`` of the reference (ref :244): a BGR array, or None if unreadable - except that a JPEG or PNG file
    inside its device decoder's subset (baseline / progressive YCbCr without EXIF rotation; 8-bit non-interlaced PNG, every PNG
    format after ``set_png_formats(True)``) stays as bytes and is decoded on the GPU (same pixels, ``csrc/p2p_jpegdec.cuh`` /
    ``csrc/p2p_pngdec.cuh``)."""
    import cv2

    path = Path(path)
    if path.suffix.lower() in (".jpg", ".jpeg", ".png"):
        try:
            data = path.read_bytes()
        except OSError:
            data = b""
        # by content, like cv2.imread (which looks at the signature, not at the suffix)
        dims = _engine.probe_encoded(data, png_formats=_png_formats) if data else None
        if dims is not None:
            return _JpegSource(data, dims, path)
    return cv2.imread(str(path))


def _decode_source(proj, src, slot=None, device_declined=False):
    """Host pixels of a source (fractional-yaw path, or a damaged file the device decoder gave up on).  ``slot``: the slot
    the caller already holds (no second one is taken).  ``device_declined``: the device decoder has already refused this
    file (``upload_jpeg`` returned -6) - running the identical decode again could only fail again, go straight to cv2."""
    import cv2

    if not isinstance(src, _JpegSource):
        return src
    if not device_declined:
        try:
            return proj.decode_encoded(src.data, slot=slot)
        except _engine.P2PError as e:
            if e.code not in _DECLINED:
                raise
    # the reference's own call: cv2.imread, not imdecode (for a truncated file libjpeg's file reader pads the scan and
    # returns an image where its memory reader gives up)
    img = cv2.imread(str(src.path))
    if img is None:
        raise ValueError("Failed to decode image")
    return img


def _resident_or_pixels(proj, slot, src):
    """None when the panorama of ``src`` is now resident in ``slot`` (decoded there from its file), else its host pixels:
    a host array as it is, or a file the device decoder declined (or could not fit, ``_DECLINED``) read by cv2.imread."""
    if not isinstance(src, _JpegSource):
        return src
    try:
        proj.upload_encoded(slot, src.data)
        return None
    except _engine.P2PError as e:
        if e.code not in _DECLINED:
            raise
        return _decode_source(proj, src, slot=slot, device_declined=True)


def _geometry(src, yaw_angles, pitch_angles, output_width, output_height, fov_deg):
    if isinstance(src, _JpegSource):
        Wp, Hp = src.Wp, src.Hp
    else:
        Hp, Wp, _ = src.shape
    consts = [get_pitch_mapping(output_width, output_height, p, Wp, Hp, fov_deg) for p in pitch_angles]
    tables = [get_yaw_mapping(Wp, Hp, y) for y in yaw_angles]
    return consts, tables


def _project(proj, pano_image, yaw_angles, pitch_angles, output_width, output_height, fov_deg, devices=None):
    """[n_yaw][n_pitch] views through the batched device path, using the module caches.  ``devices`` (default: the list
    given to ``set_devices``): split this one image over several GPUs."""
    src = pano_image if isinstance(pano_image, _JpegSource) else _engine._as_u8_image(pano_image, "pano_image")
    consts, tables = _geometry(src, yaw_angles, pitch_angles, output_width, output_height, fov_deg)
    devs = _split_devices(devices, tables, yaw_angles, pitch_angles)
    if devs:
        return _project_split(devs, src, consts, tables, yaw_angles, pitch_angles, output_width, output_height)
    if isinstance(src, _JpegSource) and yaw_angles and pitch_angles:
        # decode on the device straight into a slot, project from there (fractional yaws too: one pass, same slot)
        with proj.slots(1) as (s,):
            src = _resident_or_pixels(proj, s, src)
            if src is None:
                return proj.project_any(s, tables, consts, output_width, output_height)
    return proj.project_image(_decode_source(proj, src), yaw_angles, pitch_angles, output_width, output_height, fov_deg,
                              consts=consts, tables=tables)


def _split_upload(projs, src, stack):
    """One slot per device, the panorama in all of them: uploaded (or JPEG-decoded) on the first device, replicated to
    the others with peer copies (NVLink) ordered after it on the device.  Returns the slots."""
    slots = [stack.enter_context(pr.slots(1))[0] for pr in projs]
    p0, s0 = projs[0], slots[0]
    pano = _resident_or_pixels(p0, s0, src)
    if pano is not None:
        # host pixels: every device uploads 1 / n of the rows over its own PCIe link and fetches the rest from its peers
        stack.callback(lambda keep=scatter_upload(projs, slots, pano): None)  # the host array outlives the async copies
        return slots
    for pr, sl in zip(projs[1:], slots[1:]):     # decoded on the first device: replicate from there
        pr.copy_pano_from(sl, p0, s0)
    return slots


def scatter_upload(projs, slots, pano):
    """The panorama in every ``(projs[r], slots[r])``: device r uploads rows [Hp r / n, Hp (r + 1) / n) and copies the other
    pieces from the devices that hold them (an all-gather made of NVLink peer copies, each ordered after its source's
    upload on the device).  All asynchronous; returns the host array, which must stay alive until the slots are synced."""
    pano = _engine._as_u8_image(pano, "pano_image")
    Hp, n = pano.shape[0], len(projs)
    b = [Hp * r // n for r in range(n + 1)]
    for r in range(n):
        if b[r] < b[r + 1]:
            projs[r].upload_rows(slots[r], pano, b[r], b[r + 1])
    packed_end = lambda hi: hi + (1 if hi == Hp else 0)   # packed rows: the last piece carries the clamp row Hp as well
    if n > 1 and (n & (n - 1)) == 0 and all(b[r] < b[r + 1] for r in range(n)):
        # recursive doubling: log2(n) exchanges per device with the partner r ^ 2^k, which holds the adjacent block of
        # 2^k pieces - n log2(n) peer copies (24 for 8 GPUs) instead of n (n - 1), the same bytes per device
        have = [(b[r], b[r + 1]) for r in range(n)]
        step = 1
        while step < n:
            nxt = list(have)
            for r in range(n):
                lo, hi = have[r ^ step]
                projs[r].copy_pano_rows_from(slots[r], projs[r ^ step], slots[r ^ step], lo, packed_end(hi))
                nxt[r] = (min(have[r][0], lo), max(have[r][1], hi))
            have = nxt
            step *= 2
        return pano
    for r in range(n):
        for q in list(range(r + 1, n)) + list(range(r - 1, -1, -1)):   # outwards from the own piece: always contiguous
            if b[q] < b[q + 1]:
                projs[r].copy_pano_rows_from(slots[r], projs[q], slots[q], b[q], packed_end(b[q + 1]))
    return pano


def _project_split(devices, src, consts, tables, yaw_angles, pitch_angles, W, H):
    """[n_yaw][n_pitch] views of ONE image rendered by several GPUs: device r renders the row band
    ``shard.shard_rows(H, r, n)`` of every view straight into the shared result array (one host thread per device)."""
    from . import shard

    projs = [get_projector(d) for d in devices]
    n = len(projs)
    n_y, n_p = len(yaw_angles), len(pitch_angles)
    out = np.empty((n_y, n_p, H, W, 3), np.uint8)
    flat_tables = [tables[k] for k in range(n_y) for _ in range(n_p)]
    flat_consts = [consts[j] for _ in range(n_y) for j in range(n_p)]
    with contextlib.ExitStack() as stack:
        slots = _split_upload(projs, src, stack)

        def run(r):
            rows = shard.shard_rows(H, r, n)
            if rows[0] < rows[1]:   # (integer rolls and column tables alike)
                projs[r].project_list_tables(slots[r], flat_tables, flat_consts, W, H, rows=rows,
                                             out=out.reshape(-1, H, W, 3))
            projs[r].sync(slots[r])

        with ThreadPoolExecutor(max_workers=n) as ex:
            list(ex.map(run, range(n)))
    return out


def _project_files_split(devices, fmt, src, consts, tables, yaw_angles, pitch_angles, W, H):
    """[n_yaw][n_pitch] encoded files (bytes) of ONE image from several GPUs: the encoders need whole views, so the
    pitch-major view list is cut into contiguous runs (``shard.shard_views``) and every device projects + encodes its run,
    one call per pitch it holds (``shard.group_by_pitch``)."""
    from . import shard

    projs = [get_projector(d) for d in devices]
    n = len(projs)
    n_y, n_p = len(yaw_angles), len(pitch_angles)
    files = [[None] * n_p for _ in range(n_y)]
    integer = all(t[2] is not None for t in tables)
    with contextlib.ExitStack() as stack:
        slots = _split_upload(projs, src, stack)

        def run(r):
            if not integer:   # fractional yaws: the device's whole run of views is one call of the view-list file entry
                views = shard.shard_views(n_y, n_p, r, n)
                if views:
                    vt, vc = [tables[k] for k, _ in views], [consts[j] for _, j in views]
                    if fmt == "png":
                        got = projs[r].process_view_list_png(slots[r], None, vt, vc, W, H)[0]
                    else:
                        got = projs[r].process_view_list_jpeg(slots[r], None, vt, vc, W, H)
                    for (k, j), f in zip(views, got):
                        files[k][j] = f
                projs[r].sync(slots[r])
                return
            for j, ks in shard.group_by_pitch(shard.shard_views(n_y, n_p, r, n)).items():
                shifts = [tables[k][2] for k in ks]
                if fmt == "png":
                    got = projs[r].process_image_png(slots[r], None, shifts, [consts[j]], W, H, want_pixels=False)[0]
                else:
                    got = projs[r].project_jpeg(slots[r], shifts, [consts[j]], W, H)
                for k, f in zip(ks, got):
                    files[k][j] = f
            projs[r].sync(slots[r])

        with ThreadPoolExecutor(max_workers=n) as ex:
            list(ex.map(run, range(n)))
    return files


def _split_devices(devices, tables, yaw_angles, pitch_angles):
    """The device list if this call is to be split over several GPUs (any yaws: integer rolls and column tables), else
    None."""
    devs = _default_devices if devices is None else ([int(d) for d in devices] if devices else None)
    if not devs or len(devs) < 2 or not yaw_angles or not pitch_angles:
        return None
    return devs


_ENCODER_FALLBACK_CODES = (-3, -5)   # P2P_ERR_NOMEM, P2P_ERR_LIMIT


def _is_jpeg(output_format) -> bool:
    return str(output_format).lower() in ("jpg", "jpeg")


def _slot(proj, lease):
    """A slot for one image: released when the ``with`` block ends, or - with a ``lease`` (an ``ExitStack`` the caller
    closes after the files are written) - kept until then, so that the files can be written straight from the slot's
    page-locked file buffer instead of being copied into ``bytes`` first."""
    import contextlib

    if lease is None:
        return proj.slots(1)
    (s,) = lease.enter_context(proj.slots(1))
    return contextlib.nullcontext((s,))


def _project_files(fmt, proj, pano_image, yaw_angles, pitch_angles, output_width, output_height, fov_deg, lease=None,
                   devices=None):
    """([n_yaw][n_pitch] files, views): the views projected and encoded on the device, ``fmt`` "jpg" or "png", using the
    module caches.  Files are bytes, or with a ``lease`` zero-copy views of the slot's file buffer (see ``_slot``).  Integer
    yaw rolls go to the product entries; with a fractional yaw the view-list entries project the integer rolls and the
    column tables together.  The panorama is decoded into the slot from its file, or only the rows the views touch are
    uploaded from host pixels, so no pixels cross PCIe.  A None file is a view the PNG encoder did not handle (the ABI's
    ``sizes[i] = 0``; not produced any more): ``views`` [n_yaw, n_pitch, H, W, 3] then holds the pixels of all views so that
    ``cv2.imwrite`` can write those, exactly as the reference would; otherwise ``views`` is None."""
    W, H = output_width, output_height
    src = pano_image if isinstance(pano_image, _JpegSource) else _engine._as_u8_image(pano_image, "pano_image")
    consts, tables = _geometry(src, yaw_angles, pitch_angles, W, H, fov_deg)
    n_p = len(pitch_angles)
    devs = _split_devices(devices, tables, yaw_angles, pitch_angles)
    if devs:
        files = _project_files_split(devs, fmt, src, consts, tables, yaw_angles, pitch_angles, W, H)
        views = None
        if any(f is None for per_yaw in files for f in per_yaw):  # (the device encoder handles every image today)
            views = _project_split(devs, src, consts, tables, yaw_angles, pitch_angles, W, H)
        return files, views
    if not yaw_angles or not pitch_angles:
        return [[] for _ in yaw_angles], None
    integer = all(t[2] is not None for t in tables)
    shifts = [t[2] for t in tables]
    flat_t = [t for t in tables for _ in consts]
    flat_c = list(consts) * len(tables)
    copy = lease is None
    with _slot(proj, lease) as (s,):
        pano = _resident_or_pixels(proj, s, src)
        if fmt == "png" and integer:
            flat = proj.process_image_png(s, pano, shifts, consts, W, H, want_pixels=False, copy=copy)[0]
        elif fmt == "png":
            flat = proj.process_view_list_png(s, pano, flat_t, flat_c, W, H, copy=copy)[0]
        elif integer and pano is None:   # JPEG in, JPEG out: no pixel ever crosses PCIe
            flat = proj.project_jpeg(s, shifts, consts, W, H, copy=copy)
        elif integer:
            flat = proj.process_image_jpeg(s, pano, shifts, consts, W, H, copy=copy)
        else:
            flat = proj.process_view_list_jpeg(s, pano, flat_t, flat_c, W, H, copy=copy)
        views = None
        if any(f is None for f in flat):         # read the pixels back only when cv2 has to write some views
            if integer:
                views = proj.project(s, shifts, consts, W, H)
            else:
                views = proj.project_list_tables(s, flat_t, flat_c, W, H).reshape(len(tables), n_p, H, W, 3)
            proj.sync(s)
    return [flat[k * n_p:(k + 1) * n_p] for k in range(len(yaw_angles))], views


def _out_path(output_dir, base_name, output_width, output_height, yaw_angle, pitch_angle, output_format):
    """The reference's name of an output file (ref :275)."""
    return output_dir / f"{base_name}_{output_width}x{output_height}_yaw_{yaw_angle}_pitch_{pitch_angle}.{output_format}"


def _save_files(files, base_name, output_dir, yaw_angles, pitch_angles, output_width, output_height, output_format,
                executor):
    """Write already-encoded views (one task per yaw, reference file names, ref :275); returns the futures."""

    def save_yaw(k):
        for i in range(len(pitch_angles)):
            path = _out_path(output_dir, base_name, output_width, output_height, yaw_angles[k], pitch_angles[i],
                             output_format)
            path.write_bytes(files[k][i])
            logging.debug(f"Saved {path}")

    return [executor.submit(save_yaw, k) for k in range(len(yaw_angles))]


def process_yaw_and_pitchs(pano_image, yaw_angle, pitch_angles, output_width, output_height, fov_deg=90):
    """Process a single yaw angle and multiple pitch angles, returning all slices (ref :181-221)."""
    logging.debug(f"[Yaw/Pitch] Starting processing for yaw_angle={yaw_angle}")
    pitch_angles = list(pitch_angles)
    if not pitch_angles:
        # the reference still runs its yaw pass and returns an empty list
        _ = np.asarray(pano_image).shape[2]
        return []
    out = _project(get_projector(), pano_image, [yaw_angle], pitch_angles, output_width, output_height, fov_deg)
    return [out[0, j] for j in range(len(pitch_angles))]


def panorama_to_plane(path, FOV, output_size, yaw, pitch):
    """One planar view of the panorama file at ``path``: u8 [H, W, 3] in cv2's BGR order.

    ``output_size`` is (width, height).  Raises ``FileNotFoundError`` if the image can not be read.
    """
    pano = _open_image(path)
    if pano is None:
        raise FileNotFoundError(f"Failed to read image: {path}")
    W, H = int(output_size[0]), int(output_size[1])
    return _project(get_projector(), pano, [yaw], [pitch], W, H, FOV)[0, 0]


def process_single_image(input_image_path, output_dir, yaw_angles, pitch_angles, output_width,
                         output_height, num_workers=4, output_format="png", fov_deg=90, devices=None):
    """Read one image, project every yaw x pitch view, save the results (ref :227-280).

    The reference submits one thread-pool task per yaw; here all views come from one batched
    device call and ``num_workers`` threads only run the file encoders.  Output names are the
    reference's (ref :275).  An unreadable image is logged and skipped (ref :245-247); a failure
    while saving one yaw's results is logged and the other yaws continue (ref :279-280).
    ``devices`` (extra): split this one image over several GPUs (same files, see ``set_devices``).
    """
    import cv2

    input_image_path = Path(input_image_path)
    output_dir = Path(output_dir)
    logging.info(f"Loading image: {input_image_path}")
    input_image = _open_image(input_image_path)
    if input_image is None:
        logging.error(f"Failed to read image: {input_image_path}")
        return
    base_name = input_image_path.stem
    yaw_angles = list(yaw_angles)
    pitch_angles = list(pitch_angles)
    jpeg = _is_jpeg(output_format)
    png = str(output_format).lower() == "png"
    files = None
    # the slot stays leased until the files are on disk: they are written straight from its page-locked buffer
    with contextlib.ExitStack() as lease, ThreadPoolExecutor(max_workers=max(1, int(num_workers))) as executor:
        try:
            try:
                if jpeg or png:  # projected and encoded on the device: only the files come back
                    files, views = _project_files("jpg" if jpeg else "png", get_projector(), input_image, yaw_angles,
                                                  pitch_angles, output_width, output_height, fov_deg, lease=lease,
                                                  devices=devices)
            except _engine.P2PError as e:
                if e.code not in _ENCODER_FALLBACK_CODES:
                    raise
                # the device encoders' scratch does not fit (huge views x many slots): the reference's own route,
                # pixels back + cv2.imwrite, still produces the files
                logging.warning(f"Device encoder unavailable for {input_image_path} ({e}); writing with cv2.imwrite")
                jpeg = png = False
            if not jpeg and not png:
                views = _project(get_projector(), input_image, yaw_angles, pitch_angles, output_width, output_height,
                                 fov_deg, devices=devices)
        except Exception as e:
            for yaw_angle in yaw_angles:
                logging.error(f"Error processing yaw_angle {yaw_angle}: {e}")
            return
        if jpeg:
            tasks = _save_files(files, base_name, output_dir, yaw_angles, pitch_angles, output_width, output_height,
                                output_format, executor)
        else:
            tasks = _save_views(cv2, views, base_name, output_dir, yaw_angles, pitch_angles, output_width,
                                output_height, output_format, executor, files)
        for future, yaw_angle in zip(tasks, yaw_angles):
            try:
                future.result()
            except Exception as e:
                logging.error(f"Error processing yaw_angle {yaw_angle}: {e}")


class _YawGroup:
    """The save tasks of one yaw: ``result()`` waits for all of them and re-raises the first failure, so callers keep
    the reference's per-yaw error reporting (ref :279-280) while every view is encoded by its own worker."""

    def __init__(self, futures):
        self.futures = futures

    def result(self):
        err = None
        for f in self.futures:
            try:
                f.result()
            except Exception as e:  # noqa: BLE001 - reported per yaw by the caller
                err = err or e
        if err is not None:
            raise err


def _save_views(cv2, views, base_name, output_dir, yaw_angles, pitch_angles, output_width, output_height,
                output_format, executor, files=None):
    """Submit one task per view (reference file names, ref :275): ``files[k][i]`` when the device encoded it, else
    ``cv2.imwrite`` of ``views[k, i]``; returns one waitable per yaw."""

    def save(k, i):
        path = _out_path(output_dir, base_name, output_width, output_height, yaw_angles[k], pitch_angles[i], output_format)
        if files is not None and files[k][i] is not None:
            path.write_bytes(files[k][i])
        else:
            cv2.imwrite(str(path), views[k, i])
        logging.debug(f"Saved {path}")

    return [_YawGroup([executor.submit(save, k, i) for i in range(len(pitch_angles))]) for k in range(len(yaw_angles))]


def process_image_batch(image_files, output_dir, yaw_angles, pitch_angles, output_width, output_height,
                        num_workers=4, output_format="png", fov_deg=90, devices=None, inflight=None, host_wait=None):
    """Directory front end (ref ``main`` :320-341 processes the files one after the other).

    Same files and names out as calling ``process_single_image`` per file, but ``inflight`` images (default: one per
    worker, at most 15) are in flight at once, each on its own slot (stream) driven by its own host thread, while the writer pool saves earlier results.
    ``devices`` shards the files round-robin over several GPUs (one pipeline per device, no data exchange).
    ``host_wait``: 1 = the in-flight threads sleep while they wait for the device, 0 = they spin (lowest latency, one busy
    core each); default: sleep as soon as in-flight threads plus writers outnumber the host's cores.
    """
    import cv2

    image_files = [Path(f) for f in image_files]
    output_dir = Path(output_dir)
    yaw_angles, pitch_angles = list(yaw_angles), list(pitch_angles)
    devices = [_default_device] if not devices else [int(d) for d in devices]
    num_workers = max(1, int(num_workers))
    W, H = int(output_width), int(output_height)

    def run_device(dev, files):
        """Every image is handled start to finish by one of ``inflight`` host threads on its own slot (stream): read
        (a JPEG the device decoder handles is Huffman-decoded on this thread, everything else by ``cv2.imread``),
        upload / decode, project, read back or encode, hand the files to the writer pool.  The library calls only
        hold the context lock while they enqueue, so the threads overlap on the GPU and on the host."""
        proj = get_projector(dev)
        # the host Huffman stage of a JPEG input runs on the worker thread: as many images in flight as there are workers
        n_in = max(1, min(int(inflight) if inflight else num_workers, proj.n_slots - 1))
        jpeg_out, png_out = _is_jpeg(output_format), str(output_format).lower() == "png"
        if jpeg_out or png_out:
            # every image in flight pins a file buffer of n_views x (W x H x 4 + 4096) bytes on its slot (plus the
            # encoders' device scratch): keep the total under a budget instead of running out of memory mid-folder
            per_slot = len(yaw_angles) * len(pitch_angles) * (W * H * 4 + 4096)
            budget = float(os.environ.get("P2P_PINNED_BUDGET_GB", "8")) * 2 ** 30
            n_in = max(1, min(n_in, int(budget // max(1, per_slot))))
        wait = host_wait if host_wait is not None else os.environ.get("P2P_HOST_WAIT")   # (the environment: for experiments)
        if wait is None:
            wait = 1 if (n_in + num_workers) * len(devices) > (os.cpu_count() or 1) else 0
        proj.set_option(_engine._lib.OPT_HOST_WAIT, int(bool(int(wait))))

        def one(f, writers):
            # the slot stays leased until this image's files are on disk (written straight from its page-locked buffer)
            with contextlib.ExitStack() as lease:
                one_leased(f, writers, lease)

        def one_leased(f, writers, lease):
            logging.info(f"Loading image: {f}")
            src = _open_image(f)
            if src is None:
                logging.error(f"Failed to read image: {f}")
                return
            try:
                futs = None
                try:
                    if jpeg_out or png_out:
                        files_, views = _project_files("jpg" if jpeg_out else "png", proj, src, yaw_angles, pitch_angles,
                                                       W, H, fov_deg, lease=lease, devices=[])
                        if jpeg_out:
                            futs = _save_files(files_, f.stem, output_dir, yaw_angles, pitch_angles, W, H, output_format,
                                               writers)
                        else:
                            futs = _save_views(cv2, views, f.stem, output_dir, yaw_angles, pitch_angles, W, H, output_format,
                                               writers, files_)
                except _engine.P2PError as e:
                    if e.code not in _ENCODER_FALLBACK_CODES:
                        raise
                    logging.warning(f"Device encoder unavailable for {f} ({e}); writing with cv2.imwrite")
                if futs is None:
                    views = _project(proj, src, yaw_angles, pitch_angles, W, H, fov_deg, devices=[])
                    futs = _save_views(cv2, views, f.stem, output_dir, yaw_angles, pitch_angles, W, H, output_format,
                                       writers)
            except Exception as e:
                for yaw in yaw_angles:
                    logging.error(f"Error processing yaw_angle {yaw}: {e}")
                return
            for fut, yaw in zip(futs, yaw_angles):
                try:
                    fut.result()
                except Exception as e:
                    logging.error(f"Error processing yaw_angle {yaw}: {e}")

        with ThreadPoolExecutor(max_workers=num_workers) as writers, ThreadPoolExecutor(max_workers=n_in) as workers:
            for fut in [workers.submit(one, f, writers) for f in files]:
                fut.result()

    if not yaw_angles or not pitch_angles:
        return
    if len(devices) == 1:
        run_device(devices[0], image_files)
    else:
        from . import shard

        with ThreadPoolExecutor(max_workers=len(devices)) as ex:
            futs = [ex.submit(run_device, d, [image_files[i] for i in shard.shard_images(len(image_files), r, len(devices))])
                    for r, d in enumerate(devices)]
            for fu in futs:
                fu.result()


def main(input_path, output_path, yaw_angles, pitch_angles, output_width, output_height,
         num_workers=None, output_format="png", fov_deg=90, enable_file_logging=False, devices=None):
    """Process a single image or every image under a folder (ref :286-356)."""
    if num_workers is None:
        cpu_cores = os.cpu_count() or 1
        num_workers = max(1, int(cpu_cores * 0.9))
        logging.info(f"No num_workers specified. Using {num_workers} (~90% of CPU cores).")
    else:
        logging.info(f"Using {num_workers} worker threads.")

    output_dir = Path(output_path)
    output_dir.mkdir(parents=True, exist_ok=True)
    logging.info(f"Output directory set to: {output_dir}")

    input_path_obj = Path(input_path)
    if input_path_obj.is_dir():
        valid_exts = {".jpg", ".jpeg", ".png"}
        all_images = [f for f in input_path_obj.rglob("*") if f.suffix.lower() in valid_exts]
        if not all_images:
            logging.warning(f"No images found in directory: {input_path_obj}")
            return
        logging.info(f"Found {len(all_images)} images in folder: {input_path_obj}")
    else:
        all_images = [input_path_obj]
    if len(all_images) == 1:
        # one image: its views are split over the devices (row bands / view runs), SURVEY 8e
        process_single_image(
            input_image_path=all_images[0], output_dir=output_dir, yaw_angles=yaw_angles,
            pitch_angles=pitch_angles, output_width=output_width, output_height=output_height,
            num_workers=num_workers, output_format=output_format, fov_deg=fov_deg, devices=devices,
        )
    else:
        process_image_batch(all_images, output_dir, yaw_angles, pitch_angles, output_width, output_height,
                            num_workers=num_workers, output_format=output_format, fov_deg=fov_deg, devices=devices)
    logging.info("All processing completed.")


def check_pitch(value: str) -> int:
    """Validate the pitch angle is within 1-179 degrees (ref :362-376; CLI only)."""
    try:
        pitch = int(value)
    except ValueError:
        raise argparse.ArgumentTypeError(f"Pitch angle must be an integer, got '{value}'.")
    if not (1 <= pitch <= 179):
        raise argparse.ArgumentTypeError(f"Pitch angle must be between 1 and 179 degrees, got {pitch}.")
    return pitch


def build_parser() -> argparse.ArgumentParser:
    """The reference's flags (ref :383-455) plus ``--device``."""
    p = argparse.ArgumentParser(
        description="Process panorama images or an entire folder of images into planar projections (B200 path)."
    )
    p.add_argument("--input_path", type=str, required=True, help="Path to the input panorama image or folder of images")
    p.add_argument("--output_path", type=str, default="output_images", help="Path to save the output images")
    p.add_argument("--output_format", type=str, choices=["png", "jpg", "jpeg"], default="png",
                   help="Output image format (png, jpg, jpeg)")
    p.add_argument("--FOV", type=int, default=90, help="Field of View in degrees")
    p.add_argument("--output_width", type=int, default=800, help="Width of the output image in pixels")
    p.add_argument("--output_height", type=int, default=800, help="Height of the output image in pixels")
    p.add_argument("--pitch_angles", nargs="+", type=check_pitch, default=[30, 60, 90, 120, 150],
                   help="List of pitch angles in degrees (1-179). e.g. --pitch_angles 30 60 90")
    p.add_argument("--yaw_angles", nargs="+", type=int, default=[0, 90, 180, 270],
                   help="List of yaw angles in degrees (0-360). e.g. --yaw_angles 0 90 180 270")
    p.add_argument("--num_workers", type=int, default=None,
                   help="Number of worker threads (file encoders here). If not specified, uses ~90%% of CPU cores.")
    p.add_argument("--enable_file_logging", action="store_true", help="Enable logging to a file.")
    p.add_argument("--device", type=int, default=0, help="CUDA device index (extra flag; default 0)")
    p.add_argument("--devices", type=int, nargs="+", default=None,
                   help="several CUDA devices: the files of a folder are sharded round-robin, a single image is split "
                        "by output row bands / views (extra flag)")
    p.add_argument("--png_all_formats", action="store_true",
                   help="decode 16-bit, palette, 1/2/4-bit gray and interlaced PNG inputs on the GPU too (extra flag; same "
                        "pixels as cv2.imread)")
    p.add_argument("-v", "--version", action="version", version=f"%(prog)s {get_version()}",
                   help="Show version information")
    return p


def cli(argv=None):
    args = build_parser().parse_args(argv)
    handlers = [logging.StreamHandler()]
    if args.enable_file_logging:
        log_file_path = Path.cwd() / "logs" / "app.log"
        log_file_path.parent.mkdir(parents=True, exist_ok=True)
        handlers.append(logging.FileHandler(log_file_path, mode="a"))
    logging.basicConfig(level=logging.INFO, format="%(asctime)s [%(levelname)s] %(message)s", handlers=handlers)
    set_device(args.device)
    set_png_formats(args.png_all_formats)
    main(
        input_path=args.input_path, output_path=args.output_path, yaw_angles=args.yaw_angles,
        pitch_angles=args.pitch_angles, output_width=args.output_width, output_height=args.output_height,
        num_workers=args.num_workers, output_format=args.output_format, fov_deg=args.FOV,
        enable_file_logging=args.enable_file_logging, devices=args.devices,
    )


if __name__ == "__main__":
    cli()
