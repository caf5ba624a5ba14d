"""Host side of the B200 projection path: a thin, typed wrapper over the C ABI.

``Projector`` owns one ``p2p_ctx`` (one CUDA device, ``n_slots`` panorama slots with their own
streams).  The host scalars the kernels need are formed here with the reference's own NumPy
expressions, so they are bit-identical to the reference by construction:

* ``pitch_constants``  - ref ``get_pitch_mapping`` :64, :68 (``np.radians``) and
  ``precompute_pitch_mapping`` :119 (focal length), :142-149 (``R_pitch`` entries in f32)
* ``yaw_table``        - one row of ref ``precompute_yaw_mapping`` :85-105, quantised to the
  1/32-px fixed point ``cv2.remap`` uses; a pure integer roll for every yaw with
  ``yaw * Wp / 360`` integral

Nothing here computes pixels; without the CUDA library the import fails (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import queue
import threading
from contextlib import contextmanager

import numpy as np

from . import _lib
from ._lib import P2PError, PitchConsts


# ------------------------------------------------------------------------------------------
# host scalars (NumPy, same expressions as the reference)
# ------------------------------------------------------------------------------------------
def pitch_constants(W: int, fov_deg, pitch_deg) -> tuple:
    fov_rad = np.radians(fov_deg)
    p = np.radians(pitch_deg)
    f = np.float32((0.5 * W) / np.tan(fov_rad / 2))
    return float(f), float(np.float32(np.cos(p))), float(np.float32(np.sin(p)))


def yaw_table(pano_width: int, yaw_deg):
    """(ix, fx, shift): quantised yaw column map; ``shift`` is None unless it is a pure roll."""
    yaw_radians = np.radians(yaw_deg)
    u = np.arange(pano_width, dtype=np.float32)
    phi = (2 * np.pi * u / pano_width).astype(np.float32)
    phi_rotated = (phi + yaw_radians) % (2 * np.pi)
    U = (phi_rotated * pano_width) / (2 * np.pi)
    U = np.clip(U, 0, pano_width - 1).astype(np.float32)
    s = np.rint(U * np.float32(32)).astype(np.int32)
    ix, fx = s >> 5, s & 31
    shift = None
    if not fx.any():
        s0 = int(ix[0])
        if np.array_equal(ix, (np.arange(pano_width, dtype=np.int64) + s0) % pano_width):
            shift = s0
    return np.ascontiguousarray(ix, np.int32), np.ascontiguousarray(fx, np.int32), shift


# Inputs on which NumPy's AVX-512 (Intel SVML) f32 arccos / arctan2 differ from the correctly rounded result, with the
# bits SVML returns: a host whose NumPy reproduces all of them evaluates the reference's coordinates exactly like the kernel
# does (P2P_OPT_TRIG = 0).  (bits of the inputs, bits of the result)
_SVML_ACOS = [(0x3f4b5f9b, 0x3f27196e), (0x3f0d26ad, 0x3f7c9e37), (0xbf0cb1a5, 0x4009c542), (0x3f3f4266, 0x3f3a230f),
              (0x3f18197c, 0x3f6f420f), (0xbd8356a4, 0x3fd146b7)]
_SVML_ATAN2 = [(0xbf08228e, 0x3ef486e0, 0xbf56caa4), (0x3da43f1d, 0x3f4f9ef9, 0x3dc9dcc2), (0x3e2f4aa4, 0x3f2aa213, 0x3e80b676),
               (0xbeae3612, 0x3e94d102, 0xbf5d2563), (0x3f5bde94, 0xbeb18192, 0x3ffa2b9f), (0x3ef1b780, 0xbec103ff, 0x400fa816)]
PINNED_VERSIONS = {"numpy": "2.3", "cv2": "4.13"}   # what the bit / byte identity claims were checked against


def host_assumptions() -> dict:
    """What the bit-exact claims rest on, checked on THIS host (no GPU needed):

    * ``numpy_svml``: NumPy evaluates f32 ``arccos`` / ``arctan2`` with the SVML routines the kernel restates (AVX-512
      hosts).  Elsewhere the reference itself changes in the last ulp and the device output is within <= 1 LSB of it
      instead of identical (DESIGN 2) - ``P2P_OPT_TRIG`` then makes no difference to parity.
    * ``numpy_nep50``: NumPy >= 2 scalar promotion (``phi + np.radians(int)`` is float64, ref :98); NumPy 1.x keeps float32
      there and produces another yaw table.
    * ``versions`` / ``pinned``: the byte-identical PNG / JPEG files and the JPEG decoder are pinned to OpenCV 4.13's bundled
      zlib / libpng / libjpeg-turbo settings; another OpenCV may write different (equally valid) bytes.
    """
    u32 = np.uint32
    az = np.array([a for a, _ in _SVML_ACOS], u32).view(np.float32)
    ar = np.array([r for _, r in _SVML_ACOS], u32)
    ty = np.array([y for y, _, _ in _SVML_ATAN2], u32).view(np.float32)
    tx = np.array([x for _, x, _ in _SVML_ATAN2], u32).view(np.float32)
    tr = np.array([r for _, _, r in _SVML_ATAN2], u32)
    svml = bool(np.array_equal(np.arccos(az).view(u32), ar) and np.array_equal(np.arctan2(ty, tx).view(u32), tr))
    nep50 = (np.float32(1) + np.radians(1)).dtype == np.float64
    versions = {"numpy": np.__version__}
    try:
        import cv2

        versions["cv2"] = cv2.__version__
    except Exception:  # noqa: BLE001
        versions["cv2"] = None
    matches = {k: (versions.get(k) or "").startswith(v) for k, v in PINNED_VERSIONS.items()}
    return {"numpy_svml": svml, "numpy_nep50": bool(nep50), "versions": versions, "pinned": dict(PINNED_VERSIONS),
            "versions_match_pinned": matches}


def warn_if_host_differs(log=None) -> dict:
    """Log one warning per assumption this host does not meet (called once by the front end); returns the report."""
    import logging

    log = log or logging.getLogger(__name__)
    rep = host_assumptions()
    if not rep["numpy_svml"]:
        log.warning("NumPy on this host does not use the AVX-512 SVML arccos / arctan2: outputs are within 1 LSB of the "
                    "reference run here instead of bit-identical (see DESIGN.md section 2)")
    if not rep["numpy_nep50"]:
        log.warning("NumPy < 2 scalar promotion: the reference's yaw table differs on this host")
    for k, ok in rep["versions_match_pinned"].items():
        if not ok:
            log.warning(f"{k} {rep['versions'].get(k)} differs from the version the byte-identity claims were checked "
                        f"against ({PINNED_VERSIONS[k]}.x)")
    return rep


def jpeg_probe(data: bytes):
    """(W, H) if the device JPEG decoder handles this file, else None (read it with cv2.imread).  Headers only, no GPU."""
    w, h = C.c_int(), C.c_int()
    rc = _lib.load().p2p_jpeg_probe(data, len(data), C.byref(w), C.byref(h))
    return (w.value, h.value) if rc == 0 else None


def png_probe(data: bytes, formats: int = 0):
    """(W, H) if the device PNG decoder accepts this file's structure (``formats`` = 0: 8-bit gray / RGB / gray + alpha /
    RGBA, not interlaced; 1: every PNG colour type and bit depth, Adam7 too - see ``P2P_OPT_PNG_FORMATS``; every chunk CRC
    intact), else None (read it with cv2.imread).  Chunk walk only, no GPU."""
    w, h = C.c_int(), C.c_int()
    rc = _lib.load().p2p_png_probe_ex(data, len(data), int(formats), C.byref(w), C.byref(h))
    return (w.value, h.value) if rc == 0 else None


def probe_encoded(data: bytes, png_formats: int = 0):
    """(W, H) if one of the device decoders handles this file (PNG by its signature, else JPEG), else None.
    ``png_formats``: the PNG decoder's subset (``png_probe``)."""
    return png_probe(data, png_formats) if data[:8] == b"\x89PNG\r\n\x1a\n" else jpeg_probe(data)


def _as_u8_image(a, what="panorama") -> np.ndarray:
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
        raise ValueError(f"{what} must be uint8 [H, W, 3], got {a.dtype} {a.shape}")
    if a.strides[2] != 1 or a.strides[1] != 3 or a.strides[0] < a.shape[1] * 3:
        a = np.ascontiguousarray(a)
    return a


class PinnedBuffer:
    """Page-locked host memory exposed as a NumPy array (overlapped H2D / D2H)."""

    def __init__(self, shape, dtype=np.uint8):
        lib = _lib.load()
        self.shape = tuple(int(x) for x in shape)
        self.nbytes = int(np.prod(self.shape)) * np.dtype(dtype).itemsize
        ptr = C.c_void_p()
        rc = lib.p2p_host_alloc(C.byref(ptr), self.nbytes)
        if rc:
            raise P2PError(rc, "pinned host allocation failed")
        self._ptr = ptr
        buf = (C.c_uint8 * self.nbytes).from_address(ptr.value)
        self.array = np.frombuffer(buf, dtype=dtype).reshape(self.shape)

    def free(self):
        if self._ptr is not None:
            self.array = None
            _lib.load().p2p_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Projector:
    """One device context.  Thread-safe; slots are handed out from a pool so concurrent callers
    (the reference drives this seam from a ThreadPoolExecutor, ref :252-265) never share one."""

    def __init__(self, device: int = 0, n_slots: int = 4):
        self.lib = _lib.load()
        self.device = int(device)
        self.n_slots = int(n_slots)
        ctx = C.c_void_p()
        rc = self.lib.p2p_create(self.device, self.n_slots, C.byref(ctx))
        if rc:
            raise P2PError(rc, f"p2p_create(device={device}) failed: "
                               f"{self.lib.p2p_status_string(rc).decode()} (no CUDA device? there is no CPU fallback)")
        self.ctx = ctx
        self._pool: queue.LifoQueue = queue.LifoQueue()  # LIFO: reuse the slot whose device buffers are already allocated
        for i in reversed(range(self.n_slots)):
            self._pool.put(i)
        self._lock = threading.Lock()
        self.png_formats = 0   # P2P_OPT_PNG_FORMATS as set through set_option: the subset decode_png probes with

    # -- plumbing ---------------------------------------------------------------------------
    def close(self):
        for pb in self.__dict__.pop("_jpeg_bufs", {}).values():
            pb.free()
        if getattr(self, "ctx", None):
            self.lib.p2p_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc: int):
        if rc:
            raise P2PError(rc, self.lib.p2p_last_error(self.ctx).decode(errors="replace"))

    @contextmanager
    def slots(self, n: int = 1):
        """Borrow ``n`` slots (blocks until available)."""
        if n > self.n_slots:
            raise ValueError(f"need {n} slots, context has {self.n_slots}")
        with self._lock:  # take all n atomically so two callers can not deadlock on partial sets
            got = [self._pool.get() for _ in range(n)]
        try:
            yield got
        finally:
            for s in got:
                self._pool.put(s)

    def set_option(self, key: int, value: int):
        self._ck(self.lib.p2p_set_option(self.ctx, key, value))
        if key == _lib.OPT_PNG_FORMATS:
            self.png_formats = int(value)

    def get_option(self, key: int) -> int:
        v = C.c_int()
        self._ck(self.lib.p2p_get_option(self.ctx, key, C.byref(v)))
        return v.value

    @property
    def launches(self) -> int:
        return self.get_option(_lib.OPT_COUNT_LAUNCHES)

    def sync(self, slot: int = -1):
        self._ck(self.lib.p2p_sync(self.ctx, slot))

    def poison(self, slot: int, byte: int):
        """Debug: fill everything ``slot`` does not hold with ``byte`` (``p2p_debug_poison``); waits for the slot."""
        self._ck(self.lib.p2p_debug_poison(self.ctx, slot, int(byte)))

    # -- raw ABI calls ----------------------------------------------------------------------
    def upload(self, slot: int, pano: np.ndarray):
        pano = _as_u8_image(pano)
        Hp, Wp, _ = pano.shape
        self._ck(self.lib.p2p_upload_pano(self.ctx, slot, pano.ctypes.data, Wp, Hp, pano.strides[0]))
        return pano  # caller keeps it alive until the slot is synced

    def upload_device(self, slot: int, dev_ptr: int, Wp: int, Hp: int, row_stride: int):
        self._ck(self.lib.p2p_upload_pano_device(self.ctx, slot, C.c_void_p(dev_ptr), Wp, Hp, row_stride))

    def rotate(self, src_slot: int, dst_slot: int, ix: np.ndarray, fx: np.ndarray):
        ix = np.ascontiguousarray(ix, np.int32)
        fx = np.ascontiguousarray(fx, np.int32)
        self._ck(self.lib.p2p_rotate_pano(self.ctx, src_slot, dst_slot,
                                          ix.ctypes.data_as(C.POINTER(C.c_int32)),
                                          fx.ctypes.data_as(C.POINTER(C.c_int32))))

    @staticmethod
    def _consts_array(consts):
        arr = (PitchConsts * len(consts))()
        for i, (f, c, s) in enumerate(consts):
            arr[i].f, arr[i].c, arr[i].s = f, c, s
        return arr

    @staticmethod
    def _out_arg(out, out_device_ptr, shape):
        """(out, destination, out_on_device) of a projection: ``out_device_ptr``, else the host array ``out`` (created with
        ``shape`` if None), which must be C-contiguous uint8 with as many elements as ``shape``."""
        if out_device_ptr is not None:
            return out, C.c_void_p(out_device_ptr), 1
        if out is None:
            out = np.empty(shape, np.uint8)
        if out.dtype != np.uint8 or not out.flags.c_contiguous or out.size != int(np.prod(shape)):
            raise ValueError(f"out must be C-contiguous uint8 with {' * '.join(map(str, shape))} elements")
        return out, out.ctypes.data, 0

    def project(self, slot: int, shifts, consts, W: int, H: int, out=None, out_device_ptr: int | None = None):
        """Enqueue n_yaw x n_pitch views.  ``out``: host array [n_yaw, n_pitch, H, W, 3] (created if
        None) or ``out_device_ptr`` for device-resident results.  Returns ``out`` (valid after sync)."""
        shifts = np.ascontiguousarray(shifts, np.int32)
        n_yaw, n_pitch = int(shifts.shape[0]), len(consts)
        pc = self._consts_array(consts)
        out, dst, on_dev = self._out_arg(out, out_device_ptr, (n_yaw, n_pitch, H, W, 3))
        self._ck(self.lib.p2p_project_views(self.ctx, slot, n_yaw, shifts.ctypes.data_as(C.POINTER(C.c_int32)),
                                            n_pitch, pc, W, H, dst, on_dev))
        return out

    def project_tables(self, slot: int, tables, consts, W: int, H: int, out=None, out_device_ptr: int | None = None):
        """Enqueue n_yaw x n_pitch views for yaws that are NOT integer column rolls, in one pass: ``tables[k] = (ix, fx)``
        is yaw k's column table from :func:`yaw_table`.  Both remap passes of the reference (ref :191-199, :212-218) are
        evaluated per output pixel; bit-identical to :meth:`rotate` + :meth:`project`.  ``out`` as in :meth:`project`."""
        n_yaw, n_pitch = len(tables), len(consts)
        pc = self._consts_array(consts)
        ixs = [np.ascontiguousarray(t[0], np.int32) for t in tables]
        fxs = [np.ascontiguousarray(t[1], np.int32) for t in tables]
        P = C.POINTER(C.c_int32)
        ixp = (P * n_yaw)(*[a.ctypes.data_as(P) for a in ixs])
        fxp = (P * n_yaw)(*[a.ctypes.data_as(P) for a in fxs])
        out, dst, on_dev = self._out_arg(out, out_device_ptr, (n_yaw, n_pitch, H, W, 3))
        self._ck(self.lib.p2p_project_views_table(self.ctx, slot, n_yaw, ixp, fxp, n_pitch, pc, W, H, dst, on_dev))
        return out

    def project_any(self, slot: int, tables, consts, W: int, H: int, out: np.ndarray | None = None) -> np.ndarray:
        """All yaw x pitch views of the panorama resident in ``slot`` into the host array ``out``
        [n_yaw, n_pitch, H, W, 3]: integer-roll yaws only through :meth:`project`; with fractional yaws the whole yaw x pitch
        list is one :meth:`project_list_tables` call (integer rolls and tables, at most two launches, no host wait between
        them).  ``tables[k]`` = :func:`yaw_table` of yaw k.  Synchronous."""
        if out is None:
            out = np.empty((len(tables), len(consts), H, W, 3), np.uint8)
        if all(t[2] is not None for t in tables):
            self.project(slot, [t[2] for t in tables], consts, W, H, out=out)
        else:
            flat_tables = [t for t in tables for _ in consts]
            self.project_list_tables(slot, flat_tables, list(consts) * len(tables), W, H, out=out.reshape(-1, H, W, 3))
        self.sync(slot)
        return out

    @staticmethod
    def _view_tables(tables):
        """ABI form of a flat list of yaws, ``tables[i]`` = :func:`yaw_table` of view i: (yaw_shift with -1 for a
        fractional yaw, ix / fx pointer arrays - NULL for integer rolls, one pointer per distinct table object so that views
        of one yaw share a device table -, the arrays the pointers refer to)."""
        P = C.POINTER(C.c_int32)
        n = len(tables)
        shifts = np.array([-1 if t[2] is None else t[2] for t in tables], np.int32)
        ixp, fxp = (P * n)(), (P * n)()
        keep = []
        for i, t in enumerate(tables):
            if t[2] is None:
                ix, fx = np.ascontiguousarray(t[0], np.int32), np.ascontiguousarray(t[1], np.int32)
                keep += [ix, fx]
                ixp[i], fxp[i] = ix.ctypes.data_as(P), fx.ctypes.data_as(P)
        return shifts, ixp, fxp, keep

    def project_list_tables(self, slot: int, tables, consts, W: int, H: int, rows=None, out=None,
                            out_device_ptr: int | None = None):
        """:meth:`project_list` for any yaws: view i = (``tables[i]``, ``consts[i]``), ``tables[i]`` = :func:`yaw_table` of
        its yaw - an integer roll or, for a fractional yaw, its column table (both remap passes of the reference per output
        pixel, the bytes of :meth:`project_tables`).  ``rows``, ``out``, ``out_device_ptr`` as in :meth:`project_list`.
        The slot may be partial (``process_image``, ``upload_rows``) when it holds the rows the views touch."""
        n = len(tables)
        if len(consts) != n:
            raise ValueError("one pitch-constant triple per view")
        shifts, ixp, fxp, keep = self._view_tables(tables)
        pc = self._consts_array(consts)
        r0, r1 = (0, H) if rows is None else (int(rows[0]), int(rows[1]))
        out, dst, on_dev = self._out_arg(out, out_device_ptr, (n, H, W, 3))
        self._ck(self.lib.p2p_project_view_list_tables(self.ctx, slot, n, shifts.ctypes.data_as(C.POINTER(C.c_int32)),
                                                       ixp, fxp, pc, W, H, r0, r1, dst, on_dev))
        return out

    def project_list(self, slot: int, shifts, consts, W: int, H: int, rows=None, out=None,
                     out_device_ptr: int | None = None):
        """Enqueue a flat list of views - view i = (shifts[i], consts[i]) - in one launch; ``rows = (begin, end)`` renders
        only that band of output rows of every view (the multi-GPU split of a single image).  ``out``: host array
        [n_views, H, W, 3] (created if None; only the band is written) or ``out_device_ptr``.  Valid after sync."""
        shifts = np.ascontiguousarray(shifts, np.int32)
        n = int(shifts.shape[0])
        if len(consts) != n:
            raise ValueError("one pitch-constant triple per view")
        pc = self._consts_array(consts)
        r0, r1 = (0, H) if rows is None else (int(rows[0]), int(rows[1]))
        out, dst, on_dev = self._out_arg(out, out_device_ptr, (n, H, W, 3))
        self._ck(self.lib.p2p_project_view_list(self.ctx, slot, n, shifts.ctypes.data_as(C.POINTER(C.c_int32)), pc, W, H,
                                                r0, r1, dst, on_dev))
        return out

    def copy_pano_from(self, slot: int, src: "Projector", src_slot: int):
        """Replicate the panorama of ``src``'s slot (another device's context) into ``slot`` over NVLink / PCIe peer copy;
        asynchronous on this slot's stream, ordered after the source slot's enqueued work."""
        rc = self.lib.p2p_copy_pano(self.ctx, slot, src.ctx, src_slot)
        self._ck(rc)

    def upload_rows(self, slot: int, pano: np.ndarray, row_begin: int, row_end: int):
        """Upload + pack panorama rows [row_begin, row_end) only (a piece of an image split over GPUs)."""
        pano = _as_u8_image(pano)
        Hp, Wp, _ = pano.shape
        self._ck(self.lib.p2p_upload_pano_rows(self.ctx, slot, pano.ctypes.data, Wp, Hp, pano.strides[0],
                                               int(row_begin), int(row_end)))
        return pano

    def copy_pano_rows_from(self, slot: int, src: "Projector", src_slot: int, row_begin: int, row_end: int):
        """Fetch packed rows [row_begin, row_end) (0 .. Hp + 1: the clamp row is row Hp) from another context's slot."""
        self._ck(self.lib.p2p_copy_pano_rows(self.ctx, slot, src.ctx, src_slot, int(row_begin), int(row_end)))

    def project_list_call(self, slot: int, shifts, consts, W: int, H: int, rows=None, out=None,
                          out_device_ptr: int | None = None):
        """``project_list`` with the arguments marshalled once: returns a zero-argument callable (hot loops)."""
        shifts_a = np.ascontiguousarray(shifts, np.int32)
        pc = self._consts_array(consts)
        r0, r1 = (0, H) if rows is None else (int(rows[0]), int(rows[1]))
        dst, on_dev = (C.c_void_p(out_device_ptr), 1) if out_device_ptr is not None else (out.ctypes.data, 0)
        args = (self.ctx, slot, int(shifts_a.shape[0]), shifts_a.ctypes.data_as(C.POINTER(C.c_int32)), pc, W, H, r0, r1,
                dst, on_dev)
        fn = self.lib.p2p_project_view_list

        def call(_keep=(shifts_a, pc, out)):
            self._ck(fn(*args))

        return call

    def batch_call(self, slots, shifts, consts, W: int, H: int, out_ptrs, on_device: bool = True):
        """Prebuilt ``p2p_project_batch`` call for resident panoramas: returns a zero-argument
        callable that enqueues one launch per slot (arguments are marshalled once)."""
        slots_a = np.ascontiguousarray(slots, np.int32)
        shifts_a = np.ascontiguousarray(shifts, np.int32)
        pc = self._consts_array(consts)
        outs = (C.c_void_p * len(out_ptrs))(*[int(p) for p in out_ptrs])
        args = (self.ctx, len(slots_a), slots_a.ctypes.data_as(C.POINTER(C.c_int32)), int(shifts_a.shape[0]),
                shifts_a.ctypes.data_as(C.POINTER(C.c_int32)), len(consts), pc, W, H, outs, 1 if on_device else 0)
        fn = self.lib.p2p_project_batch

        def call(_keep=(slots_a, shifts_a, pc, outs)):
            self._ck(fn(*args))

        return call

    def process_image(self, slot: int, pano: np.ndarray, shifts, consts, W: int, H: int, out: np.ndarray):
        """upload + project + readback in one ABI call (asynchronous; sync the slot before reading)."""
        pano = _as_u8_image(pano)
        Hp, Wp, _ = pano.shape
        shifts = np.ascontiguousarray(shifts, np.int32)
        pc = self._consts_array(consts)
        self._ck(self.lib.p2p_process_image(self.ctx, slot, pano.ctypes.data, Wp, Hp, pano.strides[0],
                                            int(shifts.shape[0]), shifts.ctypes.data_as(C.POINTER(C.c_int32)),
                                            len(consts), pc, W, H, out.ctypes.data))
        return out

    # -- files (the encode side of cv2.imwrite, ref :277) ---------------------------------------
    def _file_buffer(self, slot: int, n: int, stride: int) -> np.ndarray:
        """page-locked [n, stride] file buffer of a slot (a slot is driven by one thread at a time)"""
        cache = self.__dict__.setdefault("_jpeg_bufs", {})
        pb = cache.get(slot)
        if pb is None or pb.shape[0] < n or pb.shape[1] < stride:
            if pb is not None:
                pb.free()
            pb = cache[slot] = PinnedBuffer((n, stride))
        return pb.array[:n]

    @staticmethod
    def _files(buf: np.ndarray, sizes, copy: bool) -> list:
        """The files of a slot's file buffer: ``bytes`` (copy) or zero-copy ``memoryview`` slices of the page-locked
        buffer, valid until the slot is used again (size 0 = not handled on the device -> None)."""
        if copy:
            return [buf[i, :sizes[i]].tobytes() if sizes[i] else None for i in range(len(sizes))]
        return [memoryview(buf[i, :sizes[i]]) if sizes[i] else None for i in range(len(sizes))]

    def _files_call(self, fn, slot: int, args, n: int, stride: int, copy: bool = True, pixels=()) -> list:
        """One files entry of the ABI, ``fn(ctx, slot, *args, file_buffer, file_stride, sizes, *pixels)``: the n files land
        in the slot's page-locked file buffer, ``stride`` bytes apart, and come back as :meth:`_files` returns them.
        ``pixels``: the pixel output of the PNG entries that take one, ``(array or None,)``."""
        buf = self._file_buffer(slot, n, stride)
        sizes = (C.c_size_t * n)()
        self._ck(fn(self.ctx, slot, *args, buf.ctypes.data, buf.strides[0], sizes,
                    *[None if p is None else p.ctypes.data for p in pixels]))
        return self._files(buf, sizes, copy)

    @staticmethod
    def _pano_args(pano):
        """(pointer, Wp, Hp, row stride, array) of the optional host panorama of a files entry (None: the resident one)."""
        if pano is None:
            return None, 0, 0, 0, None
        pano = _as_u8_image(pano)
        Hp, Wp, _ = pano.shape
        return pano.ctypes.data, Wp, Hp, pano.strides[0], pano

    def encode_jpeg(self, images: np.ndarray, quality: int = 95, slot: int | None = None) -> list:
        """JPEG files (bytes) of ``images`` u8 [n, H, W, 3] (BGR), encoded on the GPU; byte-identical to
        ``cv2.imencode('.jpg', image)`` at OpenCV's defaults."""
        images = np.ascontiguousarray(images, np.uint8)
        if images.ndim == 3:
            images = images[None]
        n, H, W, ch = images.shape
        if ch != 3:
            raise ValueError("images must be [n, H, W, 3]")

        def run(s):
            return self._files_call(self.lib.p2p_encode_jpeg, s, (images.ctypes.data, 0, n, W, H, int(quality)), n,
                                    W * H * 3 + 4096)

        if slot is None:
            with self.slots(1) as (s,):
                return run(s)
        return run(slot)

    def project_jpeg(self, slot: int, shifts, consts, W: int, H: int, quality: int = 95, copy: bool = True) -> list:
        """The n_yaw x n_pitch views of the panorama in ``slot`` as JPEG files (bytes, yaw-major): projection and
        encoder both run on the device, only the files cross PCIe.  ``copy=False``: memoryviews of the slot's page-locked
        file buffer instead of bytes (valid until the slot is used again)."""
        shifts = np.ascontiguousarray(shifts, np.int32)
        n_yaw, n_pitch = int(shifts.shape[0]), len(consts)
        args = (n_yaw, shifts.ctypes.data_as(C.POINTER(C.c_int32)), n_pitch, self._consts_array(consts), W, H, int(quality))
        return self._files_call(self.lib.p2p_project_views_jpeg, slot, args, n_yaw * n_pitch, W * H * 3 + 4096, copy)

    def process_image_jpeg(self, slot: int, pano: np.ndarray, shifts, consts, W: int, H: int, quality: int = 95,
                           copy: bool = True) -> list:
        """upload (the rows the views touch) + project + JPEG-encode in one ABI call: the files (bytes, yaw-major;
        ``copy=False``: memoryviews of the slot's file buffer) of all n_yaw x n_pitch views.  Blocks this thread only;
        other slots keep running."""
        src, Wp, Hp, stride, pano = self._pano_args(_as_u8_image(pano))
        shifts = np.ascontiguousarray(shifts, np.int32)
        n_yaw, n_pitch = int(shifts.shape[0]), len(consts)
        args = (src, Wp, Hp, stride, n_yaw, shifts.ctypes.data_as(C.POINTER(C.c_int32)), n_pitch, self._consts_array(consts),
                W, H, int(quality))
        return self._files_call(self.lib.p2p_process_image_jpeg, slot, args, n_yaw * n_pitch, W * H * 3 + 4096, copy)

    def project_image_jpeg(self, pano: np.ndarray, yaw_angles, pitch_angles, W: int, H: int, fov_deg=90,
                           consts=None, tables=None, quality: int = 95) -> list:
        """JPEG files [n_yaw][n_pitch] (bytes) of all views of one panorama; byte-identical to ``cv2.imwrite`` of
        the views ``project_image`` returns.  Fractional yaws render through ``project_image`` first."""
        pano = _as_u8_image(pano)
        Hp, Wp, _ = pano.shape
        yaw_angles, pitch_angles = list(yaw_angles), list(pitch_angles)
        if consts is None:
            consts = [pitch_constants(W, fov_deg, p) for p in pitch_angles]
        if tables is None:
            tables = [yaw_table(Wp, y) for y in yaw_angles]
        if not yaw_angles or not pitch_angles:
            return [[] for _ in yaw_angles]
        if all(t[2] is not None for t in tables):
            with self.slots(1) as (s,):
                flat = self.process_image_jpeg(s, pano, [t[2] for t in tables], consts, W, H, quality)
        else:
            views = self.project_image(pano, yaw_angles, pitch_angles, W, H, fov_deg, consts=consts, tables=tables)
            flat = self.encode_jpeg(views.reshape(-1, H, W, 3), quality)
        n_p = len(pitch_angles)
        return [flat[k * n_p:(k + 1) * n_p] for k in range(len(yaw_angles))]

    # -- PNG files (cv2.imwrite(<name>.png), ref :277: the default output format) -------------------
    def encode_png(self, images: np.ndarray, slot: int | None = None) -> list:
        """PNG files (bytes) of ``images`` u8 [n, H, W, 3] (BGR), encoded on the GPU; byte-identical to
        ``cv2.imencode('.png', image)`` (small images and incompressible content included).  ``None`` would mean "not
        handled on the device, encode it with cv2" (``sizes[i] = 0`` of the ABI); no input produces it any more."""
        images = np.ascontiguousarray(images, np.uint8)
        if images.ndim == 3:
            images = images[None]
        n, H, W, ch = images.shape
        if ch != 3:
            raise ValueError("images must be [n, H, W, 3]")

        def run(s):
            return self._files_call(self.lib.p2p_encode_png, s, (images.ctypes.data, 0, n, W, H), n, W * H * 4 + 4096)

        if slot is None:
            with self.slots(1) as (s,):
                return run(s)
        return run(slot)

    def process_image_png(self, slot: int, pano, shifts, consts, W: int, H: int, want_pixels: bool = True,
                          copy: bool = True):
        """upload (``pano`` = None: use the panorama resident in ``slot``) + project + PNG-encode in one ABI call.
        Returns (files, pixels): files[i] is bytes (``copy=False``: a memoryview of the slot's page-locked file buffer,
        valid until the slot is used again) or None (view not handled by the device encoder); pixels is the
        [n_yaw, n_pitch, H, W, 3] array when ``want_pixels`` (so the caller can ``cv2.imwrite`` the None views)."""
        src, Wp, Hp, stride, pano = self._pano_args(pano)
        shifts = np.ascontiguousarray(shifts, np.int32)
        n_yaw, n_pitch = int(shifts.shape[0]), len(consts)
        pixels = np.empty((n_yaw, n_pitch, H, W, 3), np.uint8) if want_pixels else None
        args = (src, Wp, Hp, stride, n_yaw, shifts.ctypes.data_as(C.POINTER(C.c_int32)), n_pitch, self._consts_array(consts),
                W, H)
        files = self._files_call(self.lib.p2p_process_image_png, slot, args, n_yaw * n_pitch, W * H * 4 + 4096, copy,
                                 (pixels,))
        return files, pixels

    # -- files of a flat list of any yaws ------------------------------------------------------------------------
    def process_view_list_jpeg(self, slot: int, pano, tables, consts, W: int, H: int, quality: int = 95,
                               copy: bool = True) -> list:
        """JPEG files of the flat view list of :meth:`project_list_tables` (file i = view i; integer rolls and fractional
        yaws alike): ``pano`` = None projects the panorama resident in ``slot`` (e.g. decoded there by
        :meth:`upload_encoded`), else only the rows the views touch are uploaded.  Only the files cross PCIe.  ``copy`` as
        in :meth:`project_jpeg`."""
        n = len(tables)
        shifts, ixp, fxp, keep = self._view_tables(tables)
        src, Wp, Hp, stride, pano = self._pano_args(pano)
        args = (src, Wp, Hp, stride, n, shifts.ctypes.data_as(C.POINTER(C.c_int32)), ixp, fxp, self._consts_array(consts),
                W, H, int(quality))
        return self._files_call(self.lib.p2p_process_view_list_jpeg, slot, args, n, W * H * 3 + 4096, copy)

    def process_view_list_png(self, slot: int, pano, tables, consts, W: int, H: int, want_pixels: bool = False,
                              copy: bool = True):
        """PNG files of the flat view list of :meth:`project_list_tables`, like :meth:`process_view_list_jpeg`.  Returns
        (files, pixels): pixels is the [n_views, H, W, 3] array when ``want_pixels`` (for views the device encoder did not
        handle, see :meth:`process_image_png`)."""
        n = len(tables)
        shifts, ixp, fxp, keep = self._view_tables(tables)
        src, Wp, Hp, stride, pano = self._pano_args(pano)
        pixels = np.empty((n, H, W, 3), np.uint8) if want_pixels else None
        args = (src, Wp, Hp, stride, n, shifts.ctypes.data_as(C.POINTER(C.c_int32)), ixp, fxp, self._consts_array(consts),
                W, H)
        return self._files_call(self.lib.p2p_process_view_list_png, slot, args, n, W * H * 4 + 4096, copy, (pixels,)), pixels

    # -- JPEG panoramas decoded on the device (the decode side of cv2.imread, ref :244) ----------
    def jpeg_probe(self, data: bytes):
        """(W, H) if the device decoder handles this file, else None (read it with cv2.imread)."""
        return jpeg_probe(data)

    def upload_jpeg(self, slot: int, data: bytes) -> tuple:
        """Decode a JPEG file into ``slot`` as its panorama; returns (Wp, Hp).  Raises ``P2PError`` with code -6 for
        files outside the supported subset."""
        w, h = C.c_int(), C.c_int()
        self._ck(self.lib.p2p_upload_pano_jpeg(self.ctx, slot, data, len(data), C.byref(w), C.byref(h)))
        return w.value, h.value

    def decode_jpeg(self, data: bytes, slot: int | None = None) -> np.ndarray:
        """The array ``cv2.imdecode(data, cv2.IMREAD_COLOR)`` returns (u8 [H, W, 3], BGR), decoded on the device."""
        dims = self.jpeg_probe(data)
        if dims is None:
            raise P2PError(-6, "JPEG file outside the supported subset (fall back to cv2.imread)")
        W, H = dims
        out = np.empty((H, W, 3), np.uint8)

        def run(s):
            self._ck(self.lib.p2p_decode_jpeg(self.ctx, s, data, len(data), out.ctypes.data, out.strides[0], H))

        if slot is None:
            with self.slots(1) as (s,):
                run(s)
        else:
            run(slot)
        return out

    # -- PNG panoramas decoded on the device (the decode side of cv2.imread for .png inputs, ref :244) ----------
    def png_probe(self, data: bytes):
        """(W, H) if the device decoder accepts this file's structure with this context's ``P2P_OPT_PNG_FORMATS``, else
        None (read it with cv2.imread)."""
        return png_probe(data, self.png_formats)

    def upload_png(self, slot: int, data: bytes) -> tuple:
        """Decode a PNG file into ``slot`` as its panorama (inflate, unfilter and packing on the device); returns (Wp, Hp).
        Raises ``P2PError`` with code -6 for files outside the supported subset or damaged files."""
        w, h = C.c_int(), C.c_int()
        self._ck(self.lib.p2p_upload_pano_png(self.ctx, slot, data, len(data), C.byref(w), C.byref(h)))
        return w.value, h.value

    def decode_png(self, data: bytes, slot: int | None = None) -> np.ndarray:
        """The array ``cv2.imdecode(data, cv2.IMREAD_COLOR)`` returns (u8 [H, W, 3], BGR), decoded on the device."""
        dims = png_probe(data, self.png_formats)
        if dims is None:
            raise P2PError(-6, "PNG file outside the supported subset (fall back to cv2.imread)")
        W, H = dims
        out = np.empty((H, W, 3), np.uint8)

        def run(s):
            self._ck(self.lib.p2p_decode_png(self.ctx, s, data, len(data), out.ctypes.data, out.strides[0], H))

        if slot is None:
            with self.slots(1) as (s,):
                run(s)
        else:
            run(slot)
        return out

    # -- either kind of file, chosen by its signature --------------------------------------------------------
    def upload_encoded(self, slot: int, data: bytes) -> tuple:
        """``upload_png`` for a PNG signature, else ``upload_jpeg``."""
        return self.upload_png(slot, data) if data[:8] == b"\x89PNG\r\n\x1a\n" else self.upload_jpeg(slot, data)

    def decode_encoded(self, data: bytes, slot: int | None = None) -> np.ndarray:
        """``decode_png`` for a PNG signature, else ``decode_jpeg``."""
        return self.decode_png(data, slot) if data[:8] == b"\x89PNG\r\n\x1a\n" else self.decode_jpeg(data, slot)

    def view_row_range(self, consts, W: int, H: int, Wp: int, Hp: int) -> tuple:
        """(first, last) panorama row (inclusive) the sampler reads for these pitch constants: what
        ``process_image`` transfers over PCIe (any yaw, any image; memoised per geometry)."""
        pc = self._consts_array(consts)
        a, b = C.c_int(), C.c_int()
        self._ck(self.lib.p2p_view_row_range(self.ctx, len(consts), pc, W, H, Wp, Hp, C.byref(a), C.byref(b)))
        return a.value, b.value

    # -- debug exports ------------------------------------------------------------------------
    def coords(self, W, H, fov_deg, pitch_deg, Wp, Hp):
        pc = self._consts_array([pitch_constants(W, fov_deg, pitch_deg)])
        U = np.empty((H, W), np.float32)
        V = np.empty((H, W), np.float32)
        self._ck(self.lib.p2p_coords(self.ctx, pc, W, H, Wp, Hp,
                                     U.ctypes.data_as(C.POINTER(C.c_float)), V.ctypes.data_as(C.POINTER(C.c_float))))
        return U, V

    def selftest(self, W, H, fov_deg, pitch_deg, exhaustive_div=False):
        """(ray_mismatches, div_mismatches) of the fast IEEE sequences vs the generic intrinsics."""
        pc = self._consts_array([pitch_constants(W, fov_deg, pitch_deg)])
        a, b = C.c_ulonglong(), C.c_ulonglong()
        self._ck(self.lib.p2p_selftest(self.ctx, pc, W, H, 1 if exhaustive_div else 0, C.byref(a), C.byref(b)))
        return a.value, b.value

    def sample_with_maps(self, slot: int, yaw_shift: int, U: np.ndarray, V: np.ndarray) -> np.ndarray:
        U = np.ascontiguousarray(U, np.float32)
        V = np.ascontiguousarray(V, np.float32)
        H, W = U.shape
        out = np.empty((H, W, 3), np.uint8)
        self._ck(self.lib.p2p_sample_with_maps(self.ctx, slot, int(yaw_shift),
                                               U.ctypes.data_as(C.POINTER(C.c_float)),
                                               V.ctypes.data_as(C.POINTER(C.c_float)), W, H, out.ctypes.data))
        return out

    def download_pano(self, slot: int, Wp: int, Hp: int) -> np.ndarray:
        out = np.empty((Hp, Wp, 3), np.uint8)
        self._ck(self.lib.p2p_download_pano(self.ctx, slot, out.ctypes.data, out.strides[0]))
        return out

    # -- events -------------------------------------------------------------------------------
    def event(self):
        e = C.c_void_p()
        self._ck(self.lib.p2p_event_create(self.ctx, C.byref(e)))
        return e

    def record(self, ev, slot: int):
        self._ck(self.lib.p2p_event_record(self.ctx, ev, slot))

    def event_wait(self, ev, slot: int):
        """Work enqueued on ``slot`` from now on waits for ``ev`` (fork / join of slot streams)."""
        self._ck(self.lib.p2p_event_wait(self.ctx, ev, slot))

    def elapsed_ms(self, start, stop) -> float:
        ms = C.c_float()
        self._ck(self.lib.p2p_event_elapsed_ms(self.ctx, start, stop, C.byref(ms)))
        return ms.value

    def set_stream(self, slot: int, stream_ptr: int):
        self._ck(self.lib.p2p_set_stream(self.ctx, slot, C.c_void_p(stream_ptr)))

    def get_stream(self, slot: int) -> int:
        st = C.c_void_p()
        self._ck(self.lib.p2p_get_stream(self.ctx, slot, C.byref(st)))
        return st.value or 0

    def share_stream(self, slots, from_slot: int = 0):
        """Run several slots on one stream (serialised launches, e.g. for event timing)."""
        st = self.get_stream(from_slot)
        for s in slots:
            if s != from_slot:
                self.set_stream(s, st)

    def flush_l2(self, slot: int, nbytes: int):
        self._ck(self.lib.p2p_flush_l2(self.ctx, slot, nbytes))

    # -- the batched hot path -------------------------------------------------------------------
    def project_image(self, pano: np.ndarray, yaw_angles, pitch_angles, W: int, H: int, fov_deg=90,
                      out: np.ndarray | None = None, consts=None, tables=None) -> np.ndarray:
        """All yaw x pitch views of one panorama: u8 [n_yaw, n_pitch, H, W, 3].

        Replaces the reference's per-image fan-out (ref :252-265): every yaw that is an integer
        column roll goes into one batched launch; the fractional yaws go into a second one that evaluates the
        reference's yaw remap (ref :191-199) per output pixel instead of materialising a rotated panorama.
        ``consts`` / ``tables`` let a caller pass memoised host scalars (the mirror module's caches).
        """
        pano = _as_u8_image(pano)
        Hp, Wp, _ = pano.shape
        yaw_angles = list(yaw_angles)
        pitch_angles = list(pitch_angles)
        if consts is None:
            consts = [pitch_constants(W, fov_deg, p) for p in pitch_angles]
        if tables is None:
            tables = [yaw_table(Wp, y) for y in yaw_angles]
        shape = (len(yaw_angles), len(pitch_angles), H, W, 3)
        if out is None:
            out = np.empty(shape, np.uint8)
        elif out.shape != shape or out.dtype != np.uint8 or not out.flags.c_contiguous:
            raise ValueError(f"out must be C-contiguous uint8 {shape}")
        if not yaw_angles or not pitch_angles:
            return out
        with self.slots(1) as (src,):
            self.upload(src, pano)
            self.project_any(src, tables, consts, W, H, out)
        return out
