"""ctypes binding of ``libp2p_b200.so`` (C ABI declared in ``include/p2p.h``).

There is no CPU fallback: if the shared library has not been built (``__graft_entry__.build()``
or ``python 360-to-planer-images_b200/build.py``) importing the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libp2p_b200.so"


class PitchConsts(C.Structure):
    """``p2p_pitch_consts``: f32 focal length, cos(pitch), sin(pitch)."""

    _fields_ = [("f", C.c_float), ("c", C.c_float), ("s", C.c_float)]


class P2PError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"p2p error {code}: {msg}")
        self.code, self.msg = code, msg

    def __reduce__(self):   # pickles with its code: a folder worker process's error is raised again in the caller
        return type(self), (self.code, self.msg), self.__dict__


# every symbol include/p2p.h declares: name -> (restype, argtypes)
_vp, _i, _sz, _u8p = C.c_void_p, C.c_int, C.c_size_t, C.c_void_p
_i32p, _f32p = C.POINTER(C.c_int32), C.POINTER(C.c_float)
_pcp = C.POINTER(PitchConsts)
SIGNATURES = {
    "p2p_abi_version": (_i, []),
    "p2p_device_count": (_i, []),
    "p2p_create": (_i, [_i, _i, C.POINTER(_vp)]),
    "p2p_destroy": (None, [_vp]),
    "p2p_last_error": (C.c_char_p, [_vp]),
    "p2p_status_string": (C.c_char_p, [_i]),
    "p2p_set_option": (_i, [_vp, _i, _i]),
    "p2p_get_option": (_i, [_vp, _i, C.POINTER(_i)]),
    "p2p_pitch_constants": (_i, [C.c_double, C.c_double, _i, _pcp]),
    "p2p_yaw_table": (_i, [_i, C.c_double, _i32p, _i32p, _i32p]),
    "p2p_host_alloc": (_i, [C.POINTER(_vp), _sz]),
    "p2p_host_free": (_i, [_vp]),
    "p2p_host_register": (_i, [_vp, _sz]),
    "p2p_host_unregister": (_i, [_vp]),
    "p2p_upload_pano": (_i, [_vp, _i, _u8p, _i, _i, _sz]),
    "p2p_upload_pano_device": (_i, [_vp, _i, _vp, _i, _i, _sz]),
    "p2p_rotate_pano": (_i, [_vp, _i, _i, _i32p, _i32p]),
    "p2p_project_views": (_i, [_vp, _i, _i, _i32p, _i, _pcp, _i, _i, _u8p, _i]),
    "p2p_project_views_table": (_i, [_vp, _i, _i, C.POINTER(_i32p), C.POINTER(_i32p), _i, _pcp, _i, _i, _u8p, _i]),
    "p2p_project_batch": (_i, [_vp, _i, _i32p, _i, _i32p, _i, _pcp, _i, _i, C.POINTER(_vp), _i]),
    "p2p_project_view_list": (_i, [_vp, _i, _i, _i32p, _pcp, _i, _i, _i, _i, _u8p, _i]),
    "p2p_project_view_list_tables": (_i, [_vp, _i, _i, _i32p, C.POINTER(_i32p), C.POINTER(_i32p), _pcp, _i, _i, _i, _i,
                                          _u8p, _i]),
    "p2p_process_view_list_jpeg": (_i, [_vp, _i, _u8p, _i, _i, _sz, _i, _i32p, C.POINTER(_i32p), C.POINTER(_i32p), _pcp,
                                        _i, _i, _i, _u8p, _sz, C.POINTER(_sz)]),
    "p2p_process_view_list_png": (_i, [_vp, _i, _u8p, _i, _i, _sz, _i, _i32p, C.POINTER(_i32p), C.POINTER(_i32p), _pcp,
                                       _i, _i, _u8p, _sz, C.POINTER(_sz), _u8p]),
    "p2p_copy_pano": (_i, [_vp, _i, _vp, _i]),
    "p2p_upload_pano_rows": (_i, [_vp, _i, _u8p, _i, _i, _sz, _i, _i]),
    "p2p_copy_pano_rows": (_i, [_vp, _i, _vp, _i, _i, _i]),
    "p2p_process_image": (_i, [_vp, _i, _u8p, _i, _i, _sz, _i, _i32p, _i, _pcp, _i, _i, _u8p]),
    "p2p_view_row_range": (_i, [_vp, _i, _pcp, _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "p2p_encode_jpeg": (_i, [_vp, _i, _u8p, _i, _i, _i, _i, _i, _u8p, _sz, C.POINTER(_sz)]),
    "p2p_project_views_jpeg": (_i, [_vp, _i, _i, _i32p, _i, _pcp, _i, _i, _i, _u8p, _sz, C.POINTER(_sz)]),
    "p2p_process_image_jpeg": (_i, [_vp, _i, _u8p, _i, _i, _sz, _i, _i32p, _i, _pcp, _i, _i, _i, _u8p, _sz, C.POINTER(_sz)]),
    "p2p_encode_png": (_i, [_vp, _i, _u8p, _i, _i, _i, _i, _u8p, _sz, C.POINTER(_sz)]),
    "p2p_process_image_png": (_i, [_vp, _i, _u8p, _i, _i, _sz, _i, _i32p, _i, _pcp, _i, _i, _u8p, _sz, C.POINTER(_sz), _u8p]),
    "p2p_jpeg_probe": (_i, [_u8p, _sz, C.POINTER(_i), C.POINTER(_i)]),
    "p2p_jpeg_coefficients": (_i, [_u8p, _sz, _vp, _sz, _i32p]),
    "p2p_jpeg_device_tables": (_i, [_u8p, _sz, _vp, _sz, _i32p]),
    "p2p_upload_pano_jpeg": (_i, [_vp, _i, _u8p, _sz, C.POINTER(_i), C.POINTER(_i)]),
    "p2p_decode_jpeg": (_i, [_vp, _i, _u8p, _sz, _u8p, _sz, _sz]),
    "p2p_png_probe": (_i, [_u8p, _sz, C.POINTER(_i), C.POINTER(_i)]),
    "p2p_png_decode_host": (_i, [_u8p, _sz, _u8p, _sz, _sz, C.POINTER(C.c_uint64)]),
    "p2p_png_probe_ex": (_i, [_u8p, _sz, _i, C.POINTER(_i), C.POINTER(_i)]),
    "p2p_png_decode_host_ex": (_i, [_u8p, _sz, _i, _u8p, _sz, _sz, C.POINTER(C.c_uint64)]),
    "p2p_upload_pano_png": (_i, [_vp, _i, _u8p, _sz, C.POINTER(_i), C.POINTER(_i)]),
    "p2p_decode_png": (_i, [_vp, _i, _u8p, _sz, _u8p, _sz, _sz]),
    "p2p_sync": (_i, [_vp, _i]),
    "p2p_set_stream": (_i, [_vp, _i, _vp]),
    "p2p_get_stream": (_i, [_vp, _i, C.POINTER(_vp)]),
    "p2p_event_create": (_i, [_vp, C.POINTER(_vp)]),
    "p2p_event_destroy": (_i, [_vp, _vp]),
    "p2p_event_record": (_i, [_vp, _vp, _i]),
    "p2p_event_wait": (_i, [_vp, _vp, _i]),
    "p2p_event_elapsed_ms": (_i, [_vp, _vp, _vp, _f32p]),
    "p2p_flush_l2": (_i, [_vp, _i, _sz]),
    "p2p_selftest": (_i, [_vp, _pcp, _i, _i, _i, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "p2p_coords": (_i, [_vp, _pcp, _i, _i, _i, _i, _f32p, _f32p]),
    "p2p_sample_with_maps": (_i, [_vp, _i, _i, _f32p, _f32p, _i, _i, _u8p]),
    "p2p_download_pano": (_i, [_vp, _i, _u8p, _sz]),
}

OPT_SAMPLER, OPT_WARP_W, OPT_YAWS_PER_THREAD, OPT_COUNT_LAUNCHES, OPT_IMAGES_PER_LAUNCH, OPT_MIRROR, OPT_INTERP, OPT_TRIG = 0, 1, 2, 3, 4, 5, 6, 7
OPT_PARTIAL_UPLOAD = 8
OPT_GPU_HUFFMAN, OPT_GPU_HUFFMAN_COUNT = 9, 10
OPT_SEG_CHUNKS = 11
OPT_SEAM_WRAP = 12
OPT_HOST_WAIT = 13
OPT_PNG_FORMATS = 14
OPT_PNG_HOST_BLOCKS = 15

_lib = None


def load() -> C.CDLL:
    """Load the shared library and declare every prototype.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("P2P_B200_LIB", LIB_PATH))
    if not path.exists():
        raise ImportError(
            f"{path} not found: the CUDA library is not built. Run `python -c 'import "
            "__graft_entry__ as g; g.build()'` at the repo root. There is no CPU fallback."
        )
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if lib.p2p_abi_version() != 1:
        raise ImportError(f"{path}: ABI version {lib.p2p_abi_version()} != 1")
    _lib = lib
    return lib
