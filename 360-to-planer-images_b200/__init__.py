"""B200-native drop-in for the projection hot path of Maxiviper117/360-to-planer-images.

The directory name follows the repo contract (``360-to-planer-images_b200``) and is not a valid
Python identifier; load it through ``__graft_entry__.load_package()`` (registers it as the module
``p2p_b200``) or ``importlib`` with ``submodule_search_locations``.

Public surface (mirrors ``app/panorama_to_plane-pitch.py`` of the reference):
``panorama_to_plane``, ``process_yaw_and_pitchs``, ``process_single_image``, ``main``,
``check_pitch``, ``get_version`` and the device-level ``Projector``.
Importing this package loads ``libp2p_b200.so``; it raises if the library is not built.
"""
from . import _lib

_lib.load()  # fail loudly: no CPU fallback

from . import folder_pool  # noqa: E402,F401
from .engine import PinnedBuffer, Projector, host_assumptions, pitch_constants, warn_if_host_differs, yaw_table  # noqa: E402
from .panorama_to_plane_pitch import (  # noqa: E402
    check_pitch,
    cli,
    get_pitch_mapping,
    get_projector,
    get_version,
    get_yaw_mapping,
    main,
    panorama_to_plane,
    pitch_mapping_cache,
    process_image_batch,
    process_single_image,
    process_yaw_and_pitchs,
    scatter_upload,
    set_device,
    set_devices,
    set_png_formats,
    yaw_mapping_cache,
)
from ._lib import P2PError, PitchConsts  # noqa: E402

__all__ = [
    "panorama_to_plane", "process_yaw_and_pitchs", "process_single_image", "process_image_batch", "main", "check_pitch",
    "get_version", "cli", "Projector", "PinnedBuffer", "pitch_constants", "yaw_table", "P2PError",
]
