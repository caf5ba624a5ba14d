"""Reading and writing the golden vectors under ``tests/golden/``.  TEST INFRASTRUCTURE.

A golden file is an ``.npz`` whose arrays ``load`` returns as a dict.  Two encodings keep every file under 1 MB without
dropping a single value of the reference's outputs:

``<name>.dx``      a u8 image stack stored as each pixel minus its left neighbour (mod 256): a smooth image deflates to
                   about a third.  ``load`` restores ``<name>`` with a running sum along the rows.
``<name>.sha256``  views of the file's synthetic panorama (``out_noise`` / ``out_smooth``: the kind follows the name) that
                   ``load`` rebuilds with the cv2.remap model (``fixedpoint``) from the reference's own maps stored in the
                   same file (``U``, ``V`` per pitch), then checks against the sha256 of each view the reference wrote.
                   Noise views do not compress, and the model is integer arithmetic on the stored maps, so the rebuild is
                   the same on every host.
"""
from __future__ import annotations

import hashlib

import numpy as np

from . import fixedpoint, synth


def _sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _views_from_maps(g: dict, name: str) -> np.ndarray:
    """[n_yaw, n_pitch, H, W, 3]: the views of ``synth.make(kind, Wp, Hp, seed)`` sampled at the stored maps."""
    kind = name.rsplit("_", 1)[1]
    Wp, Hp, W, H, fov, seed = (int(g[k]) for k in ("Wp", "Hp", "W", "H", "fov", "seed"))
    pano = synth.make(kind, Wp, Hp, seed)
    return np.stack([np.stack([fixedpoint.project_view_single_pass(pano, int(y), int(p), W, H, fov, coords=(g["U"][j], g["V"][j]))
                               for j, p in enumerate(g["pitches"])]) for y in g["yaws"]])


def load(path) -> dict:
    with np.load(path, allow_pickle=False) as z:
        g = {k: z[k] for k in z.files}
    for key in [k for k in g if k.endswith(".dx")]:
        g[key[:-3]] = np.cumsum(g.pop(key), axis=-2, dtype=np.uint8)
    for key in [k for k in g if k.endswith(".sha256")]:
        name, want = key[:-7], g.pop(key)
        views = _views_from_maps(g, name)
        got = np.array([[_sha(v) for v in row] for row in views])
        if not np.array_equal(got, want):
            raise ValueError(f"{path}: {name} rebuilt from the stored maps is not what the reference wrote "
                             f"(views (yaw index, pitch index) {np.argwhere(got != want).tolist()} differ)")
        g[name] = views
    return g


def save(path, arrays: dict, dx=(), from_maps=()) -> None:
    """``np.savez_compressed`` of ``arrays`` with the names in ``dx`` / ``from_maps`` encoded as described above; the file
    must load back to exactly ``arrays``."""
    enc = {k: v for k, v in arrays.items() if k not in dx and k not in from_maps}
    for k in dx:
        a = np.asarray(arrays[k])
        assert a.dtype == np.uint8 and a.ndim >= 3
        enc[k + ".dx"] = np.diff(a, axis=-2, prepend=np.zeros_like(a[..., :1, :]))
    for k in from_maps:
        enc[k + ".sha256"] = np.array([[_sha(v) for v in row] for row in arrays[k]])
    np.savez_compressed(path, **enc)
    back = load(path)
    assert back.keys() == arrays.keys() and all(np.array_equal(back[k], arrays[k]) for k in arrays), path
