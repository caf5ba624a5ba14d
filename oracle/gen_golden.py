"""Generate the golden vectors under ``tests/golden/`` from the UNMODIFIED reference.
TEST INFRASTRUCTURE - run in the dev container only (it reads ``/root/reference``, which does
not exist on the GPU box; the tests only read the committed fixtures).

    python -m oracle.gen_golden [--full]      # --full also re-hashes the 8K / 16K configs

The reference (``/root/reference/app/panorama_to_plane-pitch.py``) has no tests or fixtures of
its own, so these vectors - outputs of the reference itself, executed here with the library
versions recorded in ``tests/golden/manifest.json`` - are what pins the oracle.

Inputs are never stored: panoramas are regenerated from ``oracle.synth`` (seeded) and their
sha256 is recorded so a drift of the generator is detected.
"""
from __future__ import annotations

import argparse
import hashlib
import importlib.util
import json
import platform
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
REF_FILE = Path("/root/reference/app/panorama_to_plane-pitch.py")

sys.path.insert(0, str(ROOT))
from oracle import golden, synth  # noqa: E402


def load_reference():
    spec = importlib.util.spec_from_file_location("p2p_reference_live", REF_FILE)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ref_views(ref, pano, yaws, pitches, W, H, fov):
    """[n_yaw, n_pitch, H, W, 3] from the reference's own entry point (ref :181-221)."""
    out = np.empty((len(yaws), len(pitches), H, W, 3), dtype=np.uint8)
    for i, yaw in enumerate(yaws):
        for j, img in enumerate(ref.process_yaw_and_pitchs(pano, yaw, list(pitches), W, H, fov)):
            out[i, j] = img
    return out


def ref_maps(ref, pitches, W, H, fov, Wp, Hp):
    U = np.empty((len(pitches), H, W), np.float32)
    V = np.empty_like(U)
    for j, p in enumerate(pitches):
        U[j], V[j] = ref.get_pitch_mapping(W, H, p, Wp, Hp, fov)
    return U, V


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also hash the full-size C2/C4/C5 configs")
    args = ap.parse_args()
    import cv2

    ref = load_reference()
    GOLDEN.mkdir(parents=True, exist_ok=True)
    manifest = {
        "generator": "oracle/gen_golden.py",
        "reference": str(REF_FILE),
        "reference_version": ref.get_version(),
        "numpy": np.__version__,
        "cv2": cv2.__version__,
        "python": platform.python_version(),
        "machine": platform.processor() or platform.machine(),
        "pano_sha256": {},
        "hashes": {},
    }
    old = GOLDEN / "manifest.json"
    if old.exists():
        manifest["hashes"] = json.loads(old.read_text()).get("hashes", {})

    def pano(kind, Wp, Hp, seed=0):
        p = synth.make(kind, Wp, Hp, seed)
        manifest["pano_sha256"][f"{kind}_{Wp}x{Hp}_s{seed}"] = sha(p)
        return p

    # C1: the reference's own CPU-runnable case, full size
    p = pano("noise", 2048, 1024)
    out = ref_views(ref, p, [0], [90], 640, 480, 90)
    np.savez_compressed(GOLDEN / "c1.npz", out=out, yaws=[0], pitches=[90], W=640, H=480, fov=90,
                        Wp=2048, Hp=1024, kind="noise", seed=0)

    # C2 scaled by 1/8: README example shape, 12 views, noise + smooth, with the reference maps
    yaws, pitches = [0, 90, 180, 270], [30, 60, 90]
    W, H, fov, Wp, Hp = 240, 135, 120, 1024, 512
    U, V = ref_maps(ref, pitches, W, H, fov, Wp, Hp)
    golden.save(
        GOLDEN / "c2_small.npz",
        dict(out_noise=ref_views(ref, pano("noise", Wp, Hp), yaws, pitches, W, H, fov),
             out_smooth=ref_views(ref, pano("smooth", Wp, Hp), yaws, pitches, W, H, fov),
             U=U, V=V, yaws=yaws, pitches=pitches, W=W, H=H, fov=fov, Wp=Wp, Hp=Hp, seed=0),
        from_maps=("out_noise", "out_smooth"),
    )

    # C5 scaled: cube faces incl. pole pitches (function-level 0/180 and CLI-legal 1/179)
    views = [(0, 90), (90, 90), (180, 90), (270, 90), (0, 0), (0, 180), (0, 1), (0, 179)]
    W = H = 128
    fov, Wp, Hp = 90, 1024, 512
    p = pano("noise", Wp, Hp)
    outs = np.stack([ref_views(ref, p, [y], [pt], W, H, fov)[0, 0] for y, pt in views])
    upitch = sorted({pt for _, pt in views})
    U, V = ref_maps(ref, upitch, W, H, fov, Wp, Hp)
    np.savez_compressed(GOLDEN / "c5_small.npz", out=outs, views=np.array(views), map_pitches=upitch,
                        U=U, V=V, W=W, H=H, fov=fov, Wp=Wp, Hp=Hp, kind="noise", seed=0)

    # fractional yaws on a non-power-of-two panorama (two-stage interpolation, SURVEY 8f-1)
    yaws, pitches = [30, 1, 359, 77, 360, 45], [60, 120]
    W, H, fov, Wp, Hp = 150, 100, 100, 1000, 500
    p = pano("noise", Wp, Hp)
    rows = np.stack([ref.precompute_yaw_mapping(Wp, 4, y)[0][0] for y in yaws])
    np.savez_compressed(GOLDEN / "frac_yaw.npz", out=ref_views(ref, p, yaws, pitches, W, H, fov),
                        yaw_rows=rows, yaws=yaws, pitches=pitches, W=W, H=H, fov=fov, Wp=Wp, Hp=Hp,
                        kind="noise", seed=0)

    # NaN coordinate -> black pixel (abs(z_rot) > 1 by one ulp), SURVEY App. A special sets
    W, H, fov, Wp, Hp = 640, 480, 90, 2048, 1024
    p = pano("smooth", Wp, Hp)
    out = ref_views(ref, p, [0], [5, 175], W, H, fov)
    U, V = ref_maps(ref, [5, 175], W, H, fov, Wp, Hp)
    nan_px = np.argwhere(np.isnan(U) | np.isnan(V))
    golden.save(GOLDEN / "nan_case.npz", dict(out=out, nan_px=nan_px, yaws=[0], pitches=[5, 175],
                                              W=W, H=H, fov=fov, Wp=Wp, Hp=Hp, kind="smooth", seed=0), dx=("out",))

    if args.full:
        # full-size configs: hashes only (bit-exactness of the CPU oracle at BASELINE sizes)
        p = pano("noise", 8192, 4096)
        o = ref_views(ref, p, [0, 90, 180, 270], [30, 60, 90], 1920, 1080, 120)
        manifest["hashes"]["c2_noise"] = [[sha(o[i, j]) for j in range(3)] for i in range(4)]
        ref.yaw_mapping_cache.clear()
        faces = [(0, 90), (90, 90), (180, 90), (270, 90), (0, 0), (0, 180)]
        manifest["hashes"]["c5_noise"] = [
            sha(ref_views(ref, p, [y], [pt], 2048, 2048, 90)[0, 0]) for y, pt in faces
        ]
        ref.yaw_mapping_cache.clear()
        ref.pitch_mapping_cache.clear()
        del o
        p = pano("noise", 16384, 8192)
        o = ref_views(ref, p, [0], [30, 60, 90], 3840, 2160, 100)
        manifest["hashes"]["c4_noise_yaw0"] = [sha(o[0, j]) for j in range(3)]
        ref.yaw_mapping_cache.clear()
        o = ref_views(ref, p, [90], [60], 3840, 2160, 100)
        manifest["hashes"]["c4_noise_yaw90_pitch60"] = sha(o[0, 0])

    (GOLDEN / "manifest.json").write_text(json.dumps(manifest, indent=1, sort_keys=True) + "\n")
    print("wrote", sorted(x.name for x in GOLDEN.iterdir()))


if __name__ == "__main__":
    main()
