"""PNG panorama decode: cv2.imdecode (libpng + zlib, what cv2.imread does at ref :244) + upload against the device
decoder (parallel inflate + unfilter kernels, csrc/p2p_pngdec.cuh), same files, same pixels (run on the GPU box).

    python tools/bench_pngdec.py [--small] > gpurun_out/pngdec_bench.jsonl
    python tools/bench_pngdec.py --formats extended > profiles/r3_png_decoder_ext_bench.jsonl

--formats extended: the files only the wider subset takes (P2P_OPT_PNG_FORMATS = 1): 16-bit RGB written by cv2.imwrite, 8-bit
RGB Adam7 with adaptive filters at zlib level 6, 8-bit palette; the card's name and power limit are recorded in the same run.
"""
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402
sys.path.insert(0, str(ROOT / "tests"))
import png_formats_model as X  # noqa: E402
from tools import synth_inputs as synth  # noqa: E402


def card() -> dict:
    """Name and power limit of GPU 0 (a read-only query)."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, sm = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": sm}
    except Exception as e:   # (no nvidia-smi: the name at least)
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({type(e).__name__})"}


def main():
    import cv2

    g.build()
    pkg = g.load_package()
    proj = pkg.Projector(0, n_slots=2)
    extended = "--formats" in sys.argv and sys.argv[sys.argv.index("--formats") + 1] == "extended"
    Wp, Hp = (2048, 1024) if "--small" in sys.argv else (8192, 4096)
    reps = 1 if "--once" in sys.argv else 4   # --once: a single decode per file (under ncu)
    rng = np.random.default_rng(0)
    smooth = synth.smooth(Wp, Hp, 0)
    textured = np.clip(smooth.astype(np.int16) + rng.integers(-12, 13, smooth.shape, dtype=np.int16), 0, 255).astype(np.uint8)
    P = cv2
    cases = [
        ("textured, cv2.imwrite defaults (the reference's own output format: filter Sub, Z_RLE, level 1)", textured, []),
        ("textured, zlib level 6 default strategy", textured, [P.IMWRITE_PNG_STRATEGY, P.IMWRITE_PNG_STRATEGY_DEFAULT, P.IMWRITE_PNG_COMPRESSION, 6]),
        ("smooth, cv2.imwrite defaults", smooth, []),
    ]
    if extended:
        proj.set_option(pkg._lib.OPT_PNG_FORMATS, 1)
        print(json.dumps(card()), flush=True)
        pal = rng.integers(0, 256, (256, 3), dtype=np.uint8)
        idx = ((textured[:, :, 0].astype(np.uint16) + textured[:, :, 1]) // 2).astype(np.uint8)
        cases = [
            ("16-bit RGB, cv2.imwrite defaults", None, cv2.imencode(".png", textured.astype(np.uint16) * 257)[1].tobytes()),
            ("8-bit RGB Adam7, adaptive filters, zlib level 6", None,
             X.write_png(np.ascontiguousarray(textured[:, :, ::-1]), 2, interlace=1, level=6)),
            ("8-bit palette (256 entries), adaptive filters, zlib level 6", None, X.write_png(idx, 3, palette=pal, level=6)),
        ]
    for name, img, params in cases:
        data = cv2.imencode(".png", img, params)[1].tobytes() if img is not None else params
        arr = np.frombuffer(data, np.uint8)
        ref = cv2.imdecode(arr, cv2.IMREAD_COLOR)
        with proj.slots(1) as (s,):
            try:
                proj.upload_png(s, data)
            except pkg.P2PError as e:
                print(json.dumps({"panorama": name, "file_MB": len(data) / 1e6, "declined": str(e)}), flush=True)
                continue
            proj.sync(s)
            same = bool(np.array_equal(proj.download_pano(s, Wp, Hp), ref))
            t_dev = []
            for _ in range(reps):
                t0 = time.perf_counter()
                proj.upload_png(s, data)
                proj.sync(s)
                t_dev.append(time.perf_counter() - t0)
            t_cv = []
            for _ in range(1 if reps == 1 else 2):
                t0 = time.perf_counter()
                pix = cv2.imdecode(arr, cv2.IMREAD_COLOR)
                proj.upload(s, pix)
                proj.sync(s)
                t_cv.append(time.perf_counter() - t0)
        print(json.dumps({"panorama": name, "size": [Wp, Hp], "file_MB": len(data) / 1e6, "same_pixels_as_cv2": same,
                          "device_decoder_ms": min(t_dev) * 1e3, "device_decoder_ms_all": [round(t * 1e3, 2) for t in t_dev],
                          "cv2_imdecode_plus_upload_ms": min(t_cv) * 1e3, "speedup": min(t_cv) / min(t_dev)}), flush=True)
    proj.close()


if __name__ == "__main__":
    main()
