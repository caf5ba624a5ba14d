"""Fractional yaws on the bench geometry (8192 x 4096 panorama, fov 120, 1920 x 1080, yaws 0 .. 330 in 30 degree steps x
pitches 30 / 60 / 90: at Wp = 8192 only 0 / 90 / 180 / 270 are integer column rolls, the other eight yaws are column
tables).  The earlier route and the view-list route alternate in one run and their outputs are compared:
  * kernel time, CUDA events on one slot, device outputs (the packed panorama, 128 MB, does not fit the L2 whole):
      old: project (integer rolls) + host sync + project_tables (fractional yaws) - what project_any did before;
      new: one project_list_tables call;  and the fractional-only subset: project_tables against project_list_tables;
  * files flow, JPEG panorama file in -> .jpg / .png files out, ms per image (host clock around whole calls):
      old: decode_encoded -> project_image_jpeg / project_image + encode_png (pixels cross PCIe three times);
      new: the front end's view-list route (decoded into the slot, only the files come back);
    single image, and process_image_batch over 16 files (the old route patched into the front end).
    python tools/time_fractional_lists.py [--out profiles/r6_fractional_lists.jsonl]
"""
import argparse
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402
from tools import synth_inputs as synth  # noqa: E402

WP, HP, W, H, FOV = 8192, 4096, 1920, 1080, 120
YAWS, PITCHES = list(range(0, 360, 30)), [30, 60, 90]
REPS, FILE_REPS, BATCH = 20, 5, 16


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r6_fractional_lists.jsonl"))
    ap.add_argument("--kernel-only", action="store_true", help="only the kernel timings (no files flows)")
    args = ap.parse_args()
    import cv2
    import numpy as np
    import torch

    g.build()
    pkg = g.load_package()
    front = sys.modules["p2p_b200.panorama_to_plane_pitch"]
    proj = pkg.get_projector(0)
    card = gpu_name()
    rows = []

    def emit(rec):
        rec["gpu"] = card
        rows.append(rec)
        print(json.dumps(rec), flush=True)

    tables = [pkg.yaw_table(WP, y) for y in YAWS]
    consts = [pkg.pitch_constants(W, FOV, p) for p in PITCHES]
    roll = [k for k, t in enumerate(tables) if t[2] is not None]
    frac = [k for k, t in enumerate(tables) if t[2] is None]
    n_p = len(PITCHES)
    # ---- kernel time ------------------------------------------------------------------------------------------
    d_roll = torch.empty((len(roll), n_p, H, W, 3), dtype=torch.uint8, device="cuda:0")
    d_frac = torch.empty((len(frac), n_p, H, W, 3), dtype=torch.uint8, device="cuda:0")
    d_new = torch.empty((len(YAWS), n_p, H, W, 3), dtype=torch.uint8, device="cuda:0")
    d_fnew = torch.empty((len(frac), n_p, H, W, 3), dtype=torch.uint8, device="cuda:0")
    flat_t = [t for t in tables for _ in consts]
    flat_c = consts * len(tables)
    fflat_t = [tables[k] for k in frac for _ in consts]
    fflat_c = consts * len(frac)
    with proj.slots(1) as (s,):
        proj.upload(s, synth.noise(WP, HP, 0))
        proj.sync(s)
        ev0, ev1 = proj.event(), proj.event()

        def timed(fn):
            proj.record(ev0, s)
            fn()
            proj.record(ev1, s)
            return proj.elapsed_ms(ev0, ev1)

        def old_mixed():
            proj.project(s, [tables[k][2] for k in roll], consts, W, H, out_device_ptr=d_roll.data_ptr())
            proj.sync(s)
            proj.project_tables(s, [tables[k] for k in frac], consts, W, H, out_device_ptr=d_frac.data_ptr())

        routes = {
            "mixed_old": old_mixed,
            "mixed_new": lambda: proj.project_list_tables(s, flat_t, flat_c, W, H, out_device_ptr=d_new.data_ptr()),
            "frac_only_old": lambda: proj.project_tables(s, [tables[k] for k in frac], consts, W, H,
                                                         out_device_ptr=d_frac.data_ptr()),
            "frac_only_new": lambda: proj.project_list_tables(s, fflat_t, fflat_c, W, H, out_device_ptr=d_fnew.data_ptr()),
        }
        for fn in routes.values():   # warm-up: modules, texture, table buffers
            timed(fn)
        t = {k: [] for k in routes}
        for _ in range(REPS):
            for k, fn in routes.items():
                t[k].append(timed(fn))
        proj.sync(s)
        same = bool(torch.equal(d_new[roll], d_roll) and torch.equal(d_new[frac], d_frac) and torch.equal(d_fnew, d_frac))
    for what in ("mixed", "frac_only"):
        o, n = statistics.median(t[f"{what}_old"]), statistics.median(t[f"{what}_new"])
        emit({"metric": f"kernel_ms_{what}", "views": (len(YAWS) if what == "mixed" else len(frac)) * n_p,
              "old_ms": round(o, 4), "new_ms": round(n, 4), "speedup": round(o / n, 3), "reps": REPS,
              "old_ms_all": [round(x, 4) for x in t[f"{what}_old"]], "new_ms_all": [round(x, 4) for x in t[f"{what}_new"]],
              "outputs_equal": same})
    del d_roll, d_frac, d_new, d_fnew
    torch.cuda.empty_cache()
    if args.kernel_only:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in rows))
        return
    # ---- files flow ---------------------------------------------------------------------------------------------
    tmp = Path(tempfile.mkdtemp(prefix="p2p_frac_"))
    data = cv2.imencode(".jpg", synth.smooth(WP, HP, 1))[1].tobytes()
    src_file = tmp / "pano.jpg"
    src_file.write_bytes(data)

    def old_files(fmt, src):
        pix = proj.decode_encoded(src.data)
        if fmt == "jpg":
            return [f for per in proj.project_image_jpeg(pix, YAWS, PITCHES, W, H, FOV) for f in per], None
        views = proj.project_image(pix, YAWS, PITCHES, W, H, FOV)
        return proj.encode_png(views.reshape(-1, H, W, 3)), views

    def new_files(fmt, src):
        files, views = front._project_files(fmt, proj, src, YAWS, PITCHES, W, H, FOV, devices=[])
        return [f for per in files for f in per], views

    src = front._open_image(src_file)
    assert isinstance(src, front._JpegSource)
    for fmt in ("jpg", "png"):
        res = {}
        ts = {"old": [], "new": []}
        for rep in range(FILE_REPS + 1):
            for name, fn in (("old", old_files), ("new", new_files)):
                t0 = time.perf_counter()
                res[name] = fn(fmt, src)[0]
                dt = (time.perf_counter() - t0) * 1e3
                if rep:
                    ts[name].append(dt)
        o, n = statistics.median(ts["old"]), statistics.median(ts["new"])
        emit({"metric": f"files_flow_single_ms_per_image_{fmt}", "input": "jpg 8192x4096", "views": len(YAWS) * n_p,
              "old_ms": round(o, 2), "new_ms": round(n, 2), "speedup": round(o / n, 3), "reps": FILE_REPS,
              "files_equal": res["old"] == res["new"]})
    # process_image_batch over BATCH files: the parent's fractional route patched into the front end for "old"
    folder = tmp / "in"
    folder.mkdir()
    for i in range(BATCH):
        (folder / f"p{i:02d}.jpg").write_bytes(data)
    files = sorted(folder.iterdir())
    new_route = front._project_files

    def old_route(fmt, proj_, src_, yaws, pitches, W_, H_, fov, lease=None, devices=None):
        flat, views = old_files(fmt, src_)
        return [flat[k * n_p:(k + 1) * n_p] for k in range(len(yaws))], views

    for fmt in ("jpg", "png"):
        ts = {"old": [], "new": []}
        outs = {}
        for rep in range(3):
            for name, route in (("old", old_route), ("new", new_route)):
                out = tmp / f"out_{fmt}_{name}"
                if out.exists():
                    subprocess.run(["rm", "-rf", str(out)], check=True)
                out.mkdir()
                front._project_files = route
                try:
                    t0 = time.perf_counter()
                    pkg.process_image_batch(files, out, YAWS, PITCHES, W, H, num_workers=8, output_format=fmt, fov_deg=FOV)
                    ts[name].append((time.perf_counter() - t0) * 1e3 / BATCH)
                finally:
                    front._project_files = new_route
                outs[name] = out
        same = all((outs["old"] / p.name).read_bytes() == p.read_bytes() for p in outs["new"].iterdir())
        same = same and len(list(outs["new"].iterdir())) == BATCH * len(YAWS) * n_p
        o, n = statistics.median(ts["old"]), statistics.median(ts["new"])
        emit({"metric": f"files_flow_batch_ms_per_image_{fmt}", "input": f"{BATCH} x jpg 8192x4096",
              "views_per_image": len(YAWS) * n_p, "old_ms": round(o, 2), "new_ms": round(n, 2), "speedup": round(o / n, 3),
              "reps": 3, "old_ms_all": [round(x, 2) for x in ts["old"]], "new_ms_all": [round(x, 2) for x in ts["new"]],
              "files_equal": same})
    subprocess.run(["rm", "-rf", str(tmp)], check=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in rows))


if __name__ == "__main__":
    main()
