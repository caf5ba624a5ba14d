"""Wall time of the directory front end on folders of 8192x4096 JPEG panoramas (12 x 1920x1080 views each), GPU flow only:
    python tools/time_folder.py [--files 32 256] [--repeat 3] [--devices 1 2 4 8] [--one-gpu-processes 2 4]
                                [--formats jpg png] [--out FILE]
(tools/cpu_baselines.py times the reference's flow beside it).  For every folder size, output format and device list
(``[0 .. n-1]`` for every GPU count n of ``--devices`` the box has, and ``[0] * k`` - k worker processes sharing GPU 0 -
for every k of ``--one-gpu-processes``):
* warm: ``main(devices=...)`` in this process, the product's own multi-GPU front end - one worker process per list entry
  when the list has two or more (kept between the repeats, so only the first pass pays process start-up and CUDA context
  creation), in-process for one; the output files of every run are hashed and must equal the first run's;
* cold: the command line (``python -m 360-to-planer-images_b200 ... --devices ...``) as a subprocess, wall time from
  start to exit, start-up included - what a user sees.
Inputs and outputs live in /dev/shm.  The folders of 256 files repeat the 32 distinct panoramas (8 copies each, other
names).  The first line names the GPUs (``nvidia-smi``: name, power limit, max SM clock) the numbers were taken on."""
import argparse
import hashlib
import importlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools import synth_inputs as synth  # noqa: E402

YAWS, PITCHES, W, H, FOV = [0, 90, 180, 270], [30, 60, 90], 1920, 1080, 120
DISTINCT = 32


def gpus():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout
    return [dict(zip(("name", "power_limit", "max_sm_clock"), (v.strip() for v in line.split(","))))
            for line in q.strip().splitlines()]


def digest(out: Path):
    h, nbytes, count = hashlib.sha256(), 0, 0
    for f in sorted(out.iterdir()):
        data = f.read_bytes()
        h.update(f.name.encode())
        h.update(data)
        nbytes += len(data)
        count += 1
    return h.hexdigest(), nbytes, count


def main():
    import cv2

    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, nargs="+", default=[32, 256])
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--workers", type=int, default=max(1, int((os.cpu_count() or 1) * 0.9)))
    ap.add_argument("--devices", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--one-gpu-processes", type=int, nargs="*", default=[2, 4])
    ap.add_argument("--formats", nargs="+", default=["jpg", "png"])
    ap.add_argument("--no-cold", dest="cold", action="store_false")
    ap.add_argument("--out", type=str, default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    sink = open(a.out, "a") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
            sink.flush()

    pkg = importlib.import_module("360-to-planer-images_b200")
    n_avail = pkg._lib.load().p2p_device_count()
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else None
    emit({"gpus": gpus(), "devices_available": n_avail, "host_cpus": os.cpu_count(), "workers": a.workers,
          "tmp": shm, "tmp_free_gb": round(shutil.disk_usage(shm or tempfile.gettempdir()).free / 2 ** 30, 1)})
    td = Path(tempfile.mkdtemp(dir=shm))
    try:
        distinct = td / "distinct"
        distinct.mkdir()
        for i in range(min(DISTINCT, max(a.files))):
            cv2.imwrite(str(distinct / f"p{i}.jpg"), synth.smooth(8192, 4096, 100 + i))
        src = sorted(distinct.iterdir())
        for n_files in a.files:
            folder = td / f"in{n_files}"
            folder.mkdir()
            for i in range(n_files):
                shutil.copyfile(src[i % len(src)], folder / f"p{i}.jpg")
            for fmt in a.formats:
                first_hash = None
                label = f"{n_files} x 8192x4096 jpg -> {n_files * 12} x 1920x1080 {fmt}"
                lists = [list(range(n)) for n in a.devices if n <= n_avail] + [[0] * k for k in a.one_gpu_processes]
                for dev_list in lists:
                    n_dev, devs = len(set(dev_list)), (dev_list if len(dev_list) > 1 else None)
                    times, same = [], True
                    for r in range(a.repeat + 1):        # the first pass warms processes, slots and buffers
                        out = td / "out"
                        t0 = time.perf_counter()
                        pkg.main(str(folder), str(out), YAWS, PITCHES, W, H, num_workers=a.workers, output_format=fmt,
                                 fov_deg=FOV, devices=devs)
                        times.append(time.perf_counter() - t0)
                        h, nbytes, count = digest(out)
                        shutil.rmtree(out)
                        first_hash = first_hash or h
                        same = same and h == first_hash and count == n_files * 12
                    best = min(times[1:])
                    emit({"kind": "warm", "folder": label, "n_gpus": n_dev, "processes": len(dev_list), "workers": a.workers,
                          "warmup_s": round(times[0], 3), "seconds": [round(t, 4) for t in times[1:]],
                          "ms_per_image": round(best / n_files * 1e3, 3),
                          "ms_per_image_per_gpu": round(best / n_files * 1e3 * n_dev, 3),
                          "mpix_s": round(n_files * 12 * W * H / best / 1e6, 1), "output_bytes": nbytes,
                          "files_identical_to_first_run": same})
                    if not a.cold:
                        continue
                    out = td / "out"
                    cmd = [sys.executable, "-m", "360-to-planer-images_b200", "--input_path", str(folder), "--output_path",
                           str(out), "--output_format", fmt, "--FOV", str(FOV), "--output_width", str(W), "--output_height",
                           str(H), "--yaw_angles", *map(str, YAWS), "--pitch_angles", *map(str, PITCHES), "--num_workers",
                           str(a.workers), "--devices", *map(str, dev_list)]
                    t0 = time.perf_counter()
                    rc = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL).returncode
                    wall = time.perf_counter() - t0
                    h, nbytes, count = digest(out)
                    shutil.rmtree(out)
                    emit({"kind": "cold_cli", "folder": label, "n_gpus": n_dev, "processes": len(dev_list), "workers": a.workers,
                          "returncode": rc, "wall_s": round(wall, 3), "ms_per_image": round(wall / n_files * 1e3, 2),
                          "files_identical_to_first_run": h == first_hash and count == n_files * 12})
        pkg.folder_pool.close_shared()
    finally:
        shutil.rmtree(td, ignore_errors=True)


if __name__ == "__main__":
    main()
