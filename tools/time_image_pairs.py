"""Resident panoramas rendered one per launch against two per launch (the row-segment kernel's same-stream pairs), on the
bench workload (8192 x 4096 panoramas -> 12 x 1920 x 1080, fov 120, pitches 30 / 60 / 90):
  * single: one p2p_project_batch call per image - an image with no partner keeps its own launch;
  * paired: one call over all 8 images - images on the same stream share launches, two at a time;
for 8 distinct resident panoramas on one launching stream and on two (slot i on the stream of slot i % 2, as bench.py
does), and for two yaw sets: the README yaws 0 / 90 / 180 / 270 (three quarter-turn groups, read from the yaw-folded
planes) and 0 / 90 / 180 / ~271 (column rolls 0, 2048, 4096, 6167: the RGBA path, as in tools/time_folded.py).
Device time per image from CUDA events around REPS passes (fork / join over the launching streams); every line carries
the card's name, power limit and max SM clock.
    python tools/time_image_pairs.py [--label NAME] > pairs.jsonl
P2P_B200_LIB=/path/to/libp2p_b200.so times another build of the library with the same script.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402
from tools import synth_inputs as synth  # noqa: E402

WP, HP, W, H, FOV = 8192, 4096, 1920, 1080, 120
PITCHES = [30, 60, 90]
N_SLOTS, REPS = 8, 20
SETS = {"quarter_0_90_180_270": [0, 2048, 4096, 6144], "near_quarter_0_90_180_271": [0, 2048, 4096, 6167]}


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--label", default="", help="name of the library build, copied into every line")
    args = ap.parse_args()
    import torch

    g.build()
    pkg = g.load_package()
    proj = pkg.Projector(0, n_slots=N_SLOTS)
    slots = list(range(N_SLOTS))
    own = [proj.get_stream(s) for s in slots]
    for i in slots:
        d = torch.from_numpy(synth.noise(WP, HP, i)).cuda()
        torch.cuda.synchronize()
        proj.upload_device(i, d.data_ptr(), WP, HP, WP * 3)
        proj.sync(i)
        del d
    consts = [pkg.pitch_constants(W, FOV, p) for p in PITCHES]
    d_out = torch.empty((N_SLOTS, 12, H, W, 3), dtype=torch.uint8, device="cuda:0")
    ptrs = [d_out[i].data_ptr() for i in slots]
    ev0, ev1 = proj.event(), proj.event()
    ev_join = [proj.event() for _ in range(2)]
    card = gpu_name()
    for n_streams in (1, 2):
        for i in slots:
            proj.set_stream(i, own[i % n_streams])
        for name, shifts in SETS.items():
            for mode in ("single", "paired"):
                if mode == "single":
                    calls = [proj.batch_call([s], shifts, consts, W, H, [ptrs[s]]) for s in slots]
                else:
                    calls = [proj.batch_call(slots, shifts, consts, W, H, ptrs)]
                for _ in range(3):   # the second quarter-turn render of a panorama folds it
                    for f in calls:
                        f()
                proj.sync(-1)
                n0 = proj.launches
                proj.record(ev0, 0)
                for st in range(1, n_streams):
                    proj.event_wait(ev0, st)
                for _ in range(REPS):
                    for f in calls:
                        f()
                for st in range(1, n_streams):
                    proj.record(ev_join[st], st)
                    proj.event_wait(ev_join[st], 0)
                proj.record(ev1, 0)
                proj.sync(-1)
                us = proj.elapsed_ms(ev0, ev1) / (REPS * N_SLOTS) * 1e3
                print(json.dumps({"build": args.label, "views": name, "shifts": shifts, "streams": n_streams,
                                  "mode": mode, "image_us": round(us, 3),
                                  "launches_per_image": (proj.launches - n0) / (REPS * N_SLOTS),
                                  "images": REPS * N_SLOTS, "gpu": card,
                                  "note": f"8 distinct resident 8K panoramas, 12 views each, {n_streams} launching "
                                          "stream(s), CUDA events"}), flush=True)
    for i in slots:
        proj.set_stream(i, own[i])
    proj.close()


if __name__ == "__main__":
    main()
