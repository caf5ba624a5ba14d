"""Quarter-turn sampler on the bench workload (8192 x 4096 panoramas -> 12 x 1920 x 1080, fov 120):
  * device time per image of the README views (yaws 0 / 90 / 180 / 270 x pitches 30 / 60 / 90: three quarter-turn
    groups, read from the yaw-folded planes) against the same launch shape whose yaws are NOT quarter turns apart
    (0 / 90 / 180 / ~271 degrees: column rolls 0, 2048, 4096, 6167 -> the RGBA path), CUDA events, one stream,
    8 distinct resident panoramas in turn;
  * fold_kernel device time per 8K image (torch.profiler, a separate pass: each slot re-packed, then rendered twice;
    a panorama folds on its second quarter-turn render).
    python tools/time_folded.py > folded.jsonl
"""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402
from tools import synth_inputs as synth  # noqa: E402

WP, HP, W, H, FOV = 8192, 4096, 1920, 1080, 120
N_SLOTS, REPS = 8, 20


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    import torch

    g.build()
    pkg = g.load_package()
    proj = pkg.Projector(0, n_slots=N_SLOTS)
    slots = list(range(N_SLOTS))
    proj.share_stream(slots, 0)
    d_src = []
    for i in slots:
        d = torch.from_numpy(synth.noise(WP, HP, i)).cuda()
        d_src.append(d)
        torch.cuda.synchronize()
        proj.upload_device(i, d.data_ptr(), WP, HP, WP * 3)
    proj.sync(-1)
    consts = [pkg.pitch_constants(W, FOV, p) for p in (30, 60, 90)]
    sets = {"quarter_0_90_180_270": [0, 2048, 4096, 6144], "near_quarter_0_90_180_271": [0, 2048, 4096, 6167]}
    d_out = torch.empty((12, H, W, 3), dtype=torch.uint8, device="cuda:0")
    ev0, ev1 = proj.event(), proj.event()
    card = gpu_name()
    for name, shifts in sets.items():
        calls = [proj.batch_call([s], shifts, consts, W, H, [d_out.data_ptr()]) for s in slots]
        for _ in range(3):
            for f in calls:
                f()
        proj.sync(-1)
        proj.record(ev0, 0)
        for _ in range(REPS):
            for f in calls:
                f()
        proj.record(ev1, 0)
        proj.sync(-1)
        us = proj.elapsed_ms(ev0, ev1) / (REPS * N_SLOTS) * 1e3
        print(json.dumps({"views": name, "shifts": shifts, "image_us": us, "images": REPS * N_SLOTS, "gpu": card,
                          "note": "one stream, 8 distinct resident 8K panoramas in turn, 12 views per image"}), flush=True)

    from torch.profiler import ProfilerActivity, profile

    quarter = [proj.batch_call([s], sets["quarter_0_90_180_270"], consts, W, H, [d_out.data_ptr()]) for s in slots]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            for i in slots:
                proj.upload_device(i, d_src[i].data_ptr(), WP, HP, WP * 3)
                quarter[i]()   # first render of the new panorama: RGBA texture
                quarter[i]()   # second: fold, then the folded planes
        proj.sync(-1)
    per = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        for k in ("fold_kernel", "pack_kernel", "project_rows_kernel"):
            if k in e.name:
                t = per.setdefault(k, [0.0, 0])
                t[0] += e.device_time
                t[1] += 1
    print(json.dumps({"kernel_us_per_call": {k: v[0] / v[1] for k, v in per.items()},
                      "calls": {k: v[1] for k, v in per.items()}, "gpu": card,
                      "note": "torch.profiler pass: each 8K slot re-packed (upload_device), then rendered twice "
                              "(RGBA texture; fold + folded planes)"}),
          flush=True)
    proj.close()


if __name__ == "__main__":
    main()
