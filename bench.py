#!/usr/bin/env python
"""Headline benchmark: output Mpix/s of the panorama -> plane hot path (8K equirect -> 1920x1080).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this framework (CUDA)
    python bench.py ... --dump-outputs DIR                         # + a fixed sample of the last timed step's outputs
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU reference arm
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W     # N > 1, one rank per GPU

Workload (BASELINE.json configs[1]/[2]): every image is the README example - one synthetic
8192x4096 panorama, FOV 120, 1920x1080, yaw 0/90/180/270 x pitch 30/60/90 = 12 views.  One
"step" processes a batch of 32 such images per GPU (at 8 GPUs that is exactly configs[2], the
256-image batch sharded by image); per-GPU work is fixed, so scaling is weak and needs no
collective - torch.distributed only provides the barrier and the max-over-ranks of the timing.

value    device-resident throughput: the packed panoramas already sit in HBM, outputs stay in HBM,
         one CUDA-event pair on the launching stream around exactly K steps, max over ranks.
e2e      the same metric through the public API with HOST buffers: every image is uploaded from
         pinned memory (the rows its views can touch: 75 of 100.7 MB), projected and read back
         (74.6 MB) inside the timed region, pipelined over the context's slots (streams).
roofline HBM: algorithmic bytes per launch (SURVEY 8d: 3 * sum(W*H) + 3 * N_T = 141,009,384 B for
         one 12-view image) / average launch duration, against MEASURED_PEAKS.json hbm_gbs.
cpu_baseline  the reference's own script (baseline/_ref/app/panorama_to_plane-pitch.py, a git-ignored copy made by
         __graft_entry__.build(); kind "reference") under its own thread fan-out, or - when that copy is absent -
         oracle/ref_port.py (kind "port"), timed on this box's host cores on a bounded sample, N = 1 only.
e2e.frac_of_transfer_ceiling   time of the bare page-locked copies of the same bytes (no kernels, every rank at once)
         / time of the e2e step: how close the pipeline is to what PCIe and host memory give N GPUs.
e2e_files  JPEG file in -> 12 JPEG files out per image (8.6 MB instead of 150 MB over PCIe), every rank, aggregate.
parity   every rank renders one view of one of ITS OWN seeds and compares it with the CPU oracle outside the timed
         regions (bit-exact when the host's NumPy takes the SVML path the kernel restates, else >= 96 % of pixels).

--dump-outputs DIR  rank 0 writes what the last timed step computed, the [BATCH, yaw, pitch, H, W, 3] u8 views of its 32
         images (2.4 GB), at DUMP_PIXELS fixed pixel positions (seeded, the same in every view) as float32:
         DIR/views.npy [32, 4, 3, DUMP_PIXELS, 3] and the positions DIR/views_yx.npy [DUMP_PIXELS, 2] (row, column).  The
         inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the tree may be read-only: the imports below leave no __pycache__ in it

METRIC = "output Mpix/s (8K equirect -> 1920x1080)"
UNIT = "Mpix/s"

# the README example (BASELINE configs[1]) ----------------------------------------------------
WP, HP = 8192, 4096
W, H, FOV = 1920, 1080, 120
YAWS, PITCHES = [0, 90, 180, 270], [30, 60, 90]
N_VIEWS = len(YAWS) * len(PITCHES)
PX_PER_IMAGE = N_VIEWS * W * H
N_T_C2 = 22_119_928  # distinct panorama texels with non-zero weight, oracle.fixedpoint.touched_texels
B_ALG_PER_IMAGE = 3 * PX_PER_IMAGE + 3 * N_T_C2  # 141,009,384 bytes = 5.667 B / output px
BATCH = 32  # images per GPU per step (configs[2]: 256 images over 8 GPUs)
H2D_PER_IMAGE = WP * HP * 3
D2H_PER_IMAGE = PX_PER_IMAGE * 3
DUMP_PIXELS = 8192  # per view for --dump-outputs: 32 x 12 x 8192 x 3 float32 = 37.7 MB


def workload_config(extra=None):
    cfg = {
        "workload": "configs[2] share per GPU: batch of 32 synthetic 8192x4096 panoramas, each the README "
                    "example (configs[1]): FOV 120, 1920x1080, yaw 0/90/180/270 x pitch 30/60/90 = 12 views",
        "pano": [WP, HP], "out": [W, H], "fov": FOV, "yaws": YAWS, "pitches": PITCHES,
        "batch_images_per_gpu": BATCH, "views_per_image": N_VIEWS, "parallelism": "shard by image, no collective",
        "l2": "inputs larger than L2: each step reads 32 different packed panoramas (4.3 GB) and writes 2.4 GB",
    }
    if extra:
        cfg.update(extra)
    return cfg   # the same dict in both arms (kernel variant keys live in the line's "variant")


def read_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def read_traffic():
    """dram bytes per launch of the projection kernel from the committed ncu summary, or None."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get("project_kernel_dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ---------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi in a child process, killed by PID)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 8:
                self.rows.append(parts)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        sm, smax, reasons, power = [], [], set(), []
        busy = []
        for r in self.rows:
            try:
                c, m = float(r[0]), float(r[1])
            except ValueError:
                continue
            sm.append(c)
            smax.append(m)
            try:
                power.append(float(r[2]))
            except ValueError:
                pass
            try:
                if float(r[3]) > 0:
                    busy.append(c)
            except ValueError:
                pass
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        use = busy if busy else sm
        return {"sm_mhz": statistics.median(use), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm), "samples_busy": len(busy), "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------------------------
# CPU reference arm / baseline: the reference's own script when its git-ignored copy travelled with the
# snapshot (baseline/_ref, made by __graft_entry__.build() where /root/reference exists), else the oracle port
# ---------------------------------------------------------------------------------------------
REF_SCRIPT = ROOT / "baseline" / "_ref" / "app" / "panorama_to_plane-pitch.py"


def load_reference_script():
    """The UNMODIFIED reference module imported by path (its file name has a hyphen), or None."""
    if not REF_SCRIPT.exists():
        return None
    try:
        spec = importlib.util.spec_from_file_location("ref_panorama_to_plane_pitch", REF_SCRIPT)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    except Exception as e:  # noqa: BLE001 - a missing dependency of the script: fall back to the port
        print(f"reference script not importable ({e}); timing the oracle port instead", file=sys.stderr)
        return None


def cpu_reference_run(steps: int, warmup: int, budget_s: float | None = None):
    """One README-example image (12 views) per step on the host cores with warm map caches - the steady state over a
    directory of same-sized images (ref :42-73) - after one cold image that builds the maps.  The fan-out is the
    reference's: ThreadPoolExecutor(max_workers = int(0.9 * cores)) (ref :304-306), one process_yaw_and_pitchs task
    per yaw (ref :252-265), results collected in submit order (:268-272).  Returns (Mpix/s, ms_per_step, steps, info)."""
    import cv2
    from concurrent.futures import ThreadPoolExecutor

    from tools import synth_inputs as synth

    pano = synth.noise(WP, HP, 0)
    workers = max(1, int((os.cpu_count() or 1) * 0.9))
    ref = load_reference_script()
    if ref is not None:
        kind = "reference"

        def one_image():
            with ThreadPoolExecutor(max_workers=workers) as ex:
                futs = [ex.submit(ref.process_yaw_and_pitchs, pano, y, PITCHES, W, H, FOV) for y in YAWS]
                return [f.result() for f in futs]
    else:
        from oracle import ref_port

        kind = "port"
        ref_port.clear_caches()

        def one_image():
            return ref_port.process_image_views(pano, YAWS, PITCHES, W, H, FOV, num_workers=workers)

    t0 = time.perf_counter()
    one_image()  # cold: builds the yaw / pitch maps
    cold_s = time.perf_counter() - t0
    for _ in range(max(0, warmup - 1)):
        one_image()
    done = 0
    t0 = time.perf_counter()
    for _ in range(steps):
        one_image()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    el = time.perf_counter() - t0
    info = {
        "cores": os.cpu_count() or 1,
        "kind": kind,
        "sample": f"{done} README-example images (12 views 8192x4096 -> 1920x1080), one image per step, with warm map "
                  f"caches after 1 cold image ({cold_s:.2f} s incl. map precompute = {PX_PER_IMAGE / cold_s / 1e6:.1f} Mpix/s "
                  f"cold); {'the unmodified reference script baseline/_ref/app/panorama_to_plane-pitch.py' if kind == 'reference' else 'oracle/ref_port.py'}, "
                  f"ThreadPoolExecutor({workers}) one task per yaw, cv2 threads {cv2.getNumThreads()}, "
                  f"numpy {np.__version__}, cv2 {cv2.__version__}",
        "cold_mpix_s": PX_PER_IMAGE / cold_s / 1e6,
    }
    return done * PX_PER_IMAGE / el / 1e6, el / done * 1e3, done, info


def run_reference_arm(args, rank: int):
    if rank != 0:
        return
    val, ms, done, info = cpu_reference_run(args.steps, args.warmup)
    cb = {"value": val, "unit": UNIT, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]}
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# the CUDA arm
# ---------------------------------------------------------------------------------------------
def run_b200_arm(args, rank: int, local_rank: int, world: int):
    import torch

    import __graft_entry__ as g
    from tools import synth_inputs as synth  # synthetic input generator (no oracle code)

    g.build()
    pkg = g.load_package()
    from p2p_b200 import distrib

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ranks = distrib.Ranks("nccl", device=dev)  # no-op when WORLD_SIZE == 1
    barrier, max_over_ranks = ranks.barrier, ranks.max

    n_e2e_slots = 4
    proj = pkg.Projector(local_rank, n_slots=BATCH + n_e2e_slots)
    L = pkg._lib
    if args.sampler is not None:
        proj.set_option(L.OPT_SAMPLER, args.sampler)
    if args.warp_w is not None:
        proj.set_option(L.OPT_WARP_W, args.warp_w)
    if args.ny is not None:
        proj.set_option(L.OPT_YAWS_PER_THREAD, args.ny)
    if args.nb is not None:
        proj.set_option(L.OPT_IMAGES_PER_LAUNCH, args.nb)

    consts = [pkg.pitch_constants(W, FOV, p) for p in PITCHES]
    shifts = [pkg.yaw_table(WP, y)[2] for y in YAWS]
    assert all(s is not None for s in shifts)

    # ---- resident inputs: BATCH packed panoramas per GPU (seeds follow configs[2]: rank-major) ----
    res_slots = list(range(BATCH))
    # The 32 images of a step are independent launches: they alternate over n_streams launching streams (slot i on the
    # stream of slot i % n_streams), so the tail of one image's grid overlaps the ramp-up of the next one's - with a single
    # stream every launch pays its own tail and launch gap (58 vs 65-68 us per image).  Two launches are in flight at
    # most, so the L2 still holds one image's cross-view working set most of the time.  The timed region is bracketed by
    # ONE event pair on stream 0: the other streams wait for the start event, stream 0 waits for their end events.
    n_streams = max(1, min(args.streams, BATCH))
    own_streams = [proj.get_stream(i) for i in res_slots]   # given back after the resident region
    for i in res_slots:
        if i >= n_streams:
            proj.set_stream(i, own_streams[i % n_streams])
    n_distinct = min(BATCH, args.distinct)
    host = [synth.noise(WP, HP, rank * BATCH + i) for i in range(n_distinct)]
    d_stage = torch.empty((HP, WP, 3), dtype=torch.uint8, device=dev)
    for i in res_slots:
        # panorama i is noise(seed) rolled by a different column offset when fewer seeds than slots
        src = host[i % n_distinct]
        d_stage.copy_(torch.from_numpy(src))
        if i >= n_distinct:
            d_stage.copy_(torch.roll(d_stage, shifts=37 * i, dims=1))
        torch.cuda.synchronize()
        proj.upload_device(i, d_stage.data_ptr(), WP, HP, WP * 3)
        proj.sync(i)
    d_out = torch.empty((BATCH, N_VIEWS, H, W, 3), dtype=torch.uint8, device=dev)
    out_ptrs = [d_out[i].data_ptr() for i in range(BATCH)]

    resident_step = proj.batch_call(res_slots, shifts, consts, W, H, out_ptrs, on_device=True)

    for _ in range(max(3, args.warmup)):
        resident_step()
    proj.sync(-1)
    ev0, ev1 = proj.event(), proj.event()
    ev_join = [proj.event() for _ in range(n_streams)]

    def timed_steps(n_steps):
        """Device time of n_steps steps over all launching streams (fork / join through events on stream 0)."""
        proj.record(ev0, 0)
        for st in range(1, n_streams):
            proj.event_wait(ev0, st)
        for _ in range(n_steps):
            resident_step()
        for st in range(1, n_streams):
            proj.record(ev_join[st], st)
            proj.event_wait(ev_join[st], 0)
        proj.record(ev1, 0)
        proj.sync(-1)
        return proj.elapsed_ms(ev0, ev1)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = proj.launches
    barrier()
    torch.cuda.synchronize()
    ms_local = timed_steps(args.steps)
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, d_out, Path(args.dump_outputs))
    barrier()
    ms_total = max_over_ranks(ms_local)
    launches = proj.launches - launches0
    # the same launches strictly one after the other on one stream (what a single ncu-serialised launch costs)
    serial_ms = None
    if n_streams > 1:
        for i in res_slots[1:]:
            proj.set_stream(i, proj.get_stream(0))
        ns, n_streams = n_streams, 1
        timed_steps(1)
        serial_ms = timed_steps(min(5, args.steps)) / (min(5, args.steps) * BATCH)
        n_streams = ns
    for i in res_slots:   # every slot back on its own stream: the later legs (files flow) borrow these slots concurrently
        proj.set_stream(i, own_streams[i])
    ms_per_step = ms_total / args.steps
    value = world * args.steps * BATCH * PX_PER_IMAGE / (ms_total * 1e-3) / 1e6
    launch_ms = ms_total / (args.steps * BATCH)

    # ---- end to end through the public API with host buffers -------------------------------
    e2e_slots = list(range(BATCH, BATCH + n_e2e_slots))
    n_host = 3
    pin_in = [pkg.PinnedBuffer((HP, WP, 3)) for _ in range(n_host)]
    for k, b in enumerate(pin_in):
        b.array[...] = host[k % n_distinct]
    pin_out = [pkg.PinnedBuffer((len(YAWS), len(PITCHES), H, W, 3)) for _ in range(n_e2e_slots)]

    def e2e_step():
        for i in range(BATCH):
            s = e2e_slots[i % n_e2e_slots]
            proj.sync(s)  # the slot's previous image (and its readback) is complete
            proj.process_image(s, pin_in[i % n_host].array, shifts, consts, W, H, pin_out[i % n_e2e_slots].array)

    def time_e2e(n_steps):
        for _ in range(2):
            e2e_step()
        proj.sync(-1)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n_steps):
            e2e_step()
        proj.sync(-1)
        torch.cuda.synchronize()
        sec = max_over_ranks(time.perf_counter() - t0)
        barrier()
        return sec

    # the library transfers only the panorama rows these views can touch (p2p_view_row_range)
    row_first, row_last = proj.view_row_range(consts, W, H, WP, HP)
    h2d_per_image = (row_last - row_first + 1) * WP * 3 if proj.get_option(L.OPT_PARTIAL_UPLOAD) else H2D_PER_IMAGE
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_s = time_e2e(e2e_steps)
    e2e_value = world * e2e_steps * BATCH * PX_PER_IMAGE / e2e_s / 1e6
    clocks = sampler.stop() if sampler is not None else None

    # light self-check of the e2e result buffer (not timed): last image equals a device-resident render
    check = proj.project_image(pin_in[(BATCH - 1) % n_host].array, YAWS, PITCHES, W, H, FOV)
    assert np.array_equal(check, pin_out[(BATCH - 1) % n_e2e_slots].array), "e2e readback differs from resident render"

    # the same pipeline moving the WHOLE panorama (no knowledge of the view set used): secondary figure
    e2e_full = None
    if proj.get_option(L.OPT_PARTIAL_UPLOAD) and not args.no_extras:
        proj.set_option(L.OPT_PARTIAL_UPLOAD, 0)
        n_full = max(1, min(2, e2e_steps))
        full_s = time_e2e(n_full)
        proj.set_option(L.OPT_PARTIAL_UPLOAD, 1)
        e2e_full = {"value": world * n_full * BATCH * PX_PER_IMAGE / full_s / 1e6, "unit": UNIT,
                    "h2d_bytes_per_step": BATCH * H2D_PER_IMAGE, "ms_per_step": full_s / n_full * 1e3, "steps": n_full}

    # transfer ceiling: the bare page-locked copies of one e2e step (same buffers, same byte counts, two streams, no
    # kernels), every rank at the same time
    ceil_s = transfer_ceiling(torch, dev, pin_in, pin_out, h2d_per_image, D2H_PER_IMAGE, barrier, max_over_ranks)

    # ---- parity of THIS rank's own data against the CPU oracle (outside every timed region) ----
    parity = oracle_check(proj, host[0], rank * BATCH)
    parity_ranks = int(round(ranks.sum(1.0 if parity["ok"] else 0.0)))

    # ---- files flow at every N: JPEG file in, 12 JPEG files out, only files cross PCIe ----
    e2e_files = None
    if not args.no_extras:
        e2e_files = files_flow(pkg, proj, synth.smooth(WP, HP, rank), shifts, consts, "jpg", world, barrier, max_over_ranks)
        # the reference's default output format: 34 MB of PNG files per image go back over PCIe instead of 4 MB
        e2e_files["png"] = files_flow(pkg, proj, synth.smooth(WP, HP, rank), shifts, consts, "png", world, barrier, max_over_ranks,
                                      n_img=48)
        # PNG in, PNG out: the reference's default format on both sides (a second pass over its own outputs); the 8K file
        # (cv2.imwrite defaults) is inflated and unfiltered on the GPU.  A new leg: a failing image is recorded, not fatal.
        e2e_files["png_in"] = files_flow(pkg, proj, synth.smooth(WP, HP, rank), shifts, consts, "png", world, barrier,
                                         max_over_ranks, n_img=16, n_thr=4, src="png", tolerant=True)

    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        extras = files_extras(pkg, proj, synth.smooth(WP, HP, 0), shifts, consts)
        extras["configs"] = config_fractions(pkg, proj, synth, torch)
        extras["fractional_yaw"] = fractional_yaw_times(pkg, proj, synth, torch)
        extras["png_decode"] = png_decode_times(pkg, proj, synth)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, _ms, done, info = cpu_reference_run(10_000, 1, budget_s=args.cpu_seconds)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]}
    elif rank == 0:
        cpu_baseline = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1,
                        "kind": "reference" if REF_SCRIPT.exists() else "port",
                        "sample": "not run (N > 1 or --no-cpu-baseline); see the N = 1 line"}

    if rank == 0:
        peak, peak_src = read_peaks()
        achieved = B_ALG_PER_IMAGE / (launch_ms * 1e-3) / 1e9
        mirror = proj.get_option(L.OPT_MIRROR)
        kernel = {2: "p2p::project_rows_kernel<4, true, true>", 1: "p2p::project_mirror_kernel<4, true>"}.get(
            mirror if proj.get_option(L.OPT_SAMPLER) == 1 and proj.get_option(L.OPT_IMAGES_PER_LAUNCH) == 1 else 0,
            "p2p::project_kernel")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(),
            "variant": {
                "sampler": proj.get_option(L.OPT_SAMPLER), "warp_w": proj.get_option(L.OPT_WARP_W),
                "yaws_per_thread": proj.get_option(L.OPT_YAWS_PER_THREAD),
                "images_per_launch": proj.get_option(L.OPT_IMAGES_PER_LAUNCH),
                "mirror_pairs": mirror, "seg_chunks": proj.get_option(L.OPT_SEG_CHUNKS),
                "trig": "numpy_exact_svml" if proj.get_option(L.OPT_TRIG) == 0 else "minimax",
                "distinct_seeds_per_gpu": n_distinct, "launching_streams": n_streams,
            },
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": read_traffic(), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": B_ALG_PER_IMAGE, "launch_ms": launch_ms,
                "launch_ms_note": f"timed region / launches with the images alternating over {n_streams} launching stream(s)",
                "serialized_launch_ms": serial_ms,
                "serialized_frac": (B_ALG_PER_IMAGE / (serial_ms * 1e-3) / 1e9 / peak) if serial_ms else None,
                "kernel": kernel + " (one launch = one image = 12 views)",
            },
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": BATCH * h2d_per_image,
                    "d2h_bytes_per_step": BATCH * D2H_PER_IMAGE, "steps": e2e_steps,
                    "ms_per_step": e2e_s / e2e_steps * 1e3, "pipeline_slots": n_e2e_slots,
                    "h2d_rows": [row_first, row_last],
                    "h2d_note": f"rows {row_first}..{row_last} of {HP}: the only panorama rows the 12 views read "
                                f"({h2d_per_image} of {H2D_PER_IMAGE} bytes per image)",
                    "transfer_ceiling_ms_per_step": ceil_s * 1e3,
                    "frac_of_transfer_ceiling": ceil_s / (e2e_s / e2e_steps),
                    "transfer_ceiling_note": "bare cudaMemcpyAsync of the same bytes from / to the same page-locked buffers, "
                                             "upload || readback on two streams, no kernels, all ranks at once (max over ranks)",
                    "full_upload": e2e_full},
            "e2e_files": e2e_files,
            "parity": {"checked_ranks": parity_ranks, "of_ranks": world, "rank0": parity},
            "gpu_launches": launches * world,
            "clocks": clocks,
        }
        if extras is not None:
            line["extras"] = extras
        emit(line)
    for b in pin_in + pin_out:
        b.free()
    proj.close()
    ranks.close()


def dump_outputs(torch, d_out, out_dir: Path):
    """--dump-outputs: the views of the last timed step at DUMP_PIXELS fixed pixel positions (see the module docstring)."""
    flat = np.sort(np.random.default_rng(0).choice(H * W, DUMP_PIXELS, replace=False))
    idx = torch.from_numpy(flat).to(d_out.device)
    views = d_out.view(BATCH, len(YAWS), len(PITCHES), H * W, 3).index_select(3, idx)
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "views.npy", views.float().cpu().numpy())
    np.save(out_dir / "views_yx.npy", np.stack([flat // W, flat % W], axis=1).astype(np.float32))


def transfer_ceiling(torch, dev, pin_in, pin_out, h2d_bytes, d2h_bytes, barrier, max_over_ranks, steps=2):
    """Seconds per e2e step of the bare transfers: BATCH x (h2d_bytes up || d2h_bytes down) between the bench's own
    page-locked buffers and scratch device memory on two streams.  No kernel, no library code: the PCIe / host-memory
    ceiling of the step on this box with this many ranks active."""
    d_in = [torch.empty(h2d_bytes, dtype=torch.uint8, device=dev) for _ in range(2)]
    d_out = [torch.empty(d2h_bytes, dtype=torch.uint8, device=dev) for _ in range(2)]
    h_in = [torch.from_numpy(b.array.reshape(-1)[:h2d_bytes]) for b in pin_in]     # views of the page-locked buffers
    h_out = [torch.from_numpy(b.array.reshape(-1)[:d2h_bytes]) for b in pin_out]
    s_up, s_dn = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    import ctypes as C

    rt = C.CDLL("libcudart.so.12")   # resolves to the runtime torch has already loaded
    rt.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    rt.cudaMemcpyAsync.restype = C.c_int

    def step():
        for i in range(BATCH):
            # cudaMemcpyAsync directly: torch's copy_ would stage a non-torch-pinned host tensor
            rc1 = rt.cudaMemcpyAsync(d_in[i % 2].data_ptr(), h_in[i % len(h_in)].data_ptr(), h2d_bytes, 1, s_up.cuda_stream)
            rc2 = rt.cudaMemcpyAsync(h_out[i % len(h_out)].data_ptr(), d_out[i % 2].data_ptr(), d2h_bytes, 2, s_dn.cuda_stream)
            assert rc1 == 0 and rc2 == 0, (rc1, rc2)

    step()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    sec = max_over_ranks(time.perf_counter() - t0)
    barrier()
    return sec / steps


def oracle_check(proj, pano, seed):
    """One view (yaw 90, pitch 60) of this rank's own panorama against oracle.fixedpoint.project_view_single_pass.  The
    oracle is the checker here, never the thing measured."""
    from oracle import fixedpoint, svml_model

    got = proj.project_image(pano, [90], [60], W, H, FOV)[0, 0]
    want = fixedpoint.project_view_single_pass(pano, 90, 60, W, H, FOV)
    strict = bool(svml_model.host_numpy_uses_svml())
    frac = float((got == want).all(axis=-1).mean())
    return {"ok": bool(frac == 1.0 if strict else frac >= 0.96), "exact_pixel_fraction": frac, "seed": int(seed),
            "view": [90, 60], "mode": "bit-exact (host NumPy uses SVML arccos / arctan2, restated by the kernel)" if strict
            else "tolerance (host NumPy does not take the SVML path: the reference itself differs in the last ulp here)"}


def files_flow(pkg, proj, pano, shifts, consts, fmt, world, barrier, max_over_ranks, n_img=96, n_thr=8, src="jpg", tolerant=False):
    """Files to files on every rank: an 8192x4096 JPEG file in host memory -> the 12 views as files in page-locked host
    memory; Huffman decode, IDCT, projection and encode all on the GPU, n_thr images in flight per rank.  Whole-job
    Mpix/s = all ranks' images / the slowest rank's time."""
    import cv2
    from concurrent.futures import ThreadPoolExecutor

    data = cv2.imencode("." + src, pano)[1].tobytes()
    # images in flight per rank = host threads: a waiting thread spins on its stream (the CUDA default), so the ranks of one box
    # share its cores - 8 threads on each of 8 ranks of a 32-vCPU box cost a third of the throughput (profiles/r2_files_flow_*)
    n_thr = max(2, min(n_thr, (os.cpu_count() or 8) // max(1, world)))

    errors = []

    def one(_):
        try:
            with proj.slots(1) as (s,):
                proj.upload_encoded(s, data)   # JPEG: Huffman stage + IDCT on the device; PNG: inflate + unfilter on the device
                if fmt == "jpg":
                    files = proj.project_jpeg(s, shifts, consts, W, H, copy=False)
                else:
                    files = proj.process_image_png(s, None, shifts, consts, W, H, want_pixels=False, copy=False)[0]
                return sum(len(f) for f in files)
        except Exception as e:  # noqa: BLE001
            if not tolerant:
                raise
            errors.append(repr(e))   # (the collectives below must still be entered by every rank)
            return 0

    with ThreadPoolExecutor(n_thr) as ex:
        out_bytes = list(ex.map(one, range(n_thr)))[0]
        barrier()
        t0 = time.perf_counter()
        list(ex.map(one, range(n_img)))
        sec = max_over_ranks(time.perf_counter() - t0)
        barrier()
    if errors:
        return {"error": errors[0], "failed_images": len(errors), "format": f"{src} -> {fmt}"}
    return {"value": world * n_img * PX_PER_IMAGE / sec / 1e6, "unit": UNIT, "format": f"{src} -> {fmt}",
            "ms_per_image_per_gpu": sec / n_img * 1e3, "images_per_rank": n_img, "threads_per_rank": n_thr,
            "h2d_bytes_per_image": len(data), "d2h_bytes_per_image": out_bytes,
            "what": f"8192x4096 {src.upper()} file bytes (host) -> 12 x 1920x1080 files (host); decode, projection and encode on "
                    "the GPU; every rank runs the same flow at once"}


def config_fractions(pkg, proj, synth, torch):
    """Device-resident time and HBM-roofline fraction of the other BASELINE configs (C1, C4, C5), each ONE launch of the
    flat view list; the L2 is flushed before every repetition (C1 / C5 panoramas would otherwise stay L2-resident)."""
    peak, _ = read_peaks()
    cfgs = {   # name: Wp, Hp, W, H, fov, views, algorithmic bytes per output px (SURVEY 8d)
        "C1": (2048, 1024, 640, 480, 90, [(0, 90)], 4.94),
        "C4": (16384, 8192, 3840, 2160, 100, [(y, p) for y in YAWS for p in PITCHES], 5.529),
        "C5": (8192, 4096, 2048, 2048, 90, [(0, 90), (90, 90), (180, 90), (270, 90), (0, 0), (0, 180)], 6.42),
    }
    out = {}
    ev0, ev1 = proj.event(), proj.event()
    for name, (wp, hp, w, h, fov, views, b_px) in cfgs.items():
        with proj.slots(1) as (s,):
            proj.upload(s, synth.noise(wp, hp, 0))
            proj.sync(s)
            d = torch.empty((len(views), h, w, 3), dtype=torch.uint8, device=f"cuda:{proj.device}")
            sh = [pkg.yaw_table(wp, y)[2] for y, _ in views]
            pc = [pkg.pitch_constants(w, fov, q) for _, q in views]
            n0 = proj.launches
            proj.project_list(s, sh, pc, w, h, out_device_ptr=d.data_ptr())
            proj.sync(s)
            per_image = proj.launches - n0
            ts = []
            for _ in range(10):
                proj.flush_l2(s, 256 << 20)
                proj.record(ev0, s)
                proj.project_list(s, sh, pc, w, h, out_device_ptr=d.data_ptr())
                proj.record(ev1, s)
                proj.sync(s)
                ts.append(proj.elapsed_ms(ev0, ev1))
            ms = statistics.median(ts)
            px = len(views) * w * h
            gbs = b_px * px / (ms * 1e-3) / 1e9
            out[name] = {"image_us": ms * 1e3, "launches_per_image": per_image, "gpix_s": px / ms / 1e6,
                         "algorithmic_bytes_per_px": b_px, "achieved_gbs": gbs, "roofline_frac": gbs / peak}
            del d
    return out


def fractional_yaw_times(pkg, proj, synth, torch):
    """A yaw that is not an integer column roll (ref :191-199 + :212-218), 3 pitches of the README example on a resident
    8192x4096 panorama: the one-pass kernel (both remap passes per output pixel) against the materialised yaw pass +
    projection it replaces.  Device time, CUDA events, same pixels (checked)."""
    yaw = 33.3
    ix, fx, shift = pkg.yaw_table(WP, yaw)
    assert shift is None
    consts = [pkg.pitch_constants(W, FOV, p) for p in PITCHES]
    ev0, ev1 = proj.event(), proj.event()
    with proj.slots(2) as (a, b):
        proj.upload(a, synth.noise(WP, HP, 0))
        proj.sync(a)
        d1 = torch.empty((1, len(PITCHES), H, W, 3), dtype=torch.uint8, device=f"cuda:{proj.device}")
        d2 = torch.empty_like(d1)
        one, two = [], []
        for _ in range(6):
            proj.record(ev0, a)
            proj.project_tables(a, [(ix, fx)], consts, W, H, out_device_ptr=d1.data_ptr())
            proj.record(ev1, a)
            proj.sync(a)
            one.append(proj.elapsed_ms(ev0, ev1))
            proj.record(ev0, b)
            proj.rotate(a, b, ix, fx)
            proj.project(b, [0], consts, W, H, out_device_ptr=d2.data_ptr())
            proj.record(ev1, b)
            proj.sync(b)
            two.append(proj.elapsed_ms(ev0, ev1))
        same = bool(torch.equal(d1, d2))
    return {"yaw": yaw, "views": len(PITCHES), "one_pass_us": statistics.median(one[1:]) * 1e3,
            "rotate_then_project_us": statistics.median(two[1:]) * 1e3, "identical": same,
            "note": "the two-pass figure includes the yaw table upload the rotate entry point waits for"}


def png_decode_times(pkg, proj, synth):
    """Side measurement: an 8192x4096 PNG panorama (cv2.imwrite defaults) into a slot - the device decoder (parallel
    inflate + unfilter, csrc/p2p_pngdec.cuh) against cv2.imdecode + upload, one host thread, same pixels (checked)."""
    import cv2

    try:
        pano = synth.smooth(WP, HP, 3)
        data = cv2.imencode(".png", pano)[1].tobytes()
        arr = np.frombuffer(data, np.uint8)
        with proj.slots(1) as (s,):
            proj.upload_png(s, data)
            proj.sync(s)
            same = bool(np.array_equal(proj.download_pano(s, WP, HP), pano))
            t_dev, t_cv = [], []
            for _ in range(3):
                t0 = time.perf_counter()
                proj.upload_png(s, data)
                proj.sync(s)
                t_dev.append(time.perf_counter() - t0)
            for _ in range(2):
                t0 = time.perf_counter()
                proj.upload(s, cv2.imdecode(arr, cv2.IMREAD_COLOR))
                proj.sync(s)
                t_cv.append(time.perf_counter() - t0)
        return {"what": "8192x4096 PNG file bytes (host) -> packed panorama in a slot, one host thread",
                "file_bytes": len(data), "same_pixels_as_cv2": same, "device_decoder_ms": min(t_dev) * 1e3,
                "cv2_imdecode_plus_upload_ms": min(t_cv) * 1e3, "speedup": min(t_cv) / min(t_dev)}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def files_extras(pkg, proj, pano, shifts, consts):
    """Side measurement (not the headline metric): the codec rows either side of the path (SURVEY 8f-2).  One 8192x4096
    JPEG file in host memory -> the 12 views as jpg / png files in (page-locked) host memory, (a) decoded, projected and
    encoded on the GPU, 4 images in flight on 4 host threads; (b) the reference's flow on the host cores: cv2.imdecode -> oracle port of
    the projection -> cv2.imencode per view.  Same bytes out (checked)."""
    import cv2
    from concurrent.futures import ThreadPoolExecutor

    from oracle import ref_port

    data = cv2.imencode(".jpg", pano)[1].tobytes()
    n_img, n_thr = 32, 4
    out = {}
    for fmt in ("jpg", "png"):
        def gpu_one(keep):
            # the files land in the slot's page-locked host buffer; the front end writes them to disk from there
            # (copy=False), the identity check below takes a copy
            with proj.slots(1) as (s,):
                proj.upload_jpeg(s, data)
                if fmt == "jpg":
                    files = proj.project_jpeg(s, shifts, consts, W, H, copy=False)
                else:
                    files = proj.process_image_png(s, None, shifts, consts, W, H, want_pixels=False, copy=False)[0]
                return [bytes(f) for f in files] if keep else sum(len(f) for f in files)

        with ThreadPoolExecutor(n_thr) as ex:
            first = list(ex.map(gpu_one, [True] * n_thr))[0]
            t0 = time.perf_counter()
            list(ex.map(gpu_one, [False] * n_img))
            gpu_s = (time.perf_counter() - t0) / n_img
        ref_port.clear_caches()
        ref_files = None
        cpu_s = []
        for _ in range(2):  # second pass = warm map caches
            t0 = time.perf_counter()
            img = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
            views = ref_port.process_image_views(img, YAWS, PITCHES, W, H, FOV)
            ref_files = [cv2.imencode("." + fmt, v)[1].tobytes() for per_yaw in views for v in per_yaw]
            cpu_s.append(time.perf_counter() - t0)
        ref_port.clear_caches()
        out[fmt + "_files"] = {
            "what": f"8192x4096 JPEG bytes (host) -> 12 x 1920x1080 {fmt} files (host); decode (Huffman stage included), "
                    f"projection and encode on the GPU, 4 images in flight; CPU = cv2.imdecode + oracle port + cv2.imencode, "
                    f"warm maps",
            "byte_identical_to_cpu_flow": bool(first == ref_files),
            "gpu_ms_per_image": gpu_s * 1e3, "gpu_mpix_s": PX_PER_IMAGE / gpu_s / 1e6,
            "cpu_ms_per_image": min(cpu_s) * 1e3, "cpu_mpix_s": PX_PER_IMAGE / min(cpu_s) / 1e6,
            "input_file_bytes": len(data), "output_file_bytes": sum(len(f) for f in first)}
    return out


_REAL_STDOUT = None


def emit(line: dict):
    """Print the one JSON line on the real stdout (library chatter such as NCCL's version banner has
    been redirected to stderr by ``main``)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    # stdout carries exactly one JSON line: everything else any library prints to fd 1 goes to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--sampler", type=int, default=None)
    ap.add_argument("--warp-w", type=int, default=None)
    ap.add_argument("--ny", type=int, default=None)
    ap.add_argument("--nb", type=int, default=None, help="resident panoramas per launch (1, 2, 4)")
    ap.add_argument("--streams", type=int, default=2, help="launching streams the resident images alternate over")
    ap.add_argument("--distinct", type=int, default=8, help="distinct noise seeds per GPU (others are rolled copies)")
    ap.add_argument("--e2e-steps", type=int, default=5, help="cap on end-to-end steps (each moves 5.6 GB over PCIe)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the files-to-files (JPEG in, JPEG out) side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's outputs as DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), __file__, *sys.argv[1:]]
        os.dup2(_REAL_STDOUT, 1)  # the torchrun children write their own single line
        raise SystemExit(subprocess.call(cmd))
    run_b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
