"""Measures the cloud transform stage (pcl::transformPointCloud, the first cloud stage) on the current GPU; one JSON
line per case.

    python tools/transform_bench.py [--out FILE] [--quick]

(a) stage   stage time per frame: CUDA events around warm d2pc_reproject_mono8_device batches of S2 scene frames (64
            frames, 16 at 4K) with the transform on, minus the same batches in CROP mode (alternated), at 752x480,
            1280x720 and 3840x2160.  Against the HBM bound of the bytes the stage moves: every point read (16 B) and
            written (16 B), over 7.7 TB/s (HGX B200 data sheet, one GPU).  The 4K batch (2 GB per cloud buffer) does
            not fit the 126 MB L2; the 752x480 batch (275 MB) does not either.
(b) stream  d2pc_process_stream frames/s: CROP, CROP + transform, CROP_FINITE, CROP_FINITE + transform (752x480 and
            1280x720 mono8).
(c) lone    one synchronous d2pc_process_mono8 call (median of many) at 752x480 and 1280x720: CROP; CROP + transform
            into a device buffer followed by a D2H copy (direct_out 0, the default for transform plans); and CROP +
            transform with the transform kernel storing into the page-locked destination (direct_out 1).  Alternated.
(d) launch  kernel launches of one synchronous 752x480 call per plan (d2pc_launch_count).
Every line carries the card's name and power limit, read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import disparity_to_point_cloud_b200 as d2pc  # noqa: E402
from disparity_to_point_cloud_b200 import synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
# camera optical frame -> a body frame (x forward, y left, z up), slightly tilted, with an offset
POSE = np.float32([[0.0998, 0.0497, 0.9938, 0.1], [-0.9752, 0.2033, 0.0878, 0.02], [-0.1977, -0.9779, 0.0688, -0.05]])


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def n_points(w, h, border=40):
    return max(0, w - 2 * border) * max(0, h - 2 * border)


def frames_for(h, w, nf):
    return np.stack([synth.s2_scene(h, w, i) for i in range(nf)])


def time_batch(ctx, fn, args, reps):
    s = torch.cuda.ExternalStream(ctx.compute_stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(reps):
        fn(*args)
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps  # us per batch


def stage(ctx, h, w, nf, reps):
    frames = frames_for(h, w, nf)
    n = n_points(w, h)
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.empty(nf * n * 16, dtype=torch.uint8, device="cuda")
    args = (d_in.data_ptr(), nf, w, h, w, w * h, d_pts.data_ptr(), n * 16, 0)
    times = {"off": [], "on": []}
    for on in ("off", "on"):  # warm both (module load, buffer sizing)
        ctx.set_transform(POSE if on == "on" else None)
        time_batch(ctx, ctx.reproject_mono8_device, args, 2)
        ctx.sync()
    for _ in range(5):
        for on in ("off", "on"):
            ctx.set_transform(POSE if on == "on" else None)
            times[on].append(time_batch(ctx, ctx.reproject_mono8_device, args, reps))
    ctx.set_transform(None)
    off_us, on_us = float(np.median(times["off"])), float(np.median(times["on"]))
    stage_us = (on_us - off_us) / nf
    bytes_per_frame = 32 * n
    bound_us = bytes_per_frame / HBM_BYTES_PER_S * 1e6
    return dict(case="a_stage", w=w, h=h, frames=nf, crop_points=n, crop_us_per_frame=off_us / nf,
                crop_plus_transform_us_per_frame=on_us / nf, stage_us_per_frame=stage_us,
                spread_off_us=[min(times["off"]) / nf, max(times["off"]) / nf],
                spread_on_us=[min(times["on"]) / nf, max(times["on"]) / nf],
                stage_bytes_per_frame=bytes_per_frame, hbm_bound_us_per_frame=bound_us,
                share_of_hbm_bound=bound_us / stage_us if stage_us > 0 else None)


def stream(ctx, h, w, n_frames, reps):
    ring = d2pc.PinnedArray((16, h, w), np.uint8)
    ring.array[:] = frames_for(h, w, 16)
    cases = {"crop": (d2pc.FILTER_CROP, None), "crop+transform": (d2pc.FILTER_CROP, POSE),
             "finite": (d2pc.FILTER_CROP_FINITE, None), "finite+transform": (d2pc.FILTER_CROP_FINITE, POSE)}
    out = {k: [] for k in cases}

    def setup(k):
        mode, xf = cases[k]
        ctx.set_filter_mode(mode)
        ctx.set_transform(xf)

    for k in cases:
        setup(k)
        ctx.process_stream(ring.array, collect=False, n_frames=32)
    for _ in range(reps):
        for k in cases:
            setup(k)
            t0 = time.perf_counter()
            ctx.process_stream(ring.array, collect=False, n_frames=n_frames)
            out[k].append(n_frames / (time.perf_counter() - t0))
    ctx.set_transform(None)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ring.free()
    return {k: {"frames_per_s": float(np.median(v)), "spread": [min(v), max(v)]} for k, v in out.items()}


def lone(ctx, h, w, reps):
    img = synth.s2_scene(h, w, 1)
    cases = {"crop": (None, 0), "crop+transform copy": (POSE, 0), "crop+transform direct_out 1": (POSE, 1)}
    ts = {k: [] for k in cases}
    outs = {}
    for i in range(reps + 20):
        for k, (xf, direct) in cases.items():
            ctx.set_transform(xf)
            ctx.set_tuning("direct_out", direct)
            t0 = time.perf_counter()
            got = ctx.process_mono8(img, copy=False)
            if i >= 20:
                ts[k].append((time.perf_counter() - t0) * 1e6)
            if i == 0:
                outs[k] = got.tobytes()
    ctx.set_transform(None)
    ctx.set_tuning("direct_out", 0)
    assert outs["crop+transform copy"] == outs["crop+transform direct_out 1"]
    return {k: {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)),
                "p90_us": float(np.percentile(v, 90))} for k, v in ts.items()}


def launches(ctx):
    img = synth.s2_scene(480, 752, 1)
    ctx.set_voxel_grid(0.05, 0, ("z", 0.0, 10.0))
    box = (np.float32([0.5, -2, -1]), np.float32([6, 2, 1]), None)
    plans = {}
    for name, mode in (("crop", d2pc.FILTER_CROP), ("finite", d2pc.FILTER_CROP_FINITE), ("voxel", d2pc.FILTER_VOXEL)):
        for xf in (None, POSE):
            for b in (None, box):
                plans[name + ("+transform" if xf is not None else "") + ("+box" if b else "")] = (mode, xf, b)
    out = {}
    for k, (mode, xf, b) in plans.items():
        ctx.set_filter_mode(mode)
        ctx.set_transform(xf)
        ctx.set_crop_box(*(b or (None,)))
        n0 = ctx.launch_count()
        ctx.process_mono8(img)
        out[k] = ctx.launch_count() - n0
    ctx.set_crop_box(None)
    ctx.set_transform(None)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small batches and few repetitions (a rehearsal)")
    a = ap.parse_args()
    info = card()
    lines = []

    def emit(d):
        d = dict(d, **info)
        lines.append(d)
        print(json.dumps(d), flush=True)

    reps = 2 if a.quick else 10
    with d2pc.Context(n_slots=4) as ctx:
        sizes = [(480, 752, 4)] if a.quick else [(480, 752, 64), (720, 1280, 64), (2160, 3840, 16)]
        for h, w, nf in sizes:
            emit(stage(ctx, h, w, nf, reps))
        for h, w in [(480, 752), (720, 1280)]:
            r = stream(ctx, h, w, 200 if a.quick else 3000, 2 if a.quick else 5)
            emit({"case": "b_stream", "entry": "mono8", "w": w, "h": h, **r})
        for h, w in [(480, 752), (720, 1280)]:
            emit({"case": "c_lone", "entry": "mono8", "w": w, "h": h, **lone(ctx, h, w, 50 if a.quick else 500)})
        emit({"case": "d_launches", "entry": "mono8", "w": 752, "h": 480, **launches(ctx)})
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
