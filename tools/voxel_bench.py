"""Measures D2PC_FILTER_VOXEL (pcl::VoxelGrid on the device) on the current GPU; one JSON line per case.

    python tools/voxel_bench.py [--out FILE] [--quick]

(a) stage   voxel-stage time per frame: CUDA events around d2pc_reproject_{mono8,f32}_device batches in VOXEL
            minus the same batches in CROP (alternated, warm; every batch's CROP cloud is larger than the 126 MB L2).
            S2 scene frames through the mono8 entry, S3 through the float entry; leaf 0.05 / 0.2 m, with and
            without a z limit of [0, 10] m.
(b) stream  d2pc_process_stream frames/s and device-to-host bytes per frame, CROP vs VOXEL alternated in one run.
(c) lone    one synchronous 752x480 d2pc_process_mono8 call, CROP vs VOXEL (median of many).
(d) fold    the serial-fold worst case: a 10 m leaf without a limit, one frame per batch, so one voxel holds
            most of the frame.
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


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def n_points(w, h, border=40):
    return max(0, w - 2 * border) * max(0, h - 2 * border)


def frames_for(kind, h, w, nf):
    gen = synth.s2_scene if kind == "mono8" else synth.s3_float
    return np.stack([gen(h, w, i) for i in range(nf)])


def time_batch(ctx, fn, args, reps):
    s = torch.cuda.ExternalStream(ctx.compute_stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(reps):
        fn(*args)
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps  # us per batch


def stage(ctx, kind, h, w, nf, leaf, limit, reps, extra):
    frames = frames_for(kind, h, w, nf)
    n = n_points(w, h)
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.empty(nf * n * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
    step = w * frames.itemsize
    fn = ctx.reproject_mono8_device if kind == "mono8" else ctx.reproject_f32_device
    args = (d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), n * 16, d_cnt.data_ptr())
    ctx.set_voxel_grid(leaf, 0, limit)
    times = {"crop": [], "voxel": []}
    for mode in ("crop", "voxel"):  # warm both (module load, scratch sizing)
        ctx.set_filter_mode(d2pc.FILTER_CROP if mode == "crop" else d2pc.FILTER_VOXEL)
        time_batch(ctx, fn, args, 2)
    for _ in range(5):
        for mode in ("crop", "voxel"):
            ctx.set_filter_mode(d2pc.FILTER_CROP if mode == "crop" else d2pc.FILTER_VOXEL)
            times[mode].append(time_batch(ctx, fn, args, reps))
    ctx.sync()
    counts = d_cnt.cpu().numpy()
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    crop_us, vox_us = float(np.median(times["crop"])), float(np.median(times["voxel"]))
    return dict(extra, entry=kind, w=w, h=h, frames=nf, leaf=leaf, z_limit=limit[1:] if limit else None,
                crop_points=n, voxels_per_frame=float(counts.mean()), crop_us_per_frame=crop_us / nf,
                voxel_us_per_frame=vox_us / nf, voxel_stage_us_per_frame=(vox_us - crop_us) / nf,
                spread_voxel_us=[min(times["voxel"]) / nf, max(times["voxel"]) / nf])


def stream(ctx, h, w, leaf, limit, n_frames, reps):
    ring = d2pc.PinnedArray((16, h, w), np.uint8)
    ring.array[:] = frames_for("mono8", h, w, 16)
    ctx.set_voxel_grid(leaf, 0, limit)
    out = {"crop": [], "voxel": []}
    nbytes = {"crop": 0, "voxel": 0}

    def sink_for(mode):
        def sink(idx, cloud):
            nbytes[mode] += cloud.row_step * cloud.height
        return sink

    for mode in ("crop", "voxel"):
        ctx.set_filter_mode(d2pc.FILTER_CROP if mode == "crop" else d2pc.FILTER_VOXEL)
        ctx.process_stream(ring.array, collect=False, n_frames=32)
    for _ in range(reps):
        for mode in ("crop", "voxel"):
            ctx.set_filter_mode(d2pc.FILTER_CROP if mode == "crop" else d2pc.FILTER_VOXEL)
            nbytes[mode] = 0
            t0 = time.perf_counter()
            ctx.process_stream(ring.array, collect=False, sink=sink_for(mode), n_frames=n_frames)
            out[mode].append(n_frames / (time.perf_counter() - t0))
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ring.free()
    res = {}
    for mode in ("crop", "voxel"):
        d2h = nbytes[mode] / n_frames + (12 if mode == "voxel" else 0)  # the cloud (+ the count / flag fetch)
        res[mode] = {"frames_per_s": float(np.median(out[mode])), "spread": [min(out[mode]), max(out[mode])],
                     "d2h_bytes_per_frame": d2h}
    return res


def lone(ctx, leaf, limit, reps):
    img = synth.s2_scene(480, 752, 1)
    ctx.set_voxel_grid(leaf, 0, limit)
    res = {}
    ts = {"crop": [], "voxel": []}
    for i in range(reps + 20):
        for mode in ("crop", "voxel"):
            ctx.set_filter_mode(d2pc.FILTER_CROP if mode == "crop" else d2pc.FILTER_VOXEL)
            t0 = time.perf_counter()
            ctx.process_mono8(img, copy=False)
            if i >= 20:
                ts[mode].append((time.perf_counter() - t0) * 1e6)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    for mode in ts:
        res[mode] = {"median_us": float(np.median(ts[mode])), "p10_us": float(np.percentile(ts[mode], 10)),
                     "p90_us": float(np.percentile(ts[mode], 90))}
    return res


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
        sizes = [(480, 752, 64), (720, 1280, 64), (2160, 3840, 16)]
        if a.quick:
            sizes = [(480, 752, 4)]
        for h, w, nf in sizes:
            for kind in ("mono8", "f32"):
                for leaf in (0.05, 0.2):
                    for limit in (None, ("z", 0.0, 10.0)):
                        emit(stage(ctx, kind, h, w, nf, leaf, limit, reps, {"case": "a_stage"}))
        for h, w in [(480, 752), (720, 1280)]:
            for leaf, limit in [(0.05, ("z", 0.0, 10.0)), (0.2, None)]:
                r = stream(ctx, h, w, leaf, limit, 200 if a.quick else 3000, 2 if a.quick else 5)
                emit({"case": "b_stream", "entry": "mono8", "w": w, "h": h, "leaf": leaf,
                      "z_limit": limit[1:] if limit else None, **r})
        for leaf, limit in [(0.05, ("z", 0.0, 10.0)), (0.2, None)]:
            emit({"case": "c_lone", "entry": "mono8", "w": 752, "h": 480, "leaf": leaf,
                  "z_limit": limit[1:] if limit else None, **lone(ctx, leaf, limit, 50 if a.quick else 500)})
        for h, w in [(480, 752), (720, 1280)]:
            for kind in ("mono8", "f32"):
                emit(stage(ctx, kind, h, w, 1, 10.0, None, 20 if a.quick else 200, {"case": "d_fold"}))
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
