"""Measures the radius outlier stage (pcl::RadiusOutlierRemoval behind the filter mode) on the current GPU; one
JSON line per case.

    python tools/radius_outlier_bench.py [--out FILE] [--quick]

(a) stage   stage time per frame: CUDA events around d2pc_reproject_mono8_device batches of S2 scene frames
            (64 frames, 16 at 4K) with the stage on, minus the same batches with it off (alternated, warm), for
            CROP_FINITE and VOXEL (leaf 0.05 m, z in [0, 10] m) inputs; radius 0.05 / 0.1 / 0.2 m, min_neighbors
            2 / 5 / 10.
(b) stream  d2pc_process_stream frames/s and device-to-host bytes per frame: CROP, CROP_FINITE, CROP_FINITE + stage.
(c) lone    one synchronous 752x480 d2pc_process_mono8 call, CROP vs CROP + stage (median of many).
(d) worst   a 10 m radius with min_neighbors 1000: few cells, each holding most of the frame.
(e) cpu     the C reference of tests/outlier_ref (grid, one CPU core) on the same CROP_FINITE / VOXEL clouds; the
            repository's own reference, not PCL.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import disparity_to_point_cloud_b200 as d2pc  # noqa: E402
from disparity_to_point_cloud_b200 import synth  # noqa: E402

GRID = (0.05, 0, ("z", 0.0, 10.0))
MODES = {"crop": d2pc.FILTER_CROP, "finite": d2pc.FILTER_CROP_FINITE, "voxel": d2pc.FILTER_VOXEL}


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


def stage(ctx, mode, h, w, nf, radius, mn, reps, extra):
    frames = frames_for(h, w, nf)
    n = n_points(w, h)
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.empty(nf * n * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
    args = (d_in.data_ptr(), nf, w, h, w, w * h, d_pts.data_ptr(), n * 16, d_cnt.data_ptr())
    ctx.set_voxel_grid(*GRID)
    ctx.set_filter_mode(MODES[mode])
    times = {"off": [], "on": []}
    counts = {}
    for on in ("off", "on"):  # warm both (module load, scratch sizing) and keep the counts
        ctx.set_radius_outlier(radius if on == "on" else 0.0, mn)
        time_batch(ctx, ctx.reproject_mono8_device, args, 2)
        ctx.sync()
        counts[on] = float(d_cnt.cpu().numpy().mean())
    for _ in range(5):
        for on in ("off", "on"):
            ctx.set_radius_outlier(radius if on == "on" else 0.0, mn)
            times[on].append(time_batch(ctx, ctx.reproject_mono8_device, args, reps))
    ctx.set_radius_outlier(0.0)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    off_us, on_us = float(np.median(times["off"])), float(np.median(times["on"]))
    return dict(extra, mode=mode, w=w, h=h, frames=nf, radius=radius, min_neighbors=mn, crop_points=n,
                input_points_per_frame=counts["off"], kept_points_per_frame=counts["on"],
                mode_us_per_frame=off_us / nf, mode_plus_stage_us_per_frame=on_us / nf,
                stage_us_per_frame=(on_us - off_us) / nf, spread_on_us=[min(times["on"]) / nf, max(times["on"]) / nf])


def stream(ctx, h, w, radius, mn, n_frames, reps):
    ring = d2pc.PinnedArray((16, h, w), np.uint8)
    ring.array[:] = frames_for(h, w, 16)
    cases = {"crop": ("crop", 0.0), "finite": ("finite", 0.0), "finite+stage": ("finite", radius)}
    out = {k: [] for k in cases}
    nbytes = {k: 0 for k in cases}

    def sink_for(k):
        def sink(idx, cloud):
            nbytes[k] += cloud.row_step * cloud.height
        return sink

    def setup(k):
        mode, r = cases[k]
        ctx.set_filter_mode(MODES[mode])
        ctx.set_radius_outlier(r, mn)

    for k in cases:
        setup(k)
        ctx.process_stream(ring.array, collect=False, n_frames=32)
    for _ in range(reps):
        for k in cases:
            setup(k)
            nbytes[k] = 0
            t0 = time.perf_counter()
            ctx.process_stream(ring.array, collect=False, sink=sink_for(k), n_frames=n_frames)
            out[k].append(n_frames / (time.perf_counter() - t0))
    ctx.set_radius_outlier(0.0)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ring.free()
    return {k: {"frames_per_s": float(np.median(out[k])), "spread": [min(out[k]), max(out[k])],
                "d2h_bytes_per_frame": nbytes[k] / n_frames + (4 if k != "crop" else 0)}  # + the count fetch
            for k in cases}


def lone(ctx, radius, mn, reps):
    img = synth.s2_scene(480, 752, 1)
    ts = {"crop": [], "crop+stage": []}
    for i in range(reps + 20):
        for k in ts:
            ctx.set_radius_outlier(radius if k == "crop+stage" else 0.0, mn)
            t0 = time.perf_counter()
            ctx.process_mono8(img, copy=False)
            if i >= 20:
                ts[k].append((time.perf_counter() - t0) * 1e6)
    ctx.set_radius_outlier(0.0)
    return {k: {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)),
                "p90_us": float(np.percentile(v, 90))} for k, v in ts.items()}


def cpu_reference(ctx, mode, h, w, radius, mn):
    import outlier_ref
    img = synth.s2_scene(h, w, 0)
    ctx.set_voxel_grid(*GRID)
    ctx.set_filter_mode(MODES[mode])
    cloud = ctx.process_mono8(img)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    outlier_ref.radius_outlier(cloud[:16 * 100], radius, mn)  # compile / load outside the timed call
    t0 = time.perf_counter()
    kept = outlier_ref.radius_outlier(cloud, radius, mn)
    return {"case": "e_cpu_reference_one_core", "mode": mode, "w": w, "h": h, "radius": radius, "min_neighbors": mn,
            "input_points": len(cloud) // 16, "kept_points": len(kept) // 16,
            "ms_per_frame": (time.perf_counter() - t0) * 1e3}


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
        sizes = [(480, 752, 4)] if a.quick else [(480, 752, 64), (720, 1280, 64)]
        for h, w, nf in sizes:
            for mode in ("finite", "voxel"):
                for radius in (0.05, 0.1, 0.2):
                    for mn in (2, 5, 10):
                        emit(stage(ctx, mode, h, w, nf, radius, mn, reps, {"case": "a_stage"}))
        if not a.quick:
            for mode in ("finite", "voxel"):
                emit(stage(ctx, mode, 2160, 3840, 16, 0.1, 5, reps, {"case": "a_stage"}))
        for h, w in [(480, 752), (720, 1280)]:
            r = stream(ctx, h, w, 0.05, 5, 200 if a.quick else 3000, 2 if a.quick else 5)
            emit({"case": "b_stream", "entry": "mono8", "w": w, "h": h, "radius": 0.05, "min_neighbors": 5, **r})
        emit({"case": "c_lone", "entry": "mono8", "w": 752, "h": 480, "radius": 0.05, "min_neighbors": 5,
              **lone(ctx, 0.05, 5, 50 if a.quick else 500)})
        for h, w in [(480, 752), (720, 1280)]:
            emit(stage(ctx, "finite", h, w, 1, 10.0, 1000, 5 if a.quick else 50, {"case": "d_worst"}))
        for h, w in [(480, 752), (720, 1280)]:
            for mode in ("finite", "voxel"):
                for radius in (0.05, 0.2):
                    emit(dict(cpu_reference(ctx, mode, h, w, radius, 5), **{"cpu_cores": 1}))
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
