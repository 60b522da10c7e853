"""Measures the laser scan output (pointcloud_to_laserscan on the device) on the current GPU; one JSON line per case.

    python tools/laser_scan_bench.py [--out FILE] [--quick]

(a) stage   scan time per frame: CUDA events around warm d2pc_reproject_mono8_device batches of S2 scene frames (64
            frames, 16 at 4K; CROP + a transform into a z-up frame), with and without d2pc_laser_scan_device on their
            output (alternated), at 752x480, 1280x720 and 3840x2160, with 360 and 3600 bins.  Against the HBM bound of
            the bytes the stage must move: every point read once (16 B) over 7.7 TB/s (HGX B200 data sheet, one GPU).
            The wall case bins a synthetic wall 2 m in front of the camera (every warp's points in a few bins), the
            scan alone on device clouds; the same wall with every point below min_height (each point loaded and
            dropped at the height test, before any FP64 arithmetic) is the kernel's floor without its math.
(b) stream  d2pc_process_stream frames/s (752x480 and 1280x720 mono8), alternated: CROP; transform + scan with
            keep_cloud 0; the same with keep_cloud 1.  With the D2H bytes per frame each setting moves.
(c) lone    one synchronous d2pc_process_mono8 call (median of many), the same three settings, alternated.
(d) launch  kernel launches of one synchronous 752x480 call per plan with the scan on and off.
Every line carries the card's name and power limit, read in the same run."""
from __future__ import annotations

import argparse
import json
import math
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
# camera optical frame -> a z-up body frame 1 m under the camera
ZUP = np.float32([[0, 0, 1, 0], [-1, 0, 0, 0], [0, -1, 0, 1.0]])
BINS = {360: {}, 3600: dict(angle_increment=math.pi / 1800)}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def n_points(w, h, border=40):
    return max(0, w - 2 * border) * max(0, h - 2 * border)


def time_us(ctx, fn, reps):
    s = torch.cuda.ExternalStream(ctx.compute_stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(reps):
        fn()
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def stage(ctx, h, w, nf, bins, reps):
    frames = np.stack([synth.s2_scene(h, w, i) for i in range(nf)])
    n = n_points(w, h)
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.empty(nf * n * 16, dtype=torch.uint8, device="cuda")
    ctx.set_transform(ZUP)
    ctx.set_laser_scan(**BINS[bins])
    nb = d2pc.laser_scan_ranges(**BINS[bins])
    d_rng = torch.empty(nf * nb, dtype=torch.float32, device="cuda")

    def mode():
        ctx.reproject_mono8_device(d_in.data_ptr(), nf, w, h, w, w * h, d_pts.data_ptr(), n * 16, 0)

    def mode_scan():
        mode()
        ctx.laser_scan_device(d_pts.data_ptr(), nf, n, n * 16, 0, d_rng.data_ptr(), nb * 4)

    def scan():
        ctx.laser_scan_device(d_pts.data_ptr(), nf, n, n * 16, 0, d_rng.data_ptr(), nb * 4)

    for f in (mode, mode_scan, scan):
        time_us(ctx, f, 2)
    t = {"mode": [], "mode+scan": [], "scan": []}
    for _ in range(5):
        for k, f in (("mode", mode), ("mode+scan", mode_scan), ("scan", scan)):
            t[k].append(time_us(ctx, f, reps))
    ctx.set_transform(None)
    ctx.set_laser_scan(False)
    med = {k: float(np.median(v)) / nf for k, v in t.items()}
    stage_us = med["mode+scan"] - med["mode"]
    bound_us = 16 * n / HBM_BYTES_PER_S * 1e6
    return dict(case="a_stage", scene="s2", w=w, h=h, frames=nf, bins=nb, points=n, mode="crop+transform",
                mode_us_per_frame=med["mode"], mode_plus_scan_us_per_frame=med["mode+scan"],
                stage_us_per_frame=stage_us, scan_alone_us_per_frame=med["scan"],
                spread_us_per_frame={k: [min(v) / nf, max(v) / nf] for k, v in t.items()},
                hbm_bound_us_per_frame=bound_us, share_of_hbm_bound=bound_us / stage_us if stage_us > 0 else None)


def wall(ctx, n, nf, bins, reps, below=False):
    rng = np.random.default_rng(5)
    pts = np.empty((nf, n, 4), np.float32)
    pts[..., 0] = 2.0 + rng.normal(0, 0.01, (nf, n))
    pts[..., 1] = rng.uniform(-0.3, 0.3, (nf, n))  # about +-8.5 degrees: 17 of 360 bins
    pts[..., 2] = rng.uniform(0.05, 1.5, (nf, n)) * (-1 if below else 1)
    pts[..., 3] = 1.0
    d_pts = torch.from_numpy(pts.reshape(-1)).cuda()
    ctx.set_laser_scan(**BINS[bins])
    nb = d2pc.laser_scan_ranges(**BINS[bins])
    d_rng = torch.empty(nf * nb, dtype=torch.float32, device="cuda")

    def scan():
        ctx.laser_scan_device(d_pts.data_ptr(), nf, n, n * 16, 0, d_rng.data_ptr(), nb * 4)

    time_us(ctx, scan, 2)
    t = [time_us(ctx, scan, reps) / nf for _ in range(5)]
    ctx.set_laser_scan(False)
    bound_us = 16 * n / HBM_BYTES_PER_S * 1e6
    return dict(case="a_stage", scene="wall below min_height" if below else "wall", points=n, frames=nf, bins=nb, scan_alone_us_per_frame=float(np.median(t)),
                spread_us_per_frame=[min(t), max(t)], hbm_bound_us_per_frame=bound_us,
                share_of_hbm_bound=bound_us / float(np.median(t)))


SETTINGS = {"crop": None, "transform+scan keep_cloud 0": 0, "transform+scan keep_cloud 1": 1}


def apply(ctx, keep):
    if keep is None:
        ctx.set_transform(None)
        ctx.set_laser_scan(False)
    else:
        ctx.set_transform(ZUP)
        ctx.set_laser_scan(keep_cloud=keep)


def d2h_bytes(w, h, keep):
    cloud = 16 * n_points(w, h)
    return cloud if keep is None else 4 * 360 + (cloud if keep else 0)


def stream(ctx, h, w, n_frames, reps):
    ring = d2pc.PinnedArray((16, h, w), np.uint8)
    ring.array[:] = np.stack([synth.s2_scene(h, w, i) for i in range(16)])
    out = {k: [] for k in SETTINGS}
    for k, keep in SETTINGS.items():
        apply(ctx, keep)
        ctx.process_stream(ring.array, collect=False, n_frames=32)
    for _ in range(reps):
        for k, keep in SETTINGS.items():
            apply(ctx, keep)
            t0 = time.perf_counter()
            ctx.process_stream(ring.array, collect=False, n_frames=n_frames)
            out[k].append(n_frames / (time.perf_counter() - t0))
    apply(ctx, None)
    ring.free()
    return {k: {"frames_per_s": float(np.median(v)), "spread": [min(v), max(v)],
                "d2h_bytes_per_frame": d2h_bytes(w, h, SETTINGS[k])} for k, v in out.items()}


def lone(ctx, h, w, reps):
    img = synth.s2_scene(h, w, 1)
    ts = {k: [] for k in SETTINGS}
    for i in range(reps + 20):
        for k, keep in SETTINGS.items():
            apply(ctx, keep)
            t0 = time.perf_counter()
            ctx.process_mono8(img, copy=False)
            if i >= 20:
                ts[k].append((time.perf_counter() - t0) * 1e6)
    apply(ctx, None)
    return {k: {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)),
                "p90_us": float(np.percentile(v, 90)), "d2h_bytes": d2h_bytes(w, h, SETTINGS[k])}
            for k, v in ts.items()}


def launches(ctx):
    img = synth.s2_scene(480, 752, 1)
    ctx.set_voxel_grid(0.05, 0, ("z", -10.0, 10.0))
    out = {}
    for name, mode in (("crop", d2pc.FILTER_CROP), ("finite", d2pc.FILTER_CROP_FINITE), ("voxel", d2pc.FILTER_VOXEL)):
        ctx.set_filter_mode(mode)
        for label, xf, keep in (("", None, None), ("+transform", ZUP, None), ("+transform+scan keep_cloud 0", ZUP, 0),
                                ("+transform+scan keep_cloud 1", ZUP, 1)):
            ctx.set_transform(xf)
            ctx.set_laser_scan(keep is not None, keep_cloud=1 if keep is None else keep)
            n0 = ctx.launch_count()
            ctx.process_mono8(img)
            out[name + label] = ctx.launch_count() - n0
    apply(ctx, None)
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
            for bins in BINS:
                emit(stage(ctx, h, w, nf, bins, reps))
        for bins in BINS:
            for below in (False, True):
                emit(wall(ctx, n_points(752, 480), 4 if a.quick else 64, bins, reps, below))
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
