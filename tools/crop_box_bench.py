"""Measures the crop box stage (pcl::CropBox in front of VOXEL and the outlier stage) on the current GPU; one JSON line
per case.

    python tools/crop_box_bench.py [--out FILE] [--quick]

(a) stage   stage time per frame: CUDA events around warm d2pc_reproject_mono8_device batches of S2 scene frames (64
            frames, 16 at 4K) with the box on, minus the same batches in CROP mode (alternated), at 752x480, 1280x720
            and 3840x2160, for boxes keeping about 100 %, 50 % and 10 % of the finite points, identity and rotated.
            Against the HBM bound of the bytes the stage moves: the predicate scan reads every point (16 B) and
            writes a slot (4 B), the scatter reads every point and slot again (20 B) and writes the kept points
            (16 B each); over 7.7 TB/s (HGX B200 data sheet, one GPU).
(b) stream  d2pc_process_stream frames/s and device-to-host bytes per frame: CROP, CROP_FINITE, CROP + box at those
            fractions (752x480 and 1280x720 mono8).
(c) lone    one synchronous 752x480 d2pc_process_mono8 call: CROP against CROP + box (median of many).
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
FRACTIONS = (1.0, 0.5, 0.1)
GRID = (0.05, 0, ("z", 0.0, 10.0))


def rotated(roll=0.3, pitch=-0.2, yaw=0.5, t=(0.1, -0.2, 0.3)) -> np.ndarray:
    """[Rz(yaw) Ry(pitch) Rx(roll) | t] in float32."""
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    r = [[cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr], [sy * cp, sy * sp * sr + cy * cr,
         sy * sp * cr - cy * sr], [-sp, cp * sr, cp * cr]]
    return np.concatenate([r, np.reshape(t, (3, 1))], axis=1).astype(np.float32)


ROTATED = rotated()


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def n_points(w, h, border=40):
    return max(0, w - 2 * border) * max(0, h - 2 * border)


def frames_for(h, w, nf):
    return np.stack([synth.s2_scene(h, w, i) for i in range(nf)])


def box_for(ctx, img, frac, t):
    """min / max of T p (float64 quantiles) that keep about `frac` of the finite points of img's CROP cloud."""
    ctx.set_crop_box(None)
    ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
    pts = np.frombuffer(ctx.process_mono8(img).tobytes(), np.float32).reshape(-1, 4)[:, :3].astype(np.float64)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    tt = np.eye(3, 4) if t is None else t.astype(np.float64)
    loc = pts @ tt[:, :3].T + tt[:, 3]
    side = frac ** (1 / 3)
    lo, hi = (1 - side) / 2, (1 + side) / 2
    mn = np.quantile(loc, lo, axis=0) if frac < 1 else loc.min(0) - 1
    mx = np.quantile(loc, hi, axis=0) if frac < 1 else loc.max(0) + 1
    return mn, mx, t


def time_batch(ctx, fn, args, reps):
    s = torch.cuda.ExternalStream(ctx.compute_stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(reps):
        fn(*args)
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps  # us per batch


def stage(ctx, h, w, nf, frac, rotated, reps):
    frames = frames_for(h, w, nf)
    n = n_points(w, h)
    box = box_for(ctx, frames[0], frac, ROTATED if rotated else None)
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.empty(nf * n * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
    args = (d_in.data_ptr(), nf, w, h, w, w * h, d_pts.data_ptr(), n * 16, d_cnt.data_ptr())
    times = {"off": [], "on": []}
    kept = 0.0
    for on in ("off", "on"):  # warm both (module load, scratch sizing)
        ctx.set_crop_box(*(box if on == "on" else (None,)))
        time_batch(ctx, ctx.reproject_mono8_device, args, 2)
        ctx.sync()
    kept = float(d_cnt.cpu().numpy().mean())
    for _ in range(5):
        for on in ("off", "on"):
            ctx.set_crop_box(*(box if on == "on" else (None,)))
            times[on].append(time_batch(ctx, ctx.reproject_mono8_device, args, reps))
    ctx.set_crop_box(None)
    off_us, on_us = float(np.median(times["off"])), float(np.median(times["on"]))
    stage_us = (on_us - off_us) / nf
    bytes_per_frame = 16 * n + 4 * (n + 1) + 20 * n + 16 * kept
    bound_us = bytes_per_frame / HBM_BYTES_PER_S * 1e6
    return dict(case="a_stage", w=w, h=h, frames=nf, fraction=frac, rotated=rotated, crop_points=n,
                kept_points_per_frame=kept, kept_share_of_crop=kept / n, crop_us_per_frame=off_us / nf,
                crop_plus_box_us_per_frame=on_us / nf, stage_us_per_frame=stage_us,
                spread_on_us=[min(times["on"]) / nf, max(times["on"]) / nf],
                stage_bytes_per_frame=bytes_per_frame, hbm_bound_us_per_frame=bound_us,
                share_of_hbm_bound=bound_us / stage_us if stage_us > 0 else None)


def stream(ctx, h, w, n_frames, reps):
    ring = d2pc.PinnedArray((16, h, w), np.uint8)
    ring.array[:] = frames_for(h, w, 16)
    boxes = {f: box_for(ctx, ring.array[0], f, ROTATED) for f in FRACTIONS}
    cases = {"crop": (d2pc.FILTER_CROP, None), "finite": (d2pc.FILTER_CROP_FINITE, None)}
    cases.update({f"crop+box{int(f * 100)}": (d2pc.FILTER_CROP, boxes[f]) for f in FRACTIONS})
    out = {k: [] for k in cases}
    nbytes = {k: 0 for k in cases}

    def sink_for(k):
        def sink(idx, cloud):
            nbytes[k] += cloud.row_step * cloud.height
        return sink

    def setup(k):
        mode, box = cases[k]
        ctx.set_filter_mode(mode)
        ctx.set_crop_box(*(box or (None,)))

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
    ctx.set_crop_box(None)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ring.free()
    return {k: {"frames_per_s": float(np.median(out[k])), "spread": [min(out[k]), max(out[k])],
                "d2h_bytes_per_frame": nbytes[k] / n_frames + (4 if k != "crop" else 0)}  # + the count fetch
            for k in cases}


def lone(ctx, reps):
    img = synth.s2_scene(480, 752, 1)
    boxes = {f"crop+box{int(f * 100)}": box_for(ctx, img, f, ROTATED) for f in FRACTIONS}
    boxes["crop"] = None
    ts = {k: [] for k in boxes}
    for i in range(reps + 20):
        for k, box in boxes.items():
            ctx.set_crop_box(*(box or (None,)))
            t0 = time.perf_counter()
            ctx.process_mono8(img, copy=False)
            if i >= 20:
                ts[k].append((time.perf_counter() - t0) * 1e6)
    ctx.set_crop_box(None)
    return {k: {"median_us": float(np.median(v)), "p10_us": float(np.percentile(v, 10)),
                "p90_us": float(np.percentile(v, 90))} for k, v in ts.items()}


def launches(ctx):
    img = synth.s2_scene(480, 752, 1)
    box = box_for(ctx, img, 0.5, ROTATED)
    ctx.set_voxel_grid(*GRID)
    plans = {"crop": (d2pc.FILTER_CROP, None, 0.0), "finite": (d2pc.FILTER_CROP_FINITE, None, 0.0),
             "voxel": (d2pc.FILTER_VOXEL, None, 0.0), "crop+box": (d2pc.FILTER_CROP, box, 0.0),
             "finite+box": (d2pc.FILTER_CROP_FINITE, box, 0.0), "voxel+box": (d2pc.FILTER_VOXEL, box, 0.0),
             "crop+box+outlier": (d2pc.FILTER_CROP, box, 0.1), "voxel+box+outlier": (d2pc.FILTER_VOXEL, box, 0.1)}
    out = {}
    for k, (mode, b, r) in plans.items():
        ctx.set_filter_mode(mode)
        ctx.set_crop_box(*(b or (None,)))
        ctx.set_radius_outlier(r, 2)
        n0 = ctx.launch_count()
        ctx.process_mono8(img)
        out[k] = ctx.launch_count() - n0
    ctx.set_crop_box(None)
    ctx.set_radius_outlier(0.0)
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
            for frac in FRACTIONS:
                for rotated in (False, True):
                    emit(stage(ctx, h, w, nf, frac, rotated, reps))
        for h, w in [(480, 752), (720, 1280)]:
            r = stream(ctx, h, w, 200 if a.quick else 3000, 2 if a.quick else 5)
            emit({"case": "b_stream", "entry": "mono8", "w": w, "h": h, **r})
        emit({"case": "c_lone", "entry": "mono8", "w": 752, "h": 480, **lone(ctx, 50 if a.quick else 500)})
        emit({"case": "d_launches", "entry": "mono8", "w": 752, "h": 480, **launches(ctx)})
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
