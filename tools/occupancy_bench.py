"""Measures the occupancy map (octomap_server's insertScan on the device) on the current GPU; one JSON line per case.

    python tools/occupancy_bench.py [--out FILE] [--quick]

(a) map     the map step's time per frame: the first frame into an empty map, and a warm sequence of S2 scene clouds (the library's CROP cloud, transformed
            into a z-up world frame whose origin is 1 m under the camera, optionally VOXEL 0.1 in front) already on the
            device, inserted with d2pc_occupancy_insert_device; a host clock around the whole sequence, ended by a
            device sync.  At 752x480 and 1280x720, resolution 0.05 and 0.1, max_range -1 and 10 m.  With the rays
            (finite points), DDA steps (free cells, from the C recipe) and bricks touched per frame (bricks in use
            after the first frame into an empty map).
(b) cpu     the literal octomap restatement (tests/map_ref, one thread, -O2) on the first frame into an empty map:
            seconds, to set beside the GPU's first frame (the warm sequence was not timed on the CPU).
(c) stream  d2pc_process_stream frames/s at 752x480: CROP alone against transform + map (keep_cloud 0), alternated.
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
import map_ref  # noqa: E402
from disparity_to_point_cloud_b200 import synth  # noqa: E402

ZUP = np.float32([[0, 0, 1, 0], [-1, 0, 0, 0], [0, -1, 0, 1.0]])


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def clouds(ctx, h, w, n, voxel):
    ctx.set_transform(ZUP)
    if voxel:
        ctx.set_voxel_grid(0.1, 0, None)
        ctx.set_filter_mode(d2pc.FILTER_VOXEL)
    out = [ctx.process_mono8(synth.s2_scene(h, w, 100 + i)) for i in range(n)]
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ctx.set_transform(None)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    ctx = d2pc.Context(n_slots=4)
    n_frames = 4 if a.quick else 16
    origin = np.float32([[0, 0, 1.0]])
    for h, w in ((480, 752), (720, 1280)):
        for voxel in (False, True):
            cl = clouds(ctx, h, w, n_frames, voxel)
            n_max = max(len(c) // 16 for c in cl)
            stride = n_max * 16
            host = np.zeros(len(cl) * stride, np.uint8)
            counts = np.zeros(len(cl), np.uint32)
            for f, c in enumerate(cl):
                host[f * stride: f * stride + len(c)] = c
                counts[f] = len(c) // 16
            d_in = torch.from_numpy(host).cuda()
            d_cnt = torch.from_numpy(counts.view(np.int32)).cuda()
            origins = np.repeat(origin, len(cl), 0)
            for res in (0.05, 0.1):
                for max_range in (-1.0, 10.0):
                    ctx.set_occupancy(resolution=res, max_range=max_range, keep_cloud=1)
                    # the first frame into an empty map, as the CPU reference below is timed (once untimed, so that the
                    # table exists and the kernels are loaded)
                    first = []
                    for _ in range(2):
                        ctx.occupancy_reset()
                        ctx.sync()
                        t0 = time.perf_counter()
                        ctx.occupancy_insert_device(d_in.data_ptr(), 1, n_max, stride, d_cnt.data_ptr(), origins[:1])
                        ctx.sync()
                        first.append(time.perf_counter() - t0)
                    bricks = ctx.occupancy_stats()["bricks_used"]
                    # warm: the whole sequence once, then timed twice
                    ctx.occupancy_insert_device(d_in.data_ptr(), len(cl), n_max, stride, d_cnt.data_ptr(), origins)
                    ctx.sync()
                    times = []
                    for _ in range(2):
                        t0 = time.perf_counter()
                        ctx.occupancy_insert_device(d_in.data_ptr(), len(cl), n_max, stride, d_cnt.data_ptr(),
                                                    origins)
                        ctx.sync()
                        times.append((time.perf_counter() - t0) / len(cl))
                    pts = [np.frombuffer(c, np.float32).reshape(-1, 4) for c in cl[:2]]
                    fin = [p[np.isfinite(p[:, :3]).all(1)] for p in pts]
                    steps = np.mean([map_ref.rays_digest(np.repeat(origin, len(p), 0), p[:, :3], res, max_range)[:, 0]
                                     .sum() for p in fin])
                    # the literal single-thread reference on the first frame into an empty map
                    ref = map_ref.Octree(resolution=res, max_range=max_range)
                    t0 = time.perf_counter()
                    ref.insert(cl[0], origin[0])
                    cpu_s = time.perf_counter() - t0
                    st = ctx.occupancy_stats()
                    emit({"case": "map", "h": h, "w": w, "voxel": voxel, "resolution": res, "max_range": max_range,
                          "frames": len(cl), "map_us_per_frame": round(min(times) * 1e6, 1),
                          "map_us_first_frame": round(first[-1] * 1e6, 1),
                          "rays_per_frame": round(float(np.mean([len(p) for p in fin]))),
                          "dda_steps_per_frame": round(float(steps)), "bricks_first_frame": bricks,
                          "cpu_literal_s_first_frame": round(cpu_s, 3), "known_voxels": st["known_voxels"]})
            del d_in, d_cnt
    # (c) the stream at 752x480: CROP against transform + map with keep_cloud 0, alternated
    frames = np.stack([synth.s2_scene(480, 752, 200 + i) for i in range(8)])
    n = 64 if a.quick else 512
    for rep in range(2):
        for setting in ("crop", "map_keep0"):
            ctx.set_occupancy(False)
            ctx.set_transform(None)
            if setting == "map_keep0":
                ctx.set_transform(ZUP)
                ctx.set_occupancy(resolution=0.1, max_range=10.0, keep_cloud=0)
            ctx.process_stream(frames, collect=False, n_frames=16)
            ctx.sync()
            t0 = time.perf_counter()
            ctx.process_stream(frames, collect=False, n_frames=n)
            ctx.sync()
            emit({"case": "stream", "setting": setting, "rep": rep, "h": 480, "w": 752,
                  "frames_per_s": round(n / (time.perf_counter() - t0), 1)})
    ctx.close()
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
