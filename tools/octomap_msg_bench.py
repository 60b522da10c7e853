"""Measures d2pc_occupancy_octomap (the map as octomap_msgs/Octomap) on the current GPU; one JSON line per case.

    python tools/octomap_msg_bench.py [--out FILE] [--quick]

Maps of about 10^5, 10^6 and 10^7 known voxels (resolution 0.05), built with d2pc_occupancy_insert_device from
seeded rays that repeat from nearby origins, so free space clamps and the tree prunes.  Per map and format:
  - call_ms   the call's host wall time (it is synchronous: count, sort, tree, D2H into pinned memory), median of reps;
  - device_ms the summed time of the call's kernels and copies, and `launches` its kernel launches (CUB's included),
              from torch.profiler in a separate pass;
  - cpu_ms    octomap's pointer tree (tests/map_ref/octree_pointer.cpp, one core, -O2) writing the same tree with
              writeData / writeBinaryData, the tree loaded from the library's full stream;
  - centres_ms d2pc_occupancy_centers on the same map, for scale.
Every line carries the card's name and power limit, read in the same run."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import disparity_to_point_cloud_b200 as d2pc  # noqa: E402
from map_ref import octree  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def build_map(ctx, target, seed):
    """frames of 20000 rays from origins within 0.3 m of a centre until the map knows `target` voxels"""
    rng = np.random.default_rng(seed)
    reach = 1.0 + 2.0 * np.log10(target / 1e5 + 1) ** 1.5
    frames = 0
    while ctx.occupancy_stats()["known_voxels"] < target and frames < 400:
        o = rng.uniform(-0.3, 0.3, 3).astype(np.float32)
        d = rng.normal(size=(20000, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        pts = np.concatenate([o + d * rng.uniform(0.3, reach * (1 + frames / 20), (20000, 1)),
                              np.ones((20000, 1))], 1).astype(np.float32)
        dev = torch.from_numpy(pts.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(dev.data_ptr(), 1, 20000, 20000 * 16, 0, o.reshape(1, 3))
        frames += 1
    return frames


def profile(fn):
    from torch.profiler import ProfilerActivity, profile as prof
    with prof(activities=[ProfilerActivity.CUDA]) as p:
        fn()
        torch.cuda.synchronize()
    kernels = [e for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    launches = sum(1 for e in kernels if "memcpy" not in e.name.lower() and "memset" not in e.name.lower())
    return sum(e.device_time for e in kernels) / 1000.0, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    info = card()
    out = open(a.out, "w") if a.out else None
    targets = [10 ** 5, 10 ** 6] if a.quick else [10 ** 5, 10 ** 6, 10 ** 7]
    reps = 3 if a.quick else 9
    ctx = d2pc.Context()
    lib = octree._lib("octree_pointer.cpp")
    for ti, target in enumerate(targets):
        ctx.set_occupancy(resolution=0.05, max_bricks=1 << 20)
        ctx.occupancy_reset()
        frames = build_map(ctx, target, 11 + ti)
        st = ctx.occupancy_stats()
        tree = octree.PointerTree(resolution=0.05)
        full = ctx.occupancy_octomap()
        tree.load(full)
        depths = [0] * 17
        tree.voxels(depths)
        for binary in (False, True):
            ctx.occupancy_octomap(binary=binary)  # warm-up: buffers grown, modules loaded
            walls = []
            for _ in range(reps):
                t0 = time.perf_counter()
                data = ctx.occupancy_octomap(binary=binary)
                walls.append((time.perf_counter() - t0) * 1e3)
            device_ms, launches = profile(lambda: ctx.occupancy_octomap(binary=binary))
            assert data == tree.data(binary)
            cpu = []
            for _ in range(3):
                p = C.c_void_p()
                t0 = time.perf_counter()
                lib.ptr_write(tree._h, 1 if binary else 0, C.byref(p))
                cpu.append((time.perf_counter() - t0) * 1e3)
            cw = []
            for _ in range(reps):
                t0 = time.perf_counter()
                ctx.occupancy_centers()
                cw.append((time.perf_counter() - t0) * 1e3)
            rec = dict(case="octomap_msg", format="binary" if binary else "full", known_voxels=st["known_voxels"],
                       occupied_voxels=st["occupied_voxels"], frames=frames, bytes=len(data),
                       leaves_above_depth16=sum(depths[:16]), call_ms=round(statistics.median(walls), 3),
                       call_ms_min=round(min(walls), 3), device_ms=round(device_ms, 3), launches=launches,
                       cpu_ms=round(statistics.median(cpu), 3), centres_ms=round(statistics.median(cw), 3), **info)
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
    ctx.close()
    if out:
        out.close()


if __name__ == "__main__":
    main()
