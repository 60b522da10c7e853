"""Measures d2pc_occupancy_projected_map (the map as nav_msgs/OccupancyGrid) on the current GPU; one JSON line per case.

    python tools/projected_map_bench.py [--out FILE] [--quick]

Maps of about 10^5, 10^6 and 10^7 known voxels (resolution 0.05), built as tools/octomap_msg_bench.py builds them:
d2pc_occupancy_insert_device from seeded rays that repeat from nearby origins, so free space clamps and the tree prunes.
Per map, with octomap_server's default limits and with finite z limits and padding:
  - call_ms   the call's host wall time (it is synchronous: count, sort, levels, extent read back, fill, D2H of the
              cells into pinned memory), median of reps;
  - device_ms the summed time of the call's kernels and copies, and `launches` its kernel launches (CUB's included),
              from torch.profiler in a separate pass;
  - width, height, cells: the grid's size;
  - cpu_ms    octomap_server's projection restated over octomap's pointer tree (tests/map_ref/projected_map.cpp, one
              core, -O2) on the same tree, loaded from the library's full octomap stream.
Every line carries the card's name and power limit, read in the same run."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import disparity_to_point_cloud_b200 as d2pc  # noqa: E402
from map_ref import projected  # noqa: E402
from octomap_msg_bench import build_map, card, profile  # noqa: E402

CASES = {"default": dict(), "limits": dict(occupancy_min_z=-0.5, occupancy_max_z=0.5, min_x_size=40.0, min_y_size=40.0)}


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
    for ti, target in enumerate(targets):
        ctx.set_occupancy(resolution=0.05, max_bricks=1 << 20)
        ctx.occupancy_reset()
        frames = build_map(ctx, target, 11 + ti)
        st = ctx.occupancy_stats()
        tree = projected.ProjTree(resolution=0.05)
        tree.load(ctx.occupancy_octomap())
        depths = [0] * 17
        tree.voxels(depths)
        for name, kw in CASES.items():
            ctx.occupancy_projected_map(**kw)  # warm-up: buffers grown, modules loaded
            walls = []
            for _ in range(reps):
                t0 = time.perf_counter()
                cells, res, origin = ctx.occupancy_projected_map(**kw)
                walls.append((time.perf_counter() - t0) * 1e3)
            device_ms, launches = profile(lambda: ctx.occupancy_projected_map(**kw))
            cpu = []
            for _ in range(3):
                t0 = time.perf_counter()
                want = tree.projected_map(**kw)
                cpu.append((time.perf_counter() - t0) * 1e3)
            assert cells.tobytes() == want[0].tobytes() and np.float64(origin).tobytes() == np.float64(want[2]).tobytes()
            rec = dict(case="projected_map", limits=name, known_voxels=st["known_voxels"],
                       occupied_voxels=st["occupied_voxels"], frames=frames, leaves_above_depth16=sum(depths[:16]),
                       width=int(cells.shape[1]), height=int(cells.shape[0]), cells=int(cells.size),
                       occupied_cells=int((cells == 100).sum()), free_cells=int((cells == 0).sum()),
                       call_ms=round(statistics.median(walls), 3), call_ms_min=round(min(walls), 3),
                       device_ms=round(device_ms, 3), launches=launches, cpu_ms=round(statistics.median(cpu), 3),
                       **info)
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
    ctx.close()
    if out:
        out.close()


if __name__ == "__main__":
    main()
