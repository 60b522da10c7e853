#!/usr/bin/env python
"""Memory ceiling of the CROP kernel's traffic: the kernel with its arithmetic replaced by {d, d, d, 1} stores
(tuning key crop_probe), run the way bench.py runs config 4 -- 3840x2160 float frames, 16 per launch from a 16-frame
ring larger than L2, 320 launches back to back, CUDA events -- next to the real kernel in the same harness.

    python tools/crop_ceiling.py [rows,...] [crop_load,...] [out.jsonl]

One JSON line per (probe, rows per unit, load path): fraction of the measured 1:1 copy peak, SM clock and the
throttle reasons sampled during the timed launches, card name and power limit.
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, ".")
sys.path.insert(0, "tools")
import torch  # noqa: E402

import bench  # noqa: E402
import disparity_to_point_cloud_b200 as d2pc  # noqa: E402
import timing  # noqa: E402

W, H, RING, LAUNCHES, WARM = 3840, 2160, 16, 320, 64


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return [c.strip() for c in q.split(",")]


def main():
    rows_list = [int(x) for x in sys.argv[1].split(",")] if len(sys.argv) > 1 else [4, 8]
    load_list = [int(x) for x in sys.argv[2].split(",")] if len(sys.argv) > 2 else [1, 0]
    out_path = sys.argv[3] if len(sys.argv) > 3 else ""
    name, power_limit, max_sm = card()
    ctx = d2pc.Context()
    stream = torch.cuda.ExternalStream(ctx.compute_stream())
    n = (W - 80) * (H - 80)
    d_in = timing.float_batch(W, H, RING)
    d_out = torch.empty((RING, n * 16), dtype=torch.uint8, device="cuda")
    peak, _ = bench.measured_peak()

    def launch():
        ctx.reproject_f32_device(d_in.data_ptr(), RING, W, H, W * 4, W * H * 4, d_out.data_ptr(), n * 16)

    for probe in (1, 0):
        for rows in rows_list:
            for load in load_list:
                ctx.set_tuning("crop_probe", probe)
                ctx.set_tuning("rows_per_unit", rows)
                ctx.set_tuning("crop_load", load)
                for _ in range(WARM):
                    launch()
                torch.cuda.synchronize()
                sampler = bench.ClockSampler(0)
                sampler.start()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(LAUNCHES):
                    launch()
                e1.record(stream)
                torch.cuda.synchronize()
                clocks = sampler.stop()
                s = e0.elapsed_time(e1) * 1e-3 / LAUNCHES
                gbs = 20 * n * RING / s / 1e9
                line = {"probe": bool(probe), "rows_per_unit": rows, "crop_load": "ldg" if load else "tma",
                        "launch_us": round(s * 1e6, 1), "gbs": round(gbs, 1), "frac_of_copy_peak": round(gbs / peak, 4),
                        "copy_peak_gbs": peak, "launches": LAUNCHES, "frames_per_launch": RING, "shape": [W, H],
                        "gpu": name, "power_limit": power_limit, "sm_max_clock": max_sm, "clocks": clocks}
                print(json.dumps(line), flush=True)
                if out_path:
                    with open(out_path, "a") as fh:
                        fh.write(json.dumps(line) + "\n")
    ctx.set_tuning("crop_probe", 0)
    ctx.set_tuning("rows_per_unit", 0)
    ctx.set_tuning("crop_load", 0)


if __name__ == "__main__":
    main()
