#!/usr/bin/env python
"""bench.py -- disparity -> PointCloud2 throughput (BASELINE.json's metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dump-outputs DIR]
    (N > 1 is launched under torch.distributed.run, one rank per GPU)

--config selects the BASELINE.json workload (numbered as SURVEY.md section 8 numbers them, = configs[N-1]); every
config prints ONE JSON line with the same keys (value, e2e, roofline, cpu_baseline, clocks ...):

  4 (default, the headline the 1/2/4/8-GPU metric is quoted on): 3840x2160 float32 disparity frames (S3) through
    the reference's reprojection path (src/disparity_to_point_cloud.cpp:63-85): reproject with Q -> 40-px crop ->
    pack {x,y,z,1.0f}.  A step is 1024 frames PER GPU (weak scaling; --scaling strong shards 1024 in total).
  3: 1280x720 float32, a step is one batch of 64 frames (kernel-only is what BASELINE quotes; e2e reported too).
  2: 752x480 mono8 stream (S2 scene), the whole DisparityCb (cpp:46-92: median 11 -> x1/8 -> reproject -> crop ->
     pack); a step is 1000 frames.
  5: depth_map_fusion: four 1280x720 mono8 maps per frame set -> MatchingScoreCb1/2, DisparityCb1/2,
     publishFusedDepthMap (src/depth_map_fusion.cpp:46-136) -> DisparityCb on the fused 665x665 map; a step is 256
     frame sets PER GPU, frame sets sharded over the GPUs.

  value      Mpixel/s of input pixels, kernel-only: inputs resident in HBM in a ring larger than L2 (every launch
             streams from HBM), CUDA events on the launching stream, max over ranks.
  e2e        the same metric through the C ABI's host entry (d2pc_process_stream / d2pc_process_fusion_stream):
             pinned host frames, H2D, kernels, D2H of every PointCloud2 payload, three streams / slots overlapped.
             Wall clock bracketed by device synchronisation (the work spans three streams), max over ranks.
             e2e.ceiling_gbs is the raw rate of plain pinned cudaMemcpyAsync traffic of the same shape (same bytes
             per frame each way, all ranks at once): what the host / PCIe path can carry with no kernels at all.
  roofline   algorithmic bytes (SURVEY.md 8(d)) / measured kernel time vs the measured HBM peak.
  cpu_baseline  the CPU oracle port of the same path on a bounded sample, timed on this host (N=1, rank 0).

--dump-outputs DIR writes, after the timed steps, what the kernel-only leg computed in its last step, as its caller
receives it: the clouds, (units, points, 4) {x, y, z, 1.0f} with one row per unit of the device-resident ring, and for
config 5 also the per-lane results of the last frame set each lane ran (cropped_score.npy, fused_depth_map.npy,
combined_score.npy, as float32).  A zero disparity reprojects to +-inf and NaN (the reference publishes such points),
so a cloud is written as two finite float32 arrays of its shape: cloud.npy holds every finite component and 0 in place
of a non-finite one, cloud_nonfinite.npy says which is which (0 finite, 1 +inf, -1 -inf, 2 NaN).  At most 64 MB in all:
a cloud larger than what is left keeps a fixed, seeded sample of its points (the same points of every unit).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.  Rank 0 writes;
nothing is written in the repository unless DIR is in it.

--impl reference times the CPU oracle port with all host threads on the same workload, a bounded sample per step
(same sample rule as cpu_baseline).  The reference's own glue is compiled from its sources in oracle/_ref, but its
arithmetic lives in OpenCV / PCL, which this image does not have: the timed code is the cv2-pinned C port.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BORDER = 40
METRIC = "Mpixels/s disparity->PointCloud2"
DUMP_BYTES = 64 * 10**6  # --dump-outputs: all files together

# name, frame size, entry, frames (frame sets) per step per GPU, device-resident ring, workload string (shared by
# both arms, byte for byte), what one unit of work is
CONFIGS = {
    2: dict(w=752, h=480, entry="mono8", per_step=1000, ring=250,
            workload="752x480 mono8 disparity stream (S2 scene): whole DisparityCb = median 11 + x1/8 + reproject + "
                     "40px crop + XYZ1 pack (BASELINE configs[1])",
            kernel="median_hist_kernel<11, fused>: median + x1/8 + reproject + pack in one launch"),
    3: dict(w=1280, h=720, entry="f32", per_step=64, ring=64,
            workload="1280x720 float32 disparity (S3), batch of 64 frames: reproject + 40px crop + XYZ1 pack "
                     "(BASELINE configs[2])",
            kernel="reproject_crop_kernel<float,vec16,exact-rectified>"),
    4: dict(w=3840, h=2160, entry="f32", per_step=1024, ring=16,
            workload="3840x2160 float32 disparity (S3): reproject + 40px crop + XYZ1 pack (BASELINE configs[3])",
            kernel="reproject_crop_kernel<float,vec16,exact-rectified>"),
    5: dict(w=1280, h=720, entry="fusion", per_step=256, ring=64,
            workload="depth_map_fusion: four 1280x720 mono8 maps per frame set -> score preprocessing x2, merge, "
                     "median 3, trim -> DisparityCb on the fused 665x665 map (BASELINE configs[4])",
            kernel="score_tile_kernel x2 + fuse_merge_kernel + median3_net_kernel + median_hist_kernel<11, fused> "
                   "(median + x1/8 + reproject + pack)"),
}
OFFSETS = (-7, 15)  # launch/depth_map_fusion.launch


def n_points(w, h):
    return max(0, w - 2 * BORDER) * max(0, h - 2 * BORDER)


def fusion_dims(w, h):
    """(n, fused_w, fused_h) of the reference geometry at the launch offsets (SURVEY.md A.6)."""
    import oracle
    _, r1 = oracle.crop_to_square(w, h, OFFSETS[0], OFFSETS[1], OFFSETS[1])
    _, rc = oracle.crop_to_square(w, h, 0, 0, OFFSETS[1])
    return r1[2], rc[2] - 40, rc[2] - 40


def unit_pixels(cfg):
    """Input pixels of one unit of work (a frame; for config 5 the four maps of a frame set)."""
    return cfg["w"] * cfg["h"] * (4 if cfg["entry"] == "fusion" else 1)


def algorithmic_bytes(cfg, dims=None):
    """SURVEY.md 8(d), per unit of work."""
    w, h = cfg["w"], cfg["h"]
    if cfg["entry"] == "f32":
        return 20 * n_points(w, h)                                   # 4 B read + 16 B written per kept pixel
    if cfg["entry"] == "mono8":
        return (w - 70) * (h - 70) + 16 * n_points(w, h)
    n, fw, fh = dims
    nc = fw + 40
    return (2 * 2 * n * n) + 6 * n * n + (nc * nc + fw * fh) + ((fw - 70) * (fh - 70) + 16 * n_points(fw, fh))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads (and so its first-touch pinned buffers) to the NUMA node of its GPU: the
    end-to-end path is PCIe / host-DRAM bound, and a rank on the far socket halves it.  Best effort."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(local)
        bus = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def dist_setup():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier_sync(world):
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    from disparity_to_point_cloud_b200 import sharding
    return sharding.max_over_ranks(x, device="cuda") if world > 1 else x


def sum_over_ranks(x, world):
    from disparity_to_point_cloud_b200 import sharding
    return sharding.sum_over_ranks(x, device="cuda") if world > 1 else x


def dump_outputs(out_dir, cloud, **small):
    """Writes device tensors as <out_dir>/<name>.npy in float32, DUMP_BYTES at most in all.  `small` are written
    whole; `cloud` (units, points, 4) keeps as many points as fit in what is left, a seeded sample taken at the same
    indices in every unit, split into cloud.npy (finite components, 0 elsewhere) and cloud_nonfinite.npy (0 finite,
    1 +inf, -1 -inf, 2 NaN)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    for name, t in small.items():
        a = t.float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes + 4096  # 4096 B: more than an .npy header takes
    units, npts, _ = cloud.shape
    keep = min(npts, (left - 2 * 4096) // (units * 32))  # 16 B of values + 16 B of classes per point
    if keep < npts:
        idx = np.sort(np.random.default_rng(0).choice(npts, keep, replace=False))
        cloud = cloud[:, torch.from_numpy(idx).to(cloud.device)]
    c = cloud.cpu().numpy()
    kind = np.zeros(c.shape, dtype=np.float32)
    kind[np.isposinf(c)], kind[np.isneginf(c)], kind[np.isnan(c)] = 1, -1, 2
    np.save(os.path.join(out_dir, "cloud.npy"), np.where(np.isfinite(c), c, np.float32(0)))
    np.save(os.path.join(out_dir, "cloud_nonfinite.npy"), kind)


# ---------------------------------------------------------------------------------------------------------
# CPU arm: one sample rule for cpu_baseline (product arm) and for --impl reference
# ---------------------------------------------------------------------------------------------------------
class CpuSample:
    """A bounded sample of the config's workload for the CPU oracle port: `threads` units (frames / frame sets)
    processed unit-parallel on `threads` threads, PASSES times over; one call of step() is one bench step."""
    PASSES = 4

    def __init__(self, cfg, threads):
        import oracle
        from disparity_to_point_cloud_b200 import synth
        self.cfg, self.threads, self.oracle = cfg, threads, oracle
        self.q = oracle.q_from_intrinsics()
        w, h = cfg["w"], cfg["h"]
        self.units = threads * self.PASSES
        if cfg["entry"] == "fusion":
            from concurrent.futures import ThreadPoolExecutor
            rng = np.random.default_rng(5)
            self.sets = [[synth.s2_scene(h, w, 200 + 4 * i), synth.s2_scene(h, w, 201 + 4 * i),
                          rng.integers(0, 256, (h, w), dtype=np.uint8), rng.integers(0, 256, (h, w), dtype=np.uint8)]
                         for i in range(min(threads, 8))]
            self.pool = ThreadPoolExecutor(threads)
            self.desc = (f"{self.PASSES} passes over {threads} frame sets (4 x {w}x{h} mono8: score preprocessing x2, "
                         f"merge, median 3, DisparityCb), set-parallel on {threads} threads")
            return
        if cfg["entry"] == "f32":
            base = synth.s3_float(h, w, 0)
            self.frames = np.stack([np.roll(base, 97 * i, axis=1) for i in range(threads)])
        else:
            self.frames = np.stack([synth.s2_scene(h, w, i % 8) for i in range(threads)])
        self.cloud = np.zeros((threads, n_points(w, h) * 16), dtype=np.uint8)  # touched: a publisher reuses warm memory
        kind = "f32 (S3)" if cfg["entry"] == "f32" else "mono8 (S2)"
        self.desc = f"{self.PASSES} passes over {threads} frames of {w}x{h} {kind}, frame-parallel on {threads} threads"

    def _one_set(self, s):
        o = self.oracle
        d1, d2, s1, s2 = s
        h, w = d1.shape
        _, r1 = o.crop_to_square(w, h, OFFSETS[0], OFFSETS[1], OFFSETS[1])
        _, r2 = o.crop_to_square(h, w, -OFFSETS[0], -OFFSETS[1], OFFSETS[1])
        p1 = o.score_preprocess(s1, r1, False)                      # MatchingScoreCb1
        p2 = o.score_preprocess(o.rotate_cw(s2), r2, True)          # MatchingScoreCb2
        c1 = np.zeros((h, w), np.uint8)
        c1[r1[1]:r1[1] + r1[2], r1[0]:r1[0] + r1[2]] = p1
        rot = np.zeros((w, h), np.uint8)
        rot[r2[1]:r2[1] + r2[2], r2[0]:r2[0] + r2[2]] = p2
        fused, _ = o.fuse(d1, d2, c1, np.ascontiguousarray(np.rot90(rot, 1)), *OFFSETS)  # DisparityCb1/2 + merge
        return o.disparity_cb_mono8(fused, self.q).size             # DisparityCb on the fused map

    def step(self):
        """-> seconds for self.units units"""
        t0 = time.perf_counter()
        if self.cfg["entry"] == "fusion":
            work = [self.sets[i % len(self.sets)] for i in range(self.units)]
            list(self.pool.map(self._one_set, work))
        else:
            for _ in range(self.PASSES):
                self.oracle.run_frames(self.frames, self.q, self.cfg["entry"] == "mono8", self.threads, self.cloud)
        return time.perf_counter() - t0


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    sample = CpuSample(cfg, threads)
    times = []
    for i in range(args.warmup + args.steps):
        dt = sample.step()
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = sample.units * unit_pixels(cfg) / (ms / 1e3) / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mpixel/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "units_per_step": sample.units,
                   "note": "the reference's arithmetic lives in OpenCV / PCL (not installed here): the timed code is the "
                           "CPU oracle port, pinned bit-exact against cv2 and against the reference's own compiled "
                           "glue (oracle/_ref)"},
        "cpu_baseline": {"value": value, "unit": "Mpixel/s", "cores": threads, "kind": "port",
                         "sample": sample.desc + " per step"},
        "e2e": {"value": value, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------------------------------------
def pcie_ceiling(torch, world, h2d_bytes, d2h_bytes, seconds=0.5, direction="both", n_buf=3):
    """Raw pinned cudaMemcpyAsync traffic of the e2e path's shape -- h2d_bytes in and d2h_bytes out per unit, two
    streams, nothing else -- on every rank at once.  -> (GB/s summed over ranks and directions, units/s)."""
    from disparity_to_point_cloud_b200 import pcie
    return pcie.measure(torch, world, h2d_bytes, d2h_bytes, seconds, barrier_sync, max_over_ranks, sum_over_ranks,
                        n_buf=n_buf, direction=direction)


def run_ours(args):
    import torch

    import disparity_to_point_cloud_b200 as d2pc
    from disparity_to_point_cloud_b200 import sharding, synth

    cfg = CONFIGS[args.config]
    w, h, entry = cfg["w"], cfg["h"], cfg["entry"]
    rank, world, local = dist_setup()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    # units are independent: weak = every rank runs per_step units per step, strong = per_step units are sharded
    # i mod G; no data-path collective either way
    per_step = args.frames if args.frames > 0 else cfg["per_step"]
    per_rank = sharding.frames_per_rank(per_step, world, args.scaling)
    units_per_step = per_rank[rank]
    total_units_per_step = sum(per_rank)
    ring = min(cfg["ring"], max(units_per_step, 1))

    ctx = d2pc.Context(device=local, n_slots=args.slots, offset_x=OFFSETS[0], offset_y=OFFSETS[1])
    stream = torch.cuda.ExternalStream(ctx.compute_stream(), device=torch.device("cuda", local))
    dims = None
    extra_ctx, lane_streams = [], [stream]
    # ---- resident inputs: `ring` distinct units in HBM (seeded per rank so ranks do not share data)
    if entry == "f32":
        npts = n_points(w, h)
        base = torch.from_numpy(synth.s3_float(h, w, 1000 * rank)).cuda()
        d_in = torch.empty((ring, h, w), dtype=torch.float32, device="cuda")
        for i in range(ring):
            d_in[i] = torch.roll(base, shifts=131 * i + 7, dims=1)
        out_stride = npts * 16
        d_out = torch.empty((ring, out_stride), dtype=torch.uint8, device="cuda")

        def launch(n):
            ctx.reproject_f32_device(d_in.data_ptr(), n, w, h, w * 4, w * h * 4, d_out.data_ptr(), out_stride)
    elif entry == "mono8":
        npts = n_points(w, h)
        eight = torch.from_numpy(np.stack([synth.s2_scene(h, w, 1000 * rank + i) for i in range(8)])).cuda()
        d_in = eight.repeat((ring + 7) // 8, 1, 1)[:ring].contiguous()
        out_stride = npts * 16
        d_out = torch.empty((ring, out_stride), dtype=torch.uint8, device="cuda")

        def launch(n):
            ctx.reproject_mono8_device(d_in.data_ptr(), n, w, h, w, w * h, d_out.data_ptr(), out_stride)
    else:
        st, r1, r2, rc, dims = ctx.fuse_geometry(w, h)
        n_sq, fw, fh = dims
        npts = n_points(fw, fh)
        rng = np.random.default_rng(1000 * rank + 5)
        eight = np.stack([np.stack([synth.s2_scene(h, w, 1000 * rank + 2 * i), synth.s2_scene(h, w, 1000 * rank + 2 * i + 1),
                                    rng.integers(0, 256, (h, w), dtype=np.uint8), rng.integers(0, 256, (h, w), dtype=np.uint8)])
                          for i in range(8)])
        d_in = torch.from_numpy(eight).cuda().repeat((ring + 7) // 8, 1, 1, 1)[:ring].contiguous()
        # a frame set is six small kernels, none of which fills the chip, so independent frame-set streams overlap
        # on the GPU: the product's slot pipeline gives every slot its own kernel stream (what e2e runs through);
        # the resident leg does the same with one context (= one stereo stream, its own compute stream and
        # intermediates) per lane, sets dealt round-robin
        lanes = [ctx] + [d2pc.Context(device=local, n_slots=1, offset_x=OFFSETS[0], offset_y=OFFSETS[1])
                         for _ in range(max(args.slots, 1) - 1)]
        extra_ctx = lanes[1:]
        lane_streams = [torch.cuda.ExternalStream(c.compute_stream(), device=torch.device("cuda", local)) for c in lanes]
        d_pre = torch.empty((len(lanes), 2, n_sq, n_sq), dtype=torch.uint8, device="cuda")
        d_fused = torch.empty((len(lanes), fh, fw), dtype=torch.uint8, device="cuda")
        d_comb = torch.empty((len(lanes), n_sq, n_sq), dtype=torch.uint8, device="cuda")
        out_stride = npts * 16
        d_out = torch.empty((ring, out_stride), dtype=torch.uint8, device="cuda")
        fb = w * h

        def launch(n):
            # one node pass per frame set: MatchingScoreCb1/2 -> DisparityCb1/2 + publishFusedDepthMap -> DisparityCb
            for i in range(n):
                k = i % len(lanes)
                c = lanes[k]
                p = d_in.data_ptr() + i * 4 * fb
                c.preprocess_score_device(p + 2 * fb, w, h, w, 1, d_pre[k, 0].data_ptr())
                c.preprocess_score_device(p + 3 * fb, w, h, w, 2, d_pre[k, 1].data_ptr())
                c.fuse_preprocessed_device(p, p + fb, d_pre[k, 0].data_ptr(), d_pre[k, 1].data_ptr(), w, h, w,
                                           d_fused[k].data_ptr(), d_comb[k].data_ptr())
                c.reproject_mono8_device(d_fused[k].data_ptr(), 1, fw, fh, fw, fw * fh,
                                         d_out.data_ptr() + i * out_stride, out_stride)
    torch.cuda.synchronize()

    def kernel_step():
        left = units_per_step
        while left > 0:
            n = min(ring, left)
            launch(n)
            left -= n

    for _ in range(args.warmup):
        kernel_step()
    barrier_sync(world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    count_launches = lambda: ctx.launch_count() + sum(c.launch_count() for c in extra_ctx)  # noqa: E731
    l0 = count_launches()
    ev0.record(stream)
    for s_k in lane_streams[1:]:
        s_k.wait_event(ev0)  # every lane starts behind the start mark ...
    for _ in range(args.steps):
        kernel_step()
    for s_k in lane_streams[1:]:
        stream.wait_stream(s_k)  # ... and the end mark waits for every lane
    ev1.record(stream)
    barrier_sync(world)
    clocks = sampler.stop() if rank == 0 else None
    launches = count_launches() - l0
    ms_total = max_over_ranks(ev0.elapsed_time(ev1), world)
    ms_step = ms_total / args.steps
    value = total_units_per_step * unit_pixels(cfg) / (ms_step / 1e3) / 1e6

    # one cloud checked on the device path so a broken kernel can not post a number
    probe = d_out[min(1, ring - 1), :64].cpu().numpy().view(np.float32)
    assert probe[3] == 1.0 and probe[7] == 1.0, "kernel output is not XYZ1 points"
    if args.dump_outputs and rank == 0:
        # every launch of a step writes ring slot i from ring input i, so the ring holds the last step's results
        cloud = d_out.view(torch.float32).view(ring, npts, 4)
        if entry == "fusion":
            dump_outputs(args.dump_outputs, cloud, cropped_score=d_pre, fused_depth_map=d_fused, combined_score=d_comb)
        else:
            dump_outputs(args.dump_outputs, cloud)

    peak, peak_src = measured_peak()
    alg = algorithmic_bytes(cfg, dims)
    unit_s = (ms_total / 1e3) / (args.steps * units_per_step)
    achieved = alg / unit_s / 1e9
    api_calls = args.steps * ((units_per_step + ring - 1) // ring)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "kernel": cfg["kernel"],
                "bytes_per_launch": alg * ring, "launch_us": unit_s * ring * 1e6,
                "note": "per device-entry call of %d unit(s); achieved = algorithmic bytes / CUDA-event time" % ring}
    if entry == "fusion":
        roofline["note"] = ("six kernels per frame set, sets dealt round-robin over %d contexts (one compute stream each, "
                            "as the slot pipeline's per-slot kernel streams); achieved = algorithmic bytes / CUDA-event "
                            "time from the start mark to the last lane's end" % len(lane_streams))

    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            t = json.load(open(tr))
            roofline["traffic"] = t.get("by_config", {}).get(str(args.config)) or (
                t.get("dram_bytes_per_launch_ring16") if args.config == 4 else None)
        except Exception:
            pass

    # ---- end to end: pinned host frames -> H2D -> kernels -> D2H, through the C ABI's streaming entry
    e2e_units = args.e2e_frames if args.e2e_frames > 0 else max(units_per_step, 256 if entry != "fusion" else 128)
    e2e_total = sum_over_ranks(e2e_units, world)
    host_ring = 8
    if entry == "fusion":
        pin = d2pc.PinnedArray((host_ring, 4, h, w), np.uint8)
        pin.array[:] = eight
        in_bytes = 4 * w * h
    elif entry == "mono8":
        pin = d2pc.PinnedArray((host_ring, h, w), np.uint8)
        for i in range(host_ring):
            pin.array[i] = synth.s2_scene(h, w, 1000 * rank + 100 + i)
        in_bytes = w * h
    else:
        pin = d2pc.PinnedArray((host_ring, h, w), np.float32)
        hb = synth.s3_float(h, w, 1000 * rank + 1)
        for i in range(host_ring):
            pin.array[i] = np.roll(hb, 61 * i, axis=1)
        in_bytes = 4 * w * h
    out_bytes = npts * 16
    checks = {}

    def sink(idx, cloud):
        if idx == 1:
            checks["width"] = cloud.width

    def e2e_step(n, check=False):
        # the timed call hands every cloud to a NULL sink inside the C ABI (no Python per frame);
        # the warm-up call looks at one cloud so a broken pipeline can not post a number
        if entry == "fusion":
            ctx.process_fusion_stream(pin.array, collect=False, sink=sink if check else None, n_sets=n)
        else:
            ctx.process_stream(pin.array, collect=False, sink=sink if check else None, n_frames=n)

    e2e_step(host_ring, check=True)  # warm-up: allocates the slot buffers
    barrier_sync(world)
    t0 = time.perf_counter()
    if args.stagger_us:
        time.sleep(rank * args.stagger_us * 1e-6)  # experiment: ranks out of phase (the delay is inside the timed span)
    e2e_step(e2e_units)
    barrier_sync(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    e2e_value = e2e_total * unit_pixels(cfg) / e2e_s / 1e6
    assert checks.get("width") == npts
    e2e = {"value": e2e_value, "unit": "Mpixel/s", "h2d_bytes_per_step": units_per_step * in_bytes,
           "d2h_bytes_per_step": units_per_step * out_bytes, "frames_timed": int(e2e_total),
           "frames_per_s": e2e_total / e2e_s, "gbs": e2e_total * (in_bytes + out_bytes) / e2e_s / 1e9,
           "timer": "wall clock between device syncs, max over ranks; frames_timed and gbs are all-rank totals",
           "slots": args.slots, "pinned": "thp" if os.environ.get("D2PC_PINNED_THP", "0") not in ("", "0") else "cudaHostAlloc",
           "stagger_us": args.stagger_us}
    pin.free()
    if not args.no_ceiling:
        ceil_gbs, ceil_units = pcie_ceiling(torch, world, in_bytes, out_bytes, n_buf=max(args.slots, 3))
        e2e["ceiling_gbs"] = ceil_gbs
        e2e["frac_of_ceiling"] = e2e["gbs"] / ceil_gbs if ceil_gbs else None
        e2e["ceiling_note"] = ("plain pinned cudaMemcpyAsync, %d B in + %d B out per unit on two free-running streams, "
                               "all %d rank(s) at once, no kernels" % (in_bytes, out_bytes, world))
        # the bound no schedule can beat: each direction alone (two free-running streams contend more than the
        # pipeline's partially overlapped copies do, so a unit with comparable traffic each way can exceed `ceiling`)
        _, u_in = pcie_ceiling(torch, world, in_bytes, out_bytes, 0.3, "h2d", max(args.slots, 3))
        _, u_out = pcie_ceiling(torch, world, in_bytes, out_bytes, 0.3, "d2h", max(args.slots, 3))
        # (a direction demonstrably sustains at least what it carried in the two-direction run: on some hosts of the
        # pool the short one-direction runs come out below that, so the bound is never taken lower than it)
        bound = max(min(u_in, u_out), ceil_units)
        e2e["one_way_bound_units_per_s"] = bound
        e2e["one_way_bound_direction"] = "h2d" if u_in < u_out else "d2h"
        e2e["frac_of_one_way_bound"] = e2e["frames_per_s"] / bound if bound else None

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        sample = CpuSample(cfg, threads)
        sample.step()
        dts = [sample.step() for _ in range(3)]
        dt = sum(dts) / len(dts)
        cpu_baseline = {"value": sample.units * unit_pixels(cfg) / dt / 1e6, "unit": "Mpixel/s", "cores": threads,
                        "kind": "port", "sample": sample.desc + f"; mean of 3 timed steps of {dt:.2f} s after 1 warm-up"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64" if entry != "fusion" else "u8+f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "config": args.config,
                       "units_per_step_per_gpu": units_per_step, "resident_ring_units": ring,
                       "l2_policy": "the ring of resident inputs+outputs is %.0f MB (> 126 MB L2), no flush needed"
                                    % (ring * (in_bytes + out_bytes) / 1e6),
                       "arith": "EXACT (bit-identical to cv::reprojectImageTo3D)", "filter": "CROP (reference)",
                       "units_per_s": total_units_per_step / (ms_step / 1e3),
                       "sharding": "unit i -> rank i mod G, no collective on the data path"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches),
            "api_calls_timed": api_calls, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
        if args.append:
            with open(args.append, "a") as f:
                f.write(json.dumps(line) + "\n")
    for c in extra_ctx:
        c.close()
    ctx.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS), help="BASELINE workload (SURVEY 8 numbering)")
    ap.add_argument("--frames", type=int, default=0, help="units per GPU per step (0 = the config's own)")
    ap.add_argument("--e2e-frames", type=int, default=0, help="units timed end to end (0 = one full step, >= 256)")
    ap.add_argument("--slots", type=int, default=4, help="pipeline slots per GPU of the end-to-end path")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: per-step units per GPU; strong: per-step units in total, sharded i mod G")
    ap.add_argument("--stagger-us", type=int, default=0, help="experiment: rank r starts its end-to-end stream r x this late")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-ceiling", action="store_true", help="skip the raw-copy ceiling of the e2e path")
    ap.add_argument("--append", default="", help="also append the JSON line to this file (profiles/configs_r2.json)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (float32, 64 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the product path's outputs (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it
    main()
