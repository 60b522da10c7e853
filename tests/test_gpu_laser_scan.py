"""GPU: the laser scan output (pointcloud_to_laserscan on the device) byte for byte against the CPU recipe
tests/scan_ref, composed with the cloud references of the other stages (tests/transform_ref, box_ref, voxel_ref,
outlier_ref): the ranges and every message field, through every host entry, the device entry, the node mirror and the
wire format, with canaries around the outputs.  D2PC_SCAN_FUZZ_CASES / D2PC_SCAN_FUZZ_SEED set the fuzz (default 60)."""
import math
import os
import struct
import subprocess

import numpy as np
import pytest

import oracle
import scan_ref
import transform_ref
from disparity_to_point_cloud_b200 import synth
from test_gpu_crop_box import box_for, set_mode, transform_of
from test_gpu_transform import ROR, reset, u8, want
from test_gpu_voxel import ENTRIES, check, crop_of, run_entry

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_SCAN_FUZZ_CASES", "60"))
SEED0 = int(os.environ.get("D2PC_SCAN_FUZZ_SEED", "91000"))
INVALID_ARG, NOT_READY, BAD_DIMS = -1, -8, -3
MODES = ["crop", "finite", "voxel"]
# camera optical frame -> a z-up body frame whose origin is 1 m under the camera
ZUP = np.float32([[0, 0, 1, 0], [-1, 0, 0, 0], [0, -1, 0, 1.0]])
GRID_ZUP = (0.05, 0, ("z", -10.0, 10.0))
NARROW = dict(angle_min=-0.8, angle_max=0.8, angle_increment=0.8 / 1800, min_height=0.2, max_height=1.8,
              range_min=0.3, range_max=15.0, use_inf=0, inf_epsilon=0.25)


@pytest.fixture(scope="module")
def env():
    import disparity_to_point_cloud_b200 as d2pc
    ctx = d2pc.Context(n_slots=3)
    cap = 3840 * 2160 * 16 + 256
    pin = d2pc.PinnedArray((cap,), np.uint8)
    reg = d2pc.RegisteredArray(np.empty(cap, np.uint8))
    yield d2pc, ctx, pin, reg
    pin.free()
    reg.free()
    ctx.close()


def off(d2pc, ctx):
    reset(d2pc, ctx)
    ctx.set_laser_scan(False)
    ctx.set_tuning("direct_out", 0)


def check_scan(ctx, cloud_bytes, what, **p):
    fields, ranges = ctx.last_scan()
    want_r = scan_ref.scan(u8(cloud_bytes), **p)
    assert ranges.tobytes() == want_r.tobytes(), (what, np.nonzero(ranges.view(np.uint32) != want_r.view(np.uint32)))
    wf = scan_ref.fields(**p)
    for k, v in wf.items():
        assert np.float32(fields[k]).tobytes() == np.float32(v).tobytes(), (what, k, fields[k], v)
    return ranges


@pytest.mark.parametrize("ror", [False, True])
@pytest.mark.parametrize("box", [False, True])
@pytest.mark.parametrize("mode", MODES)
def test_every_host_entry_matches_the_reference(env, mode, box, ror):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    try:
        for frame in (synth.s2_scene(480, 752, 3), synth.s3_float(480, 752, 4)):
            crop = crop_of(frame, q)
            bx = box_for(u8(transform_ref.transform(crop, ZUP)), 0.6, None) if box else None
            wv = want(crop, mode, ZUP, bx, ROR if ror else None, GRID_ZUP)
            set_mode(d2pc, ctx, mode, GRID_ZUP)
            ctx.set_radius_outlier(*(ROR if ror else (0.0,)))
            ctx.set_crop_box(*(bx or (None,)))
            ctx.set_transform(ZUP)
            for p in ({}, NARROW):
                ctx.set_laser_scan(**p)
                for entry in ENTRIES:
                    got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                    check(got, wv, (entry, frame.dtype, mode, box, ror), cl)
                    check_scan(ctx, wv[0], (entry, frame.dtype, mode, box, ror, bool(p)), **p)
    finally:
        off(d2pc, ctx)


def test_scan_off_is_not_ready_and_launches(env):
    d2pc, ctx, _, _ = env
    frame = synth.s2_scene(480, 752, 9)
    try:
        ctx.process_mono8(frame)
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.last_scan()
        assert e.value.status == NOT_READY
        ctx.set_transform(ZUP)
        n0 = ctx.launch_count()
        ctx.process_mono8(frame)
        base = ctx.launch_count() - n0
        ctx.set_laser_scan()
        n0 = ctx.launch_count()
        ctx.process_mono8(frame)
        assert ctx.launch_count() - n0 == base + 2  # the fill and the binning
        ctx.set_laser_scan(False)
        ctx.process_mono8(frame)
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.last_scan()
        assert e.value.status == NOT_READY
    finally:
        off(d2pc, ctx)


@pytest.mark.parametrize("mode", ["crop", "finite"])
def test_stream_fusion_and_4k(env, mode):
    d2pc, ctx, pin, _ = env
    q = ctx.get_q()
    try:
        set_mode(d2pc, ctx, mode, GRID_ZUP)
        ctx.set_transform(ZUP)
        ctx.set_laser_scan(**NARROW)
        # the stream: last_scan inside the sink is the scan of the cloud handed to it
        frames = np.stack([synth.s2_scene(480, 752, 20 + i) for i in range(5)])
        seen = []
        ctx.process_stream(frames, collect=False, sink=lambda i, cl: seen.append(
            (i, np.ctypeslib.as_array(cl.data, shape=(cl.row_step,)).tobytes() if cl.row_step else b"",
             ctx.last_scan()[1])), n_frames=8)
        for i, data, ranges in seen:
            wv = want(crop_of(frames[i % 5], q), mode, ZUP)
            assert data == wv[0]
            assert ranges.tobytes() == scan_ref.scan(u8(wv[0]), **NARROW).tobytes(), i
        # 4K frames, mono8 and f32
        for frame in (synth.s2_scene(2160, 3840, 5), synth.s3_float(2160, 3840, 6)):
            wv = want(crop_of(frame, q), mode, ZUP)
            got, cl = run_entry(d2pc, ctx, pin, None, frame, "library")
            check(got, wv, ("4k", frame.dtype), cl)
            check_scan(ctx, wv[0], "4k", **NARROW)
        # fusion: fuse_then_process, submit_fusion + wait, the fusion stream, on the library's own CROP cloud of the
        # fused map
        four = [synth.s2_scene(480, 752, 30 + i) for i in range(4)]
        off(d2pc, ctx)
        base = ctx.fuse_then_process(*four)
        set_mode(d2pc, ctx, mode, GRID_ZUP)
        ctx.set_transform(ZUP)
        ctx.set_laser_scan(**NARROW)
        wv = want(base, mode, ZUP)
        check(ctx.fuse_then_process(*four), wv, "fuse_then_process", ctx.last_cloud)
        check_scan(ctx, wv[0], "fuse_then_process", **NARROW)
        ctx.submit_fusion(0, *four, preprocess_scores=False)
        check(ctx.wait(0), wv, "submit_fusion", ctx.last_cloud)
        check_scan(ctx, wv[0], "submit_fusion", **NARROW)
        sets = np.stack([np.stack(four)] * 2)
        got = []
        ctx.process_fusion_stream(sets, preprocess_scores=False, collect=False,
                                  sink=lambda i, cl: got.append(ctx.last_scan()[1]), n_sets=3)
        assert len(got) == 3 and all(g.tobytes() == scan_ref.scan(u8(wv[0]), **NARROW).tobytes() for g in got)
    finally:
        off(d2pc, ctx)


def test_voxel_fallback_and_keep_cloud_0(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 11)
    crop = crop_of(frame, q)
    try:
        # VOXEL's overflow fallback (a tiny leaf) publishes the CROP cloud; the scan is of that cloud
        grid = (1e-6, 0, None)
        wv = want(crop, "voxel", ZUP, None, None, grid)
        assert wv[1] == 0
        set_mode(d2pc, ctx, "voxel", grid)
        ctx.set_transform(ZUP)
        ctx.set_laser_scan()
        check(ctx.process_mono8(frame), wv, "voxel fallback", ctx.last_cloud)
        check_scan(ctx, wv[0], "voxel fallback")
        # keep_cloud 0: width 0, data NULL, no write into dst and no cap check, the ranges only leave the device
        for mode in MODES:
            set_mode(d2pc, ctx, mode, GRID_ZUP)
            wv = want(crop, mode, ZUP, None, None, GRID_ZUP)
            ctx.set_laser_scan(keep_cloud=0)
            for entry in ENTRIES:
                # every entry that takes a destination gets a 64-byte canary as its whole dst: a cap far below the
                # cloud, and bytes that must stay as they are
                dst = {"pinned": pin.array[:64], "registered": reg.array[:64], "pageable": np.empty(64, np.uint8),
                       "slot_into": pin.array[:64]}.get(entry)
                if dst is None:
                    got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry)
                else:
                    dst[:] = 0xA5
                    if entry == "slot_into":
                        ctx.submit(2, frame, dst)
                        got, cl = ctx.wait(2), ctx.last_cloud
                    else:
                        got, cl = ctx.process_into(frame, dst), ctx.last_cloud
                    assert np.all(dst == 0xA5), (mode, entry)
                assert got.size == 0 and cl.width == 0 and cl.row_step == 0 and not cl.data, (mode, entry)
                check_scan(ctx, wv[0], ("keep 0", mode, entry))
        # the slot spans: no payload in d2h_us with keep_cloud 0
        set_mode(d2pc, ctx, "crop")
        big = synth.s2_scene(2160, 3840, 12)
        ctx.set_timing(True)
        d2h = {}
        for keep in (1, 0):
            ctx.set_laser_scan(keep_cloud=keep)
            for _ in range(3):
                ctx.submit(0, big)
                ctx.wait(0)
            t = ctx.slot_timing(0)
            d2h[keep] = t.d2h_us
            assert t.points == (0 if keep == 0 else crop_of(big, q).nbytes // 16)
        assert d2h[0] < 0.1 * d2h[1], d2h
    finally:
        ctx.set_timing(False)
        off(d2pc, ctx)


def test_slots_submitted_under_different_settings(env):
    d2pc, ctx, _, _ = env
    q = ctx.get_q()
    frames = [synth.s2_scene(480, 752, 40 + i) for i in range(3)]
    try:
        ctx.set_transform(ZUP)
        ctx.set_laser_scan()
        ctx.submit(0, frames[0])
        ctx.set_laser_scan(**NARROW)
        ctx.submit(1, frames[1])
        ctx.set_laser_scan(False)
        ctx.submit(2, frames[2])
        ctx.set_laser_scan(angle_increment=0.5)
        ctx.wait(0)
        check_scan(ctx, want(crop_of(frames[0], q), "crop", ZUP)[0], "slot 0")
        ctx.wait(1)
        check_scan(ctx, want(crop_of(frames[1], q), "crop", ZUP)[0], "slot 1", **NARROW)
        ctx.wait(2)
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.last_scan()
        assert e.value.status == NOT_READY
        # a counted cloud that does not fit the caller's buffer: d2pc_wait returns no cloud, and no scan either
        ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
        ctx.set_laser_scan()
        ctx.process_mono8(frames[0])
        ctx.last_scan()
        ctx.submit(1, frames[1], np.empty(64, np.uint8))
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.wait(1)
        assert e.value.status == -9
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.last_scan()
        assert e.value.status == NOT_READY
    finally:
        off(d2pc, ctx)


def device_scan(ctx, pts, n_frames, n_max, counts=None, canary=True, stride_pad=0):
    """d2pc_laser_scan_device on a (n_frames, n_max, 4) float32 cloud array; returns (ranges per frame, n)."""
    import torch
    import disparity_to_point_cloud_b200 as d2pc
    p = ctx.get_laser_scan()
    n = d2pc.laser_scan_ranges(**{k: getattr(p, k) for k in scan_ref.DEFAULTS})
    stride = n * 4 + stride_pad
    d_in = torch.from_numpy(np.ascontiguousarray(pts).reshape(-1)).cuda()
    d_out = torch.full((n_frames * stride // 4 + 64,), np.float32(-7.0).item(), dtype=torch.float32, device="cuda")
    d_cnt = torch.from_numpy(counts.view(np.int32)).cuda() if counts is not None else None
    ctx.laser_scan_device(d_in.data_ptr(), n_frames, n_max, n_max * 16, d_cnt.data_ptr() if d_cnt is not None else 0,
                          d_out.data_ptr(), stride)
    ctx.sync()
    raw = d_out.cpu().numpy()
    out = np.stack([raw[f * stride // 4: f * stride // 4 + n] for f in range(n_frames)]) if n_frames else raw[:0]
    if canary:  # nothing beyond each frame's n ranges is written
        pad = [raw[f * stride // 4 + n: (f + 1) * stride // 4] for f in range(n_frames)] + [raw[n_frames * stride // 4:]]
        assert all(np.all(x == np.float32(-7.0)) for x in pad)
    return out, n


def params_of(ctx):
    p = ctx.get_laser_scan()
    return {k: getattr(p, k) for k in scan_ref.DEFAULTS}


@pytest.mark.parametrize("bins", [360, 4096, 4097, 2 ** 20])
def test_device_entry_bins_on_both_sides_of_the_shared_limit(env, bins):
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(bins)
    nf, n_max = 6, 50000
    pts = rng.normal(0, 4, (nf, n_max, 4)).astype(np.float32)
    pts[..., 2] = rng.uniform(-0.5, 2, (nf, n_max))
    pts[rng.random((nf, n_max)) < 0.01, 0] = np.nan
    counts = rng.integers(0, n_max + 100, nf).astype(np.uint32)
    try:
        ctx.set_laser_scan(angle_increment=float(np.float32(2 * math.pi) / np.float32(bins)) * 1.0000001,
                           range_max=30.0)
        p = params_of(ctx)
        for cnt in (None, counts):
            got, n = device_scan(ctx, pts, nf, n_max, cnt, stride_pad=8)
            assert abs(n - bins) <= 1
            for f in range(nf):
                k = n_max if cnt is None else min(int(cnt[f]), n_max)
                assert got[f].tobytes() == scan_ref.scan(pts[f, :k], **p).tobytes(), (bins, f, cnt is None)
    finally:
        off(d2pc, ctx)


def test_device_entry_70000_tiny_frames_in_chunks(env):
    """70 000 frames of n_max 32768 positions (2.3e9 > 2^31 - 2: the batch runs in two chunks), 5 points each."""
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(93)
    nf, n_max, k = 70000, 32768, 5
    small = rng.normal(0, 3, (nf, k, 4)).astype(np.float32)
    small[..., 2] = rng.uniform(0.01, 2, (nf, k))
    counts = rng.integers(0, k + 1, nf).astype(np.uint32)
    try:
        ctx.set_laser_scan(angle_increment=math.pi / 8)
        p = params_of(ctx)
        n = d2pc.laser_scan_ranges(**p)
        d_in = torch.zeros((nf, n_max * 4), dtype=torch.float32, device="cuda")
        d_in[:, : k * 4] = torch.from_numpy(small.reshape(nf, k * 4)).cuda()
        d_cnt = torch.from_numpy(counts.view(np.int32)).cuda()
        d_out = torch.full((nf * n,), -7.0, dtype=torch.float32, device="cuda")
        n0 = ctx.launch_count()
        ctx.laser_scan_device(d_in.data_ptr(), nf, n_max, n_max * 16, d_cnt.data_ptr(), d_out.data_ptr(), n * 4)
        ctx.sync()
        assert ctx.launch_count() - n0 == 4  # two chunks of fill + binning
        del d_in
        got = d_out.cpu().numpy().reshape(nf, n)
        for f in range(nf):
            assert got[f].tobytes() == scan_ref.scan(small[f, : counts[f]], **p).tobytes(), f
    finally:
        off(d2pc, ctx)


def test_points_straddling_bin_edges(env):
    """For bin edges across the span, the two float points next to the edge (one float step of y apart, one on each
    side by the library's angle, found on the host): one point per frame, so each frame's ranges show which bin the
    device picked.  The host's and the device's angle must agree to the last bit for these to match."""
    d2pc, ctx, _, _ = env
    try:
        ctx.set_laser_scan(angle_min=-1.3, angle_max=1.3, angle_increment=0.01)
        p = params_of(ctx)
        amin, inc = float(np.float32(-1.3)), float(np.float32(0.01))
        sel, gaps = [], []
        for kk in range(1, 260, 3):
            th = amin + kk * inc
            for radius in (0.7, 2.5, 9.0):
                x0, y0 = np.float32(radius * math.cos(th)), np.float32(radius * math.sin(th))
                ys = [y0]
                for _ in range(12):
                    ys.insert(0, np.nextafter(ys[0], np.float32(-np.inf)))
                    ys.append(np.nextafter(ys[-1], np.float32(np.inf)))
                ys = np.float32(ys)
                _, a = scan_ref.math_arrays(np.full(len(ys), x0, np.float32), ys)
                k = np.floor((a - amin) / inc)
                step = np.nonzero(np.diff(k))[0]
                for j in step:
                    sel += [(x0, ys[j]), (x0, ys[j + 1])]
                    edge = amin + k[j + 1] * inc
                    gaps.append(min(abs(a[j] - edge), abs(a[j + 1] - edge)) / math.ulp(edge))
        assert len(sel) >= 100, len(sel)
        pts = np.zeros((len(sel), 1, 4), np.float32)
        pts[:, 0, :2] = np.float32(sel)
        pts[:, 0, 2] = 0.5
        got, n = device_scan(ctx, pts, len(sel), 1)
        for f in range(len(sel)):
            assert got[f].tobytes() == scan_ref.scan(pts[f], **p).tobytes(), (f, sel[f])
        print(f"{len(sel)} points next to {len(gaps)} bin edges, nearest {min(gaps):.0f} ulp of the edge angle: "
              "device and host agree")
    finally:
        off(d2pc, ctx)


def test_wall_scene(env):
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(95)
    nf, n = 8, 268800
    pts = np.empty((nf, n, 4), np.float32)
    pts[..., 0] = 2.0 + rng.normal(0, 0.01, (nf, n))
    pts[..., 1] = rng.uniform(-0.3, 0.3, (nf, n))
    pts[..., 2] = rng.uniform(0.05, 1.5, (nf, n))
    pts[..., 3] = 1.0
    try:
        for kw in ({}, dict(angle_increment=math.pi / 1800), dict(angle_increment=2 * math.pi / 2 ** 19)):
            ctx.set_laser_scan(**kw)
            p = params_of(ctx)
            got, _ = device_scan(ctx, pts, nf, n)
            for f in range(nf):
                assert got[f].tobytes() == scan_ref.scan(pts[f], **p).tobytes(), (kw, f)
    finally:
        off(d2pc, ctx)


def test_settings_refused_and_kept_and_device_arguments(env):
    import torch
    d2pc, ctx, _, _ = env
    try:
        ctx.set_laser_scan(**NARROW)
        before = bytes(ctx.get_laser_scan())
        for kw in (dict(angle_increment=0.0), dict(range_min=-1.0), dict(angle_min=math.nan), dict(min_height=math.nan),
                   dict(inf_epsilon=-1.0), dict(angle_min=2.0, angle_max=1.0), dict(angle_increment=1e-9)):
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.set_laser_scan(**kw)
            assert e.value.status == INVALID_ARG, kw
            assert bytes(ctx.get_laser_scan()) == before
        d = torch.zeros(4096, dtype=torch.float32, device="cuda")
        lib, h = d2pc.lib(), ctx._h
        base = d.data_ptr()
        assert lib.d2pc_laser_scan_device(h, base + 4, 1, 10, 160, None, base + 8192, 8192) == BAD_DIMS
        assert lib.d2pc_laser_scan_device(h, base, 2, 10, 80, None, base + 8192, 8192) == BAD_DIMS
        assert lib.d2pc_laser_scan_device(h, base, 1, 10, 160, None, base + 8194, 8192) == BAD_DIMS
        assert lib.d2pc_laser_scan_device(h, base, 1, 10, 160, None, base + 80, 8192) == INVALID_ARG  # overlap
        assert lib.d2pc_laser_scan_device(h, base, 0, 10, 160, None, base + 8192, 8192) == 0
        ctx.set_laser_scan(False)
        assert lib.d2pc_laser_scan_device(h, base, 1, 10, 160, None, base + 8192, 8192) == INVALID_ARG
    finally:
        off(d2pc, ctx)


def test_wire_bytes(env):
    d2pc, ctx, _, _ = env
    try:
        ctx.set_transform(ZUP)
        ctx.set_laser_scan(**NARROW)
        ctx.process_mono8(synth.s2_scene(480, 752, 50))
        s = ctx.last_scan_raw()
        wire = ctx.serialize_laserscan(s, seq=7, sec=11, nsec=13)
        fid = ctx.cfg.frame_id
        ranges = np.ctypeslib.as_array(s.ranges, shape=(s.n_ranges,))
        want_b = (struct.pack("<III", 7, 11, 13) + struct.pack("<I", len(fid)) + fid +
                  struct.pack("<7f", *(getattr(s, k) for k in s.FIELDS)) + struct.pack("<I", s.n_ranges) +
                  ranges.astype("<f4").tobytes() + struct.pack("<I", 0))
        assert wire == want_b
    finally:
        off(d2pc, ctx)


def test_node1_publishes_scan(tmp_path):
    """The node mirror with transform_* and scan_* params: /scan carries the scan of the cloud it publishes, with the
    cloud's header and frame_id (transform_target_frame); with scan_keep_cloud 0 /point_cloud is not published."""
    from disparity_to_point_cloud_b200 import build
    harness = build.build_harness()
    img = synth.s2_scene(480, 752, 60)
    raw = tmp_path / "in.raw"
    raw.write_bytes(np.ascontiguousarray(img).tobytes())
    crop = oracle.disparity_cb_mono8(img, oracle.q_from_intrinsics())
    pose = dict(tx=0.0, ty=0.0, tz=1.0, roll=-1.5707963, pitch=0.0, yaw=-1.5707963)  # optical -> z-up, 1 m up
    t = transform_of((pose["roll"], pose["pitch"], pose["yaw"]), (pose["tx"], pose["ty"], pose["tz"]))
    cloud_want = want(crop, "crop", t)
    p = dict(angle_min=-0.6, angle_max=0.6, angle_increment=0.002, range_max=20.0, min_height=0.1, max_height=1.9,
             use_inf=0, inf_epsilon=0.5)
    for keep in (1, 0):
        params = dict(transform_enable=1, transform_target_frame="/body", scan_enable=1, scan_keep_cloud=keep,
                      **{f"transform_{k}": v for k, v in pose.items()}, **{f"scan_{k}": v for k, v in p.items()})
        launch = tmp_path / f"n{keep}.launch"
        launch.write_text('<launch>\n  <node name="n" pkg="p" type="t">\n' +
                          "".join(f'    <param name="{k}" value="{v}"/>\n' for k, v in params.items()) +
                          "  </node>\n</launch>\n")
        cloud_bin, scan_bin = tmp_path / f"c{keep}.bin", tmp_path / f"s{keep}.bin"
        subprocess.run([harness, "node1scan", str(launch), "752", "480", str(raw), str(cloud_bin), str(scan_bin)],
                       check=True)
        ranges = scan_ref.scan(u8(cloud_want[0]), **p)
        assert np.count_nonzero(ranges != np.float32(20.5)) > 50
        f = scan_ref.fields(**p)
        fid = b"/body"
        want_b = (struct.pack("<III", 0, 3, 4) + struct.pack("<I", len(fid)) + fid +
                  struct.pack("<7f", f["angle_min"], f["angle_max"], f["angle_increment"], 0.0, f["scan_time"],
                              f["range_min"], f["range_max"]) + struct.pack("<I", len(ranges)) +
                  ranges.astype("<f4").tobytes() + struct.pack("<I", 0))
        assert scan_bin.read_bytes() == want_b, keep
        if keep:
            assert cloud_bin.read_bytes() == oracle.serialize_pointcloud2(u8(cloud_want[0]), seq=0, sec=3, nsec=4,
                                                                          frame_id="/body", is_dense=cloud_want[1])
        else:
            assert cloud_bin.read_bytes() == b""


def _fuzz_case(case, env):
    d2pc, ctx, pin, reg = env
    rng = np.random.default_rng(SEED0 + case)
    q = ctx.get_q()
    h, w = [(480, 640), (480, 752), (720, 1280), (200, 300)][rng.integers(0, 4)]
    frame = synth.s2_scene(h, w, int(rng.integers(0, 1000))) if rng.random() < 0.6 else synth.s3_float(h, w, int(rng.integers(0, 1000)))
    mode = MODES[rng.integers(0, 3)]
    box = rng.random() < 0.3
    ror = rng.random() < 0.2
    crop = crop_of(frame, q)
    bx = box_for(u8(transform_ref.transform(crop, ZUP)), float(rng.uniform(0.3, 0.9)), None) if box else None
    wv = want(crop, mode, ZUP, bx, ROR if ror else None, GRID_ZUP)
    amin = float(rng.uniform(-math.pi, 0.5))
    amax = float(amin + rng.uniform(0.1, math.pi - amin))
    kw = dict(angle_min=amin, angle_max=amax, angle_increment=(amax - amin) / float(rng.choice([1, 7, 360, 3600, 5000])),
              min_height=float(rng.uniform(-2, 0.5)), max_height=float(rng.uniform(0.5, 3)),
              range_min=float(rng.uniform(0, 1)), range_max=float(rng.uniform(2, 30)), use_inf=int(rng.integers(0, 2)),
              inf_epsilon=float(rng.uniform(0, 2)), scan_time=float(rng.uniform(0.01, 0.2)))
    keep = int(rng.random() < 0.8)
    set_mode(d2pc, ctx, mode, GRID_ZUP)
    ctx.set_radius_outlier(*(ROR if ror else (0.0,)))
    ctx.set_crop_box(*(bx or (None,)))
    ctx.set_transform(ZUP)
    ctx.set_laser_scan(keep_cloud=keep, **kw)
    entry = ENTRIES[rng.integers(0, len(ENTRIES))]
    got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
    if keep:
        check(got, wv, (case, entry), cl)
    else:
        assert cl.width == 0
    check_scan(ctx, wv[0], (case, entry, mode, box, ror, kw), **kw)


def test_scan_fuzz_against_reference(env):
    d2pc, ctx, _, _ = env
    try:
        for case in range(N_FUZZ):
            _fuzz_case(case, env)
    finally:
        off(d2pc, ctx)
