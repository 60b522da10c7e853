"""GPU: the occupancy map (octomap_server's insertScan on the device) byte for byte against the literal restatement of
octomap (tests/map_ref/octomap_literal.cpp), fed the cloud the composed references of the other stages publish
(tests/transform_ref, box_ref, voxel_ref, outlier_ref): every known voxel's key and log-odds bits, and the centres
cloud, after sequences of frames under per-frame poses, through every host entry, the device entry and the fusion
entries, with canaries around the outputs.  D2PC_MAP_FUZZ_CASES / D2PC_MAP_FUZZ_SEED set the fuzz (default 40)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import map_ref
import transform_ref
from disparity_to_point_cloud_b200 import synth
from test_gpu_crop_box import box_for, set_mode
from test_gpu_transform import ROR, reset, u8, want
from test_gpu_voxel import ENTRIES, check, crop_of, run_entry

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_MAP_FUZZ_CASES", "40"))
SEED0 = int(os.environ.get("D2PC_MAP_FUZZ_SEED", "93000"))
INVALID_ARG, BUFFER_TOO_SMALL = -1, -9
GRID = (0.1, 0, None)
MAP = dict(resolution=0.1, max_range=12.0)


def pose(tx, ty, tz):
    """camera optical frame -> a z-up world frame, the camera at (tx, ty, tz)"""
    return np.float32([[0, 0, 1, tx], [-1, 0, 0, ty], [0, -1, 0, tz]])


POSES = [pose(0.0, 0.0, 1.0), pose(0.7, -0.3, 1.2)]


@pytest.fixture(scope="module")
def env():
    import disparity_to_point_cloud_b200 as d2pc
    ctx = d2pc.Context(n_slots=3)
    cap = 1280 * 720 * 16 + 256
    pin = d2pc.PinnedArray((cap,), np.uint8)
    reg = d2pc.RegisteredArray(np.empty(cap, np.uint8))
    yield d2pc, ctx, pin, reg
    pin.free()
    reg.free()
    ctx.close()


def off(d2pc, ctx):
    reset(d2pc, ctx)
    ctx.set_laser_scan(False)
    ctx.set_occupancy(False)
    ctx.occupancy_reset()


def same_map(ctx, ref, what):
    k, lo = ctx.occupancy_voxels()
    wk, wlo = ref.voxels()
    assert len(k) == len(wk), (what, len(k), len(wk))
    assert k.tobytes() == wk.tobytes(), (what, "keys")
    assert lo.tobytes() == wlo.tobytes(), (what, "log-odds", np.nonzero(lo.view(np.uint32) != wlo.view(np.uint32)))
    c = ctx.occupancy_centers()
    assert c.tobytes() == ref.centers().tobytes(), (what, "centres")
    assert len(k) > 0 or what == "empty"
    return len(k)


def origin_of(m):
    return (m[0][3], m[1][3], m[2][3])


@pytest.mark.parametrize("mode,box,ror", [("crop", False, False), ("finite", False, False), ("voxel", False, False),
                                          ("crop", True, True), ("finite", True, False), ("voxel", False, True)])
def test_every_host_entry_matches_the_literal_octree(env, mode, box, ror):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = [synth.s2_scene(480, 752, 3), synth.s3_float(480, 752, 4)]
    try:
        ref = map_ref.Octree(**MAP)
        seq = []
        for frame, m in zip(frames, POSES):
            crop = crop_of(frame, q)
            bx = box_for(u8(transform_ref.transform(crop, m)), 0.6, None) if box else None
            wv = want(crop, mode, m, bx, ROR if ror else None, GRID)
            ref.insert(u8(wv[0]), origin_of(m))
            seq.append((frame, m, bx, wv))
        set_mode(d2pc, ctx, mode, GRID)
        ctx.set_radius_outlier(*(ROR if ror else (0.0,)))
        for entry in ENTRIES:
            ctx.occupancy_reset()
            ctx.set_occupancy(**MAP)
            for frame, m, bx, wv in seq:
                ctx.set_crop_box(*(bx or (None,)))
                ctx.set_transform(m)
                got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                check(got, wv, (entry, mode, box, ror), cl)
            same_map(ctx, ref, (entry, mode, box, ror))
            st = ctx.occupancy_stats()
            assert st["frames_inserted"] == 2 and st["frames_dropped"] == 0
    finally:
        off(d2pc, ctx)


def test_launches_and_map_off(env):
    d2pc, ctx, _, _ = env
    frame = synth.s2_scene(480, 752, 9)
    try:
        ctx.set_transform(POSES[0])
        n0 = ctx.launch_count()
        ctx.process_mono8(frame)
        base = ctx.launch_count() - n0
        ctx.set_occupancy(**MAP)
        n0 = ctx.launch_count()
        ctx.process_mono8(frame)
        assert ctx.launch_count() - n0 == base + 3  # mark, apply, finish
        k0, lo0 = ctx.occupancy_voxels()
        # enabled 0 stops updates and keeps the map readable
        ctx.set_occupancy(False, **MAP)
        n0 = ctx.launch_count()
        ctx.process_mono8(synth.s2_scene(480, 752, 10))
        assert ctx.launch_count() - n0 == base
        k1, lo1 = ctx.occupancy_voxels()
        assert k1.tobytes() == k0.tobytes() and lo1.tobytes() == lo0.tobytes() and len(k0)
    finally:
        off(d2pc, ctx)


def test_720p_stream_and_fusion(env):
    d2pc, ctx, pin, _ = env
    q = ctx.get_q()
    try:
        ctx.set_transform(POSES[1])
        ctx.set_occupancy(**MAP)
        # 1280x720 frames through the stream (a ring of 3 frames, 5 submitted)
        frames = np.stack([synth.s2_scene(720, 1280, 20 + i) for i in range(3)])
        ref = map_ref.Octree(**MAP)
        ctx.process_stream(frames, collect=False, n_frames=5)
        for i in range(5):
            ref.insert(u8(want(crop_of(frames[i % 3], q), "crop", POSES[1])[0]), origin_of(POSES[1]))
        same_map(ctx, ref, "720p stream")
        # fusion: fuse_then_process, submit_fusion + wait, the fusion stream (the library's CROP cloud of the fused map)
        four = [synth.s2_scene(480, 752, 30 + i) for i in range(4)]
        ctx.set_occupancy(False, **MAP)
        ctx.set_transform(None)
        base = ctx.fuse_then_process(*four)
        ctx.set_transform(POSES[0])
        wv = want(base, "crop", POSES[0])
        ctx.occupancy_reset()
        ctx.set_occupancy(**MAP)
        ref.clear()
        check(ctx.fuse_then_process(*four), wv, "fuse_then_process", ctx.last_cloud)
        ctx.submit_fusion(0, *four, preprocess_scores=False)
        check(ctx.wait(0), wv, "submit_fusion", ctx.last_cloud)
        ctx.process_fusion_stream(np.stack([np.stack(four)] * 2), preprocess_scores=False, collect=False, n_sets=3)
        for _ in range(5):
            ref.insert(u8(wv[0]), origin_of(POSES[0]))
        same_map(ctx, ref, "fusion")
        assert ctx.occupancy_stats()["frames_inserted"] == 5
    finally:
        off(d2pc, ctx)


def test_slots_submitted_under_different_poses_and_params(env):
    d2pc, ctx, _, _ = env
    q = ctx.get_q()
    frames = [synth.s2_scene(480, 752, 40 + i) for i in range(3)]
    setups = [(POSES[0], dict(prob_hit=0.7)), (POSES[1], dict(prob_hit=0.9, prob_miss=0.3)),
              (pose(-0.5, 0.5, 0.8), dict(clamp_max=0.8, max_range=6.0))]
    try:
        ref = map_ref.Octree(**MAP)
        for s, (frame, (m, p)) in enumerate(zip(frames, setups)):
            ctx.set_transform(m)
            ctx.set_occupancy(**{**MAP, **p})
            ctx.submit(s, frame)
        for s, (frame, (m, p)) in enumerate(zip(frames, setups)):
            ctx.wait(s)
            ref.set_params(**{**{k: v for k, v in map_ref.DEFAULTS.items() if k != "resolution"}, **MAP, **p})
            ref.insert(u8(want(crop_of(frame, q), "crop", m)[0]), origin_of(m))
        same_map(ctx, ref, "slots")
    finally:
        off(d2pc, ctx)


def test_keep_cloud_0_alone_and_with_the_scan(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 11)
    wv = want(crop_of(frame, q), "crop", POSES[0])
    try:
        ctx.set_transform(POSES[0])
        # (map keep, scan): the cloud leaves unless an enabled scan or map says keep_cloud 0
        for map_keep, scan in ((0, None), (0, 1), (1, 0), (0, 0), (1, 1)):
            ctx.occupancy_reset()
            ctx.set_occupancy(keep_cloud=map_keep, **MAP)
            if scan is None:
                ctx.set_laser_scan(False)
            else:
                ctx.set_laser_scan(keep_cloud=scan)
            kept = map_keep == 1 and scan in (None, 1)
            ref = map_ref.Octree(**MAP)
            for entry in ENTRIES:
                dst = {"pinned": pin.array[:64], "registered": reg.array[:64], "pageable": np.empty(64, np.uint8),
                       "slot_into": pin.array[:64]}.get(entry)
                if kept or dst is None:
                    got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                else:
                    dst[:] = 0xA5
                    if entry == "slot_into":
                        ctx.submit(2, frame, dst)
                        got, cl = ctx.wait(2), ctx.last_cloud
                    else:
                        got, cl = ctx.process_into(frame, dst), ctx.last_cloud
                    assert np.all(dst == 0xA5), (map_keep, scan, entry)
                if kept:
                    check(got, wv, (map_keep, scan, entry), cl)
                else:
                    assert got.size == 0 and cl.width == 0 and not cl.data, (map_keep, scan, entry)
                ref.insert(u8(wv[0]), origin_of(POSES[0]))
            same_map(ctx, ref, ("keep", map_keep, scan))
    finally:
        off(d2pc, ctx)


def test_wait_with_a_too_small_destination_still_updates_the_map(env):
    d2pc, ctx, pin, _ = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 12)
    try:
        ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
        ctx.set_transform(POSES[0])
        ctx.set_occupancy(**MAP)
        ctx.submit(2, frame, pin.array[:64])
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.wait(2)
        assert e.value.status == BUFFER_TOO_SMALL
        ref = map_ref.Octree(**MAP)
        ref.insert(u8(want(crop_of(frame, q), "finite", POSES[0])[0]), origin_of(POSES[0]))
        same_map(ctx, ref, "too small")
    finally:
        off(d2pc, ctx)


def test_reset_and_resolution_change_against_a_probability_change(env):
    d2pc, ctx, _, _ = env
    q = ctx.get_q()
    f0, f1 = synth.s2_scene(480, 752, 50), synth.s2_scene(480, 752, 51)
    c0, c1 = (u8(want(crop_of(f, q), "crop", POSES[0])[0]) for f in (f0, f1))
    o = origin_of(POSES[0])
    try:
        ctx.set_transform(POSES[0])
        ctx.set_occupancy(**MAP)
        ctx.submit(0, f0)
        ctx.occupancy_reset()  # clears the frame submitted before it, even one still in flight
        ctx.submit(1, f1)
        ctx.wait(0), ctx.wait(1)
        ref = map_ref.Octree(**MAP)
        ref.insert(c1, o)
        same_map(ctx, ref, "reset")
        # a probability change keeps the map
        ctx.set_occupancy(**{**MAP, "prob_hit": 0.8})
        ctx.process_mono8(f0)
        ref.set_params(prob_hit=0.8)
        ref.insert(c0, o)
        same_map(ctx, ref, "probability change")
        # a resolution change clears it
        ctx.set_occupancy(**{**MAP, "resolution": 0.2})
        ctx.process_mono8(f1)
        ref = map_ref.Octree(**{**MAP, "resolution": 0.2})
        ref.insert(c1, o)
        same_map(ctx, ref, "resolution change")
    finally:
        off(d2pc, ctx)


def test_overflow_when_only_the_endpoints_bricks_are_new(env):
    """A map filled to max_bricks exactly by one frame; then rays that run through those bricks and end in a new one
    (the ray's last cells and the endpoint in the brick the map cannot take): the frame is dropped, the map stays bit
    for bit, and the first frame again applies."""
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(61)
    try:
        # at 0.1 m a brick is 0.8 m: points along +x up to 3.15 m need the four bricks x in [0, 3.2); many threads race
        # to create each brick, the last one included, and the frame fits exactly
        ctx.set_occupancy(resolution=0.1, max_bricks=4)
        n = 4000
        fill = np.zeros((n, 4), np.float32)
        fill[:, 0] = rng.uniform(0.0, 3.19, n)
        fill[:, 1:3] = rng.uniform(0.0, 0.79, (n, 2))
        fill[:, 3] = 1
        d_fill = torch.from_numpy(fill.view(np.uint8).reshape(-1).copy()).cuda()
        ref = map_ref.Octree(resolution=0.1)
        for _ in range(3):
            ctx.occupancy_insert_device(d_fill.data_ptr(), 1, n, n * 16, 0, np.zeros((1, 3)))
            ref.insert(fill)
        st = ctx.occupancy_stats()
        assert st["frames_inserted"] == 3 and st["frames_dropped"] == 0 and st["bricks_used"] == 4
        same_map(ctx, ref, "full")
        k0, lo0 = ctx.occupancy_voxels()
        # endpoints 3.25-3.55 m: the ray leaves the four bricks, its last cells and the endpoint share the fifth
        past = np.zeros((n, 4), np.float32)
        past[:, 0] = rng.uniform(3.25, 3.55, n)
        past[:, 1:3] = rng.uniform(0.0, 0.79, (n, 2))
        past[:, 3] = 1
        d_past = torch.from_numpy(past.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d_past.data_ptr(), 1, n, n * 16, 0, np.zeros((1, 3)))
        k1, lo1 = ctx.occupancy_voxels()
        assert k1.tobytes() == k0.tobytes() and lo1.tobytes() == lo0.tobytes()
        st = ctx.occupancy_stats()
        assert st["frames_dropped"] == 1 and st["frames_inserted"] == 3 and st["bricks_used"] == 4
        ctx.occupancy_insert_device(d_fill.data_ptr(), 1, n, n * 16, 0, np.zeros((1, 3)))
        ref.insert(fill)
        same_map(ctx, ref, "after")
        assert ctx.occupancy_stats()["frames_inserted"] == 4
    finally:
        off(d2pc, ctx)
        ctx.set_occupancy(False)


def test_overflow_drops_the_whole_frame_and_the_next_fitting_frame_applies(env):
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(60)
    try:
        ctx.set_occupancy(resolution=0.1, max_bricks=8)
        small = np.float32([[0.35, 0.05, 0.05, 1], [0.05, 0.45, 0.05, 1]])  # one brick, next to the origin
        ctx.process_f32(np.zeros((1, 1), np.float32))  # a frame of no points: inserted, nothing known
        import torch
        d = torch.from_numpy(small.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d.data_ptr(), 1, 2, 32, 0, np.zeros((1, 3)))
        ref = map_ref.Octree(resolution=0.1)
        ref.insert(small)
        same_map(ctx, ref, "before")
        k0, lo0 = ctx.occupancy_voxels()
        big = np.concatenate([rng.uniform(-20, 20, (500, 3)), np.ones((500, 1))], 1).astype(np.float32)
        db = torch.from_numpy(big.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(db.data_ptr(), 1, 500, 500 * 16, 0, np.zeros((1, 3)))
        k1, lo1 = ctx.occupancy_voxels()
        assert k1.tobytes() == k0.tobytes() and lo1.tobytes() == lo0.tobytes()
        st = ctx.occupancy_stats()
        assert st["frames_dropped"] == 1 and st["bricks_used"] >= 8 and st["bricks_capacity"] == 8
        # a frame within the bricks the map already has applies
        ctx.occupancy_insert_device(d.data_ptr(), 1, 2, 32, 0, np.zeros((1, 3)))
        ref.insert(small)
        same_map(ctx, ref, "after")
        assert ctx.occupancy_stats()["frames_inserted"] == 3
    finally:
        off(d2pc, ctx)
        ctx.set_occupancy(False)


def test_points_and_origins_outside_the_key_range(env):
    d2pc, ctx, _, _ = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 13)
    try:
        # at 0.05 m the keys end at +-1638.4 m: a translation of 1630 m puts part of the cloud beyond them
        m = pose(1630.0, 0.0, 1.0)
        ctx.set_transform(m)
        ctx.set_occupancy(resolution=0.05)
        ctx.process_mono8(frame)
        ref = map_ref.Octree(resolution=0.05)
        ref.insert(u8(want(crop_of(frame, q), "crop", m)[0]), origin_of(m))
        same_map(ctx, ref, "edge of the key range")
        # an origin beyond them (x = -1640 m) looking along +x at points 3-32 m away, inside them: no ray, only the
        # endpoints, each one hit
        ctx.occupancy_reset()
        m = pose(-1640.0, 0.0, 1.0)
        ctx.set_transform(m)
        ctx.process_mono8(frame)
        ref.clear()
        ref.insert(u8(want(crop_of(frame, q), "crop", m)[0]), origin_of(m))
        n = same_map(ctx, ref, "origin outside")
        _, lo = ctx.occupancy_voxels()
        assert n > 1000 and (lo == np.float32(map_ref.logodds(0.7))).all()
    finally:
        off(d2pc, ctx)


def test_device_entry_counts_origins_and_refusals(env):
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(70)
    try:
        with pytest.raises(d2pc.D2pcError):  # the map must be on
            ctx.occupancy_insert_device(1 << 20, 1, 1, 16, 0, np.zeros((1, 3)))
        ctx.set_occupancy(resolution=0.1, max_range=8.0)
        n_max, nf = 3000, 4
        stride = n_max * 16 + 64
        host = np.zeros(nf * stride // 4, np.float32)
        pts = np.concatenate([rng.uniform(-12, 12, (nf * n_max, 3)), np.ones((nf * n_max, 1))], 1).astype(np.float32)
        pts[::97, 1] = np.nan
        pts[::89, 0] = np.inf
        for f in range(nf):
            host.view(np.uint8)[f * stride: f * stride + n_max * 16] = pts[f * n_max:(f + 1) * n_max].view(np.uint8).reshape(-1)
        counts = np.uint32([n_max, 1234, 0, n_max * 3])
        origins = rng.uniform(-2, 2, (nf, 3)).astype(np.float32)
        d_in = torch.from_numpy(host.view(np.uint8).copy()).cuda()
        d_cnt = torch.from_numpy(counts.view(np.int32)).cuda()
        ctx.occupancy_insert_device(d_in.data_ptr(), nf, n_max, stride, d_cnt.data_ptr(), origins)
        ref = map_ref.Octree(resolution=0.1, max_range=8.0)
        for f in range(nf):
            k = min(int(counts[f]), n_max)
            ref.insert(pts[f * n_max: f * n_max + k], origins[f])
        same_map(ctx, ref, "device entry")
        for bad in (dict(d=d_in.data_ptr() + 4), dict(stride=stride + 4), dict(stride=16)):
            with pytest.raises(d2pc.D2pcError):
                ctx.occupancy_insert_device(bad.get("d", d_in.data_ptr()), nf, n_max, bad.get("stride", stride), 0,
                                            origins)
    finally:
        off(d2pc, ctx)


def test_refused_settings_keep_the_previous_one(env):
    d2pc, ctx, _, _ = env
    try:
        ctx.set_occupancy(resolution=0.2)
        for bad in (dict(resolution=0.0), dict(resolution=float("inf")), dict(resolution=float("nan")),
                    dict(prob_hit=0.4), dict(prob_miss=0.6), dict(prob_hit=1.0), dict(clamp_min=0.0),
                    dict(clamp_min=0.9, clamp_max=0.8), dict(occupancy_thres=1.0), dict(max_range=float("nan")),
                    dict(max_bricks=0), dict(max_bricks=(1 << 26) + 1)):
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.set_occupancy(**bad)
            assert e.value.status == INVALID_ARG, bad
            assert ctx.get_occupancy().resolution == 0.2
        p = d2pc.occupancy_params()
        p.struct_size = 8
        assert d2pc.lib().d2pc_set_occupancy(ctx._h, C.byref(p)) == INVALID_ARG
        dflt = d2pc.OccupancyParams()
        d2pc.lib().d2pc_occupancy_params_default(C.byref(dflt))
        assert (dflt.enabled, dflt.resolution, dflt.prob_hit, dflt.prob_miss, dflt.clamp_min, dflt.clamp_max,
                dflt.occupancy_thres, dflt.max_range, dflt.keep_cloud) == (0, 0.05, 0.7, 0.4, 0.12, 0.97, 0.5, -1.0, 1)
    finally:
        off(d2pc, ctx)


def test_export_buffers_canaries_and_wire_format(env):
    d2pc, ctx, _, _ = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 14)
    try:
        ctx.set_transform(POSES[0])
        ctx.set_occupancy(**MAP)
        ctx.process_mono8(frame)
        ref = map_ref.Octree(**MAP)
        ref.insert(u8(want(crop_of(frame, q), "crop", POSES[0])[0]), origin_of(POSES[0]))
        want_c = ref.centers()
        n = len(want_c)
        L = d2pc.lib()
        cl = d2pc.Cloud()
        assert L.d2pc_occupancy_centers(ctx._h, None, 0, C.byref(cl)) == BUFFER_TOO_SMALL and cl.width == n
        buf = np.full(n * 16 + 128, 0xA5, np.uint8)
        assert L.d2pc_occupancy_centers(ctx._h, buf.ctypes.data + 64, n * 16 - 1, C.byref(cl)) == BUFFER_TOO_SMALL
        assert (buf == 0xA5).all()
        assert L.d2pc_occupancy_centers(ctx._h, buf.ctypes.data + 64, n * 16, C.byref(cl)) == 0
        assert buf[64:-64].tobytes() == want_c.tobytes() and (buf[:64] == 0xA5).all() and (buf[-64:] == 0xA5).all()
        assert cl.width == n and cl.is_dense == 1 and cl.point_step == 16
        wire = ctx.serialize_pointcloud2(cl, seq=3, sec=4, nsec=5)
        assert wire.find(want_c.tobytes()) > 0 and wire[-1] == 1
        wk, wlo = ref.voxels()
        m = len(wk)
        nn = C.c_uint64()
        keys = np.full(m + 8, 0xA5A5A5A5A5A5A5A5, np.uint64)
        lo = np.full(m + 8, -7.0, np.float32)
        assert L.d2pc_occupancy_voxels(ctx._h, keys.ctypes.data, lo.ctypes.data, m - 1, C.byref(nn)) == BUFFER_TOO_SMALL
        assert nn.value == m and (keys == 0xA5A5A5A5A5A5A5A5).all()
        assert L.d2pc_occupancy_voxels(ctx._h, keys.ctypes.data, lo.ctypes.data, m, C.byref(nn)) == 0
        assert (keys[m:] == 0xA5A5A5A5A5A5A5A5).all() and (lo[m:] == -7.0).all()
        packed = wk[:, 0].astype(np.uint64) | (wk[:, 1].astype(np.uint64) << 16) | (wk[:, 2].astype(np.uint64) << 32)
        assert keys[:m].tobytes() == packed.tobytes() and lo[:m].tobytes() == wlo.tobytes()
    finally:
        off(d2pc, ctx)


def _fuzz_case(case, ctx):
    import torch
    rng = np.random.default_rng(SEED0 + case)
    res = float(rng.choice([0.05, 0.1, 0.13, 0.5]))
    p = dict(resolution=res, prob_hit=float(rng.uniform(0.5, 0.95)), prob_miss=float(rng.uniform(0.05, 0.5)),
             clamp_min=float(rng.uniform(0.01, 0.3)), clamp_max=float(rng.uniform(0.7, 0.99)),
             occupancy_thres=float(rng.uniform(0.2, 0.8)), max_range=float(rng.choice([-1.0, 2.0, 7.5])))
    ctx.occupancy_reset()
    ctx.set_occupancy(**p)
    ref = map_ref.Octree(**p)
    for f in range(int(rng.integers(1, 5))):
        n = int(rng.integers(1, 4000))
        scale = float(rng.choice([1.0, 10.0, 30.0]))
        pts = np.concatenate([rng.uniform(-scale, scale, (n, 3)), np.ones((n, 1))], 1).astype(np.float32)
        snap = rng.random(n) < 0.3  # points on voxel faces and corners
        pts[snap, :3] = np.round(pts[snap, :3] / res).astype(np.float32) * np.float32(res)
        pts[rng.random(n) < 0.02, int(rng.integers(0, 3))] = np.nan
        o = (rng.uniform(-2, 2, 3) if rng.random() < 0.7 else np.round(rng.uniform(-2, 2, 3) / res) * res).astype(np.float32)
        if rng.random() < 0.3:  # the clamp bounds change between frames
            p2 = dict(clamp_min=float(rng.uniform(0.01, 0.3)), clamp_max=float(rng.uniform(0.7, 0.99)))
            ctx.set_occupancy(**{**p, **p2})
            ref.set_params(**p2)
        d = torch.from_numpy(pts.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d.data_ptr(), 1, n, n * 16, 0, o.reshape(1, 3))
        ref.insert(pts, o)
    ctx.set_occupancy(**p)
    ref.set_params(occupancy_thres=p["occupancy_thres"])
    same_map(ctx, ref, ("fuzz", case, p))


def test_occupancy_fuzz_against_the_literal_octree(env):
    d2pc, ctx, _, _ = env
    try:
        for case in range(N_FUZZ):
            _fuzz_case(case, ctx)
    finally:
        off(d2pc, ctx)


def _node_launch(tmp_path, name, params):
    launch = tmp_path / f"{name}.launch"
    launch.write_text('<launch>\n  <node name="n" pkg="p" type="t">\n' +
                      "".join(f'    <param name="{k}" value="{v}"/>\n' for k, v in params.items()) +
                      "  </node>\n</launch>\n")
    return launch


NODE_POSE = dict(tx=0.5, ty=-0.2, tz=1.0, roll=-1.5707963, pitch=0.0, yaw=-1.5707963)  # optical -> z-up


def test_node1_publishes_the_map_centres(tmp_path):
    """The node mirror with transform_* and map_* params: after each frame /octomap_point_cloud_centers carries the
    occupied voxel centres of the map of every cloud so far, with the cloud's header and frame_id; with
    map_keep_cloud 0 /point_cloud is not published.  The same bytes under ASan / UBSan."""
    import oracle
    from disparity_to_point_cloud_b200 import build
    from test_gpu_crop_box import transform_of
    from test_host_mirror import ASAN_ENV
    harness, harness_asan = build.build_harness(), build.build_harness(sanitize=True)
    imgs = [synth.s2_scene(480, 752, 70 + i) for i in range(2)]
    raws = []
    for i, img in enumerate(imgs):
        raws.append(tmp_path / f"in{i}.raw")
        raws[-1].write_bytes(np.ascontiguousarray(img).tobytes())
    q = oracle.q_from_intrinsics()
    t = transform_of((NODE_POSE["roll"], NODE_POSE["pitch"], NODE_POSE["yaw"]),
                     (NODE_POSE["tx"], NODE_POSE["ty"], NODE_POSE["tz"]))
    clouds = [want(oracle.disparity_cb_mono8(img, q), "crop", t) for img in imgs]
    mp = dict(resolution=0.1, sensor_model_hit=0.75, sensor_model_miss=0.35, sensor_model_min=0.15,
              sensor_model_max=0.95, occupancy_thres=0.6, max_range=9.0, max_bricks=100000)
    ref = map_ref.Octree(resolution=0.1, prob_hit=0.75, prob_miss=0.35, clamp_min=0.15, clamp_max=0.95,
                         occupancy_thres=0.6, max_range=9.0)
    for c in clouds:
        ref.insert(u8(c[0]), origin_of(t))
    centres = ref.centers()
    assert len(centres) > 100
    fid = "/map"
    want_centres = oracle.serialize_pointcloud2(centres.view(np.uint8).reshape(-1), seq=0, sec=4, nsec=4,
                                                frame_id=fid, is_dense=1)
    for keep in (1, 0):
        params = dict(transform_enable=1, transform_target_frame=fid, map_enable=1, map_keep_cloud=keep,
                      **{f"transform_{k}": v for k, v in NODE_POSE.items()}, **{f"map_{k}": v for k, v in mp.items()})
        launch = _node_launch(tmp_path, f"m{keep}", params)
        outs = {}
        for name, exe in (("plain", harness), ("asan", harness_asan)):
            cloud_bin, map_bin = tmp_path / f"c{keep}{name}.bin", tmp_path / f"m{keep}{name}.bin"
            r = subprocess.run([exe, "node1map", str(launch), "752", "480", str(cloud_bin), str(map_bin)] +
                               [str(r_) for r_ in raws], env=ASAN_ENV, capture_output=True, text=True)
            assert r.returncode == 0, (name, r.stderr[-3000:])
            outs[name] = (cloud_bin.read_bytes(), map_bin.read_bytes())
        assert outs["plain"] == outs["asan"], keep
        cloud_b, map_b = outs["plain"]
        assert map_b == want_centres, keep
        if keep:
            assert cloud_b == oracle.serialize_pointcloud2(u8(clouds[-1][0]), seq=0, sec=4, nsec=4, frame_id=fid,
                                                           is_dense=clouds[-1][1])
        else:
            assert cloud_b == b""
