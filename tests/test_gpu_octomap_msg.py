"""GPU: the occupancy map serialized as octomap_msgs/Octomap (d2pc_occupancy_octomap) byte for byte against octomap's
pointer OcTree restated literally (tests/map_ref/octree_pointer.cpp, updateNode with pruning, writeData and
writeBinaryData), fed the very clouds the library published: through the host entries, the device entry and the
fusion entry, under per-frame poses, clamp and threshold changes, a reset and a dropped frame; a seeded fuzz; a 720p
map of more than 10^6 known voxels against the C recipe (tests/map_ref/octomap_msg.c) fed d2pc_occupancy_voxels; and
the node's /octomap_full and /octomap_binary through the offline harness.  D2PC_OCTOMAP_FUZZ_CASES /
D2PC_OCTOMAP_FUZZ_SEED set the fuzz (default 30)."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import map_ref
from map_ref import octree
from disparity_to_point_cloud_b200 import synth

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_OCTOMAP_FUZZ_CASES", "30"))
SEED0 = int(os.environ.get("D2PC_OCTOMAP_FUZZ_SEED", "94000"))
INVALID_ARG = -1
MAP = dict(resolution=0.1, max_range=12.0)
PARAM_KEYS = ("prob_hit", "prob_miss", "clamp_min", "clamp_max", "occupancy_thres", "max_range")


def pose(tx, ty, tz):
    """camera optical frame -> a z-up world frame, the camera at (tx, ty, tz)"""
    return np.float32([[0, 0, 1, tx], [-1, 0, 0, ty], [0, -1, 0, tz]])


POSES = [pose(0.0, 0.0, 1.0), pose(0.05, -0.03, 1.02), pose(0.7, -0.3, 1.2)]


def origin_of(m):
    return (m[0][3], m[1][3], m[2][3])


@pytest.fixture(scope="module")
def env():
    import disparity_to_point_cloud_b200 as d2pc
    ctx = d2pc.Context(n_slots=3)
    yield d2pc, ctx
    ctx.close()


def off(ctx):
    ctx.set_transform(None)
    ctx.set_occupancy(False)
    ctx.occupancy_reset()


def ptree(**params):
    p = {**MAP, **params}
    return octree.PointerTree(**p)


def same(ctx, ref, what, prunes=True):
    """both formats byte for byte; returns the full stream's size"""
    full, binary = ctx.occupancy_octomap(), ctx.occupancy_octomap(binary=True)
    want_full, want_binary = ref.data(), ref.data(True)
    assert len(full) == len(want_full) and full == want_full, (what, "full", len(full), len(want_full))
    assert binary == want_binary, (what, "binary", len(binary), len(want_binary))
    if prunes:
        depths = [0] * 17
        ref.voxels(depths)
        assert sum(depths[:16]) > 0, (what, depths)  # the map really has pruned leaves
    return len(full)


def test_entries_poses_params_reset_and_drop(env):
    import torch
    d2pc, ctx = env
    try:
        ref = ptree()
        ctx.set_occupancy(**MAP)
        assert ctx.occupancy_octomap() == b"" and ctx.occupancy_octomap(binary=True) == b""  # empty map
        for b in (-1, 2):
            assert d2pc.lib().d2pc_occupancy_octomap(ctx._h, b, C.byref(d2pc.Octomap())) == INVALID_ARG
        # repeated frames from nearby poses through several host entries: free space clamps and prunes
        steps = []
        for i in range(8):
            frame = synth.s2_scene(480, 752, 5 + (i % 2)) if i % 3 else synth.s3_float(480, 752, 7)
            steps.append((frame, POSES[i % 2], {}))
        steps.append((synth.s2_scene(480, 752, 9), POSES[2], dict(clamp_max=0.9, occupancy_thres=0.6)))
        steps.append((synth.s2_scene(480, 752, 10), POSES[0], dict(clamp_min=0.2, prob_hit=0.8)))
        for i, (frame, m, p) in enumerate(steps):
            ctx.set_transform(m)
            ctx.set_occupancy(**{**MAP, **p})
            ref.set_params(**{k: v for k, v in {**map_ref.DEFAULTS, **MAP, **p}.items() if k in PARAM_KEYS})
            entry = i % 3
            if entry == 0:
                cloud = ctx.process_mono8(frame) if frame.dtype == np.uint8 else ctx.process_f32(frame)
            elif entry == 1:
                ctx.submit(1, frame)
                cloud = ctx.wait(1)
            else:
                ctx.submit(2, frame)
                cloud = ctx.wait(2)
            ref.insert(cloud, origin_of(m))
            same(ctx, ref, ("host", i), prunes=i == len(steps) - 1)
        # the device entry, two frames in one call
        rng = np.random.default_rng(3)
        pts = []
        for f in range(2):
            d = rng.normal(size=(4000, 3))
            d /= np.linalg.norm(d, axis=1, keepdims=True)
            pts.append(np.concatenate([d * rng.uniform(1, 4, (4000, 1)), np.ones((4000, 1))], 1).astype(np.float32))
        origins = np.float32([[0.1, 0.0, 1.0], [0.0, 0.1, 1.0]])
        dev = torch.from_numpy(np.concatenate(pts).view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(dev.data_ptr(), 2, 4000, 4000 * 16, 0, origins)
        for f in range(2):
            ref.insert(pts[f], origins[f])
        same(ctx, ref, "device", prunes=False)
        # the fusion entry
        ctx.set_transform(POSES[0])
        four = [synth.s2_scene(480, 752, 30 + i) for i in range(4)]
        for _ in range(2):
            ref.insert(ctx.fuse_then_process(*four), origin_of(POSES[0]))
        same(ctx, ref, "fusion", prunes=False)
        # a frame the map cannot take is dropped whole: the bytes stay those of the map before it.  A new max_bricks
        # clears the map: one small frame, then a far-reaching one that needs more bricks than the map has
        ref.clear()
        ctx.set_transform(POSES[0])
        small = np.float32([[0.55, 0.05, 1.05, 1]])
        d_small = torch.from_numpy(small.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.set_occupancy(**{**MAP, **steps[-1][2], "max_bricks": 4})
        ctx.occupancy_insert_device(d_small.data_ptr(), 1, 1, 16, 0, np.zeros((1, 3)))
        ref.insert(small, (0, 0, 0))
        big = pts[0]
        d_big = torch.from_numpy(big.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d_big.data_ptr(), 1, len(big), len(big) * 16, 0, np.zeros((1, 3)))
        assert ctx.occupancy_stats()["frames_dropped"] == 1
        same(ctx, ref, "dropped", prunes=False)
        # after a reset
        ctx.set_occupancy(**MAP)
        ctx.occupancy_reset()
        assert ctx.occupancy_octomap() == b"" and ctx.occupancy_octomap(binary=True) == b""
        ref = ptree()
        for i in range(6):
            ctx.set_transform(POSES[i % 2])
            ref.insert(ctx.process_mono8(synth.s2_scene(480, 752, 40 + (i % 2))), origin_of(POSES[i % 2]))
        same(ctx, ref, "reset", prunes=False)
    finally:
        off(ctx)


def test_octomap_fuzz_against_the_pointer_tree(env):
    import torch
    d2pc, ctx = env
    try:
        for case in range(N_FUZZ):
            rng = np.random.default_rng(SEED0 + case)
            res = float(rng.choice([0.05, 0.1, 0.2]))
            p0 = dict(resolution=res, max_range=float(rng.choice([-1.0, 3.0, 8.0])))
            ctx.set_occupancy(**p0)
            ctx.occupancy_reset()
            ref = octree.PointerTree(**p0)
            centre = rng.uniform(-2, 2, 3)
            for f in range(int(rng.integers(1, 7))):
                p = dict(p0)
                if rng.random() < 0.4:
                    p.update(clamp_min=float(rng.uniform(0.05, 0.3)), clamp_max=float(rng.uniform(0.7, 0.99)),
                             occupancy_thres=float(rng.uniform(0.3, 0.8)), prob_hit=float(rng.uniform(0.55, 0.9)))
                ctx.set_occupancy(**p)
                ref.set_params(**{k: v for k, v in {**map_ref.DEFAULTS, **p}.items() if k in PARAM_KEYS})
                n = int(rng.integers(1, 3000))
                o = (centre + rng.uniform(-0.2, 0.2, 3)).astype(np.float32)
                d = rng.normal(size=(n, 3))
                d /= np.linalg.norm(d, axis=1, keepdims=True)
                pts = np.concatenate([o + d * rng.uniform(0.05, 5, (n, 1)), np.ones((n, 1))], 1).astype(np.float32)
                if rng.random() < 0.3:  # a dense wall: uniform octants
                    g = np.arange(-0.6, 0.6, res / 3, dtype=np.float32)
                    yy, zz = np.meshgrid(g, g)
                    w = np.stack([np.full(yy.size, o[0] + 1.5), o[1] + yy.ravel(), o[2] + zz.ravel(),
                                  np.ones(yy.size)], 1).astype(np.float32)
                    pts = np.concatenate([pts, w])
                dev = torch.from_numpy(pts.view(np.uint8).reshape(-1).copy()).cuda()
                ctx.occupancy_insert_device(dev.data_ptr(), 1, len(pts), len(pts) * 16, 0, o.reshape(1, 3))
                ref.insert(pts, o)
            same(ctx, ref, ("fuzz", case), prunes=False)
    finally:
        off(ctx)


def test_large_720p_map_against_the_recipe(env):
    d2pc, ctx = env
    try:
        ctx.set_occupancy(resolution=0.02, max_bricks=1 << 20)
        ctx.occupancy_reset()
        frames = np.stack([synth.s2_scene(720, 1280, 50 + i) for i in range(3)])
        for i in range(6):
            ctx.set_transform(pose(0.3 * i, 0.1 * i, 1.0))
            ctx.process_stream(frames, collect=False, n_frames=3)
            if ctx.occupancy_stats()["known_voxels"] >= 10 ** 6:
                break
        st = ctx.occupancy_stats()
        assert st["known_voxels"] >= 10 ** 6 and st["frames_dropped"] == 0, st
        keys, lo = ctx.occupancy_voxels()
        for binary in (False, True):
            got = ctx.occupancy_octomap(binary=binary)
            assert got == octree.octomap_data(keys, lo, binary, 0.5), binary
        # the full stream reads back to the flat map
        rk, rlo = octree.read_full(ctx.occupancy_octomap())
        assert rk.tobytes() == keys.tobytes() and rlo.tobytes() == lo.tobytes()
    finally:
        off(ctx)


def octomap_wire(binary, data, res, sec, nsec, frame_id):
    f = frame_id.encode()
    return (struct.pack("<IIII", 0, sec, nsec, len(f)) + f + struct.pack("<BI", binary, 6) + b"OcTree" +
            struct.pack("<dI", res, len(data)) + data)


def test_node_publishes_octomap_full_and_binary(tmp_path):
    """The node mirror with map_enable: /octomap_full and /octomap_binary carry the API's data with the cloud's header,
    only while subscribed; /point_cloud and the centres are what node1map gives; with the map off nothing octomap is
    advertised."""
    import disparity_to_point_cloud_b200 as d2pc
    from disparity_to_point_cloud_b200 import build
    from test_gpu_crop_box import transform_of
    from test_gpu_occupancy import NODE_POSE, _node_launch
    harness = build.build_harness()
    imgs = [synth.s2_scene(480, 752, 70 + i) for i in range(3)]
    raws = []
    for i, img in enumerate(imgs):
        raws.append(tmp_path / f"in{i}.raw")
        raws[-1].write_bytes(np.ascontiguousarray(img).tobytes())
    mp = dict(resolution=0.1, sensor_model_hit=0.75, sensor_model_miss=0.35, sensor_model_min=0.15,
              sensor_model_max=0.95, occupancy_thres=0.6, max_range=9.0, max_bricks=100000)
    fid = "/map"
    params = dict(transform_enable=1, transform_target_frame=fid, map_enable=1,
                  **{f"transform_{k}": v for k, v in NODE_POSE.items()}, **{f"map_{k}": v for k, v in mp.items()})
    # the API's data for the same frames
    t = transform_of((NODE_POSE["roll"], NODE_POSE["pitch"], NODE_POSE["yaw"]),
                     (NODE_POSE["tx"], NODE_POSE["ty"], NODE_POSE["tz"]))
    with d2pc.Context() as ctx:
        ctx.set_transform(t)
        ctx.set_occupancy(resolution=0.1, prob_hit=0.75, prob_miss=0.35, clamp_min=0.15, clamp_max=0.95,
                          occupancy_thres=0.6, max_range=9.0, max_bricks=100000)
        for img in imgs:
            ctx.process_mono8(img)
        api = [ctx.occupancy_octomap(), ctx.occupancy_octomap(binary=True)]
    assert len(api[0]) > 1000 and len(api[1]) > 100
    sec = 3 + len(imgs) - 1
    launch = _node_launch(tmp_path, "on", params)
    out = {k: tmp_path / f"{k}.bin" for k in ("c", "m", "f", "b", "c1", "m1")}
    r = subprocess.run([harness, "node1octomap", str(launch), "752", "480", str(out["c"]), str(out["m"]),
                        str(out["f"]), str(out["b"])] + [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["f"].read_bytes() == octomap_wire(0, api[0], 0.1, sec, 4, fid)
    assert out["b"].read_bytes() == octomap_wire(1, api[1], 0.1, sec, 4, fid)
    # /point_cloud and the centres are those of node1map
    r = subprocess.run([harness, "node1map", str(launch), "752", "480", str(out["c1"]), str(out["m1"])] +
                       [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["c"].read_bytes() == out["c1"].read_bytes() and len(out["c"].read_bytes()) > 0
    assert out["m"].read_bytes() == out["m1"].read_bytes() and len(out["m"].read_bytes()) > 0
    # only /octomap_binary subscribed: /octomap_full is never filled, the binary message is the same
    out["b"].unlink()
    r = subprocess.run([harness, "node1octomap", str(launch), "752", "480", str(out["c"]), str(out["m"]), "-",
                        str(out["b"])] + [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["b"].read_bytes() == octomap_wire(1, api[1], 0.1, sec, 4, fid)
    # map off: no octomap topic is advertised (the harness checks), the cloud is node1map's
    off_launch = _node_launch(tmp_path, "off", {k: v for k, v in params.items() if k != "map_enable"})
    r = subprocess.run([harness, "node1octomap", str(off_launch), "752", "480", str(out["c1"]), str(out["m1"]),
                        str(out["f"]), str(out["b"])] + [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["f"].read_bytes() == b"" and out["b"].read_bytes() == b"" and out["m1"].read_bytes() == b""
    assert out["c1"].read_bytes() == out["c"].read_bytes()
