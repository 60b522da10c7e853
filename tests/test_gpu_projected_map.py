"""GPU: the occupancy map projected to 2-D (d2pc_occupancy_projected_map, octomap_server's /projected_map) byte for byte
against octomap_server's projection restated literally over octomap's pointer tree (tests/map_ref/projected_map.cpp),
fed the very clouds the library published: through the host entries, the device entry and the fusion entry, under
per-frame poses, clamp and threshold changes, a reset and a dropped frame, finite z limits and padding; a seeded fuzz;
a 720p map of more than 10^6 known voxels against the C recipe (tests/map_ref/projected_map.c) fed
d2pc_occupancy_voxels; the empty map, argument refusal, the key range, the octomap export unchanged by a projection,
the grid's cells kept while the octomap export grows its buffer; and the node's /projected_map through the offline harness.  D2PC_PROJMAP_FUZZ_CASES / D2PC_PROJMAP_FUZZ_SEED set the
fuzz (default 30)."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import map_ref
from map_ref import projected
from disparity_to_point_cloud_b200 import synth
from test_gpu_octomap_msg import MAP, PARAM_KEYS, POSES, origin_of, pose

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_PROJMAP_FUZZ_CASES", "30"))
SEED0 = int(os.environ.get("D2PC_PROJMAP_FUZZ_SEED", "95000"))
INVALID_ARG, BAD_DIMS = -1, -3
LIMITS = [dict(), dict(occupancy_min_z=0.3, occupancy_max_z=1.6), dict(occupancy_min_z=1.05, occupancy_max_z=1.1),
          dict(min_x_size=40.0, min_y_size=3.0), dict(occupancy_max_z=0.9, min_x_size=0.5, min_y_size=25.0)]


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


def same(ctx, ref, what, limits=LIMITS):
    """the device grid byte for byte against the pointer tree's under every set of limits; returns the grids"""
    out = []
    for kw in limits:
        cells, res, origin = ctx.occupancy_projected_map(**kw)
        want = ref.projected_map(**kw)
        assert want is not None and not isinstance(want, str), (what, kw, want)
        wc, wr, wo = want
        assert cells.shape == wc.shape, (what, kw, cells.shape, wc.shape)
        assert cells.tobytes() == wc.tobytes(), (what, kw, int((cells != wc).sum()))
        assert np.float32(res) == np.float32(wr), (what, kw)
        assert np.float64(origin).tobytes() == np.float64(wo).tobytes(), (what, kw, origin, wo)
        out.append(cells)
    return out


def empty(ctx):
    cells, res, origin = ctx.occupancy_projected_map()
    return cells.shape == (0, 0) and origin == (0.0, 0.0)


def test_entries_poses_params_reset_and_drop(env):
    import torch
    d2pc, ctx = env
    try:
        ref = projected.ProjTree(**MAP)
        ctx.set_occupancy(**MAP)
        assert empty(ctx)
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
            same(ctx, ref, ("host", i), LIMITS if i in (0, len(steps) - 1) else LIMITS[:2])
        depths = [0] * 17
        ref.voxels(depths)
        assert sum(depths[:16]) > 0, depths  # the map really has coarse leaves
        grids = same(ctx, ref, "final")
        assert all((g == 100).any() and (g == 0).any() and (g == -1).any() for g in grids[:2])
        # a projection leaves the octomap export as it was
        full, binary = ctx.occupancy_octomap(), ctx.occupancy_octomap(binary=True)
        ctx.occupancy_projected_map(occupancy_min_z=0.5)
        assert ctx.occupancy_octomap() == full == ref.data() and ctx.occupancy_octomap(binary=True) == binary
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
        same(ctx, ref, "device")
        # the fusion entry
        ctx.set_transform(POSES[0])
        four = [synth.s2_scene(480, 752, 30 + i) for i in range(4)]
        for _ in range(2):
            ref.insert(ctx.fuse_then_process(*four), origin_of(POSES[0]))
        same(ctx, ref, "fusion")
        # a dropped frame leaves the grid of the map before it (a new max_bricks clears the map)
        ref.clear()
        small = np.float32([[0.55, 0.05, 1.05, 1]])
        d_small = torch.from_numpy(small.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.set_occupancy(**{**MAP, **steps[-1][2], "max_bricks": 4})
        ctx.occupancy_insert_device(d_small.data_ptr(), 1, 1, 16, 0, np.zeros((1, 3)))
        ref.insert(small, (0, 0, 0))
        d_big = torch.from_numpy(pts[0].view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d_big.data_ptr(), 1, len(pts[0]), len(pts[0]) * 16, 0, np.zeros((1, 3)))
        assert ctx.occupancy_stats()["frames_dropped"] == 1
        same(ctx, ref, "dropped")
        # after a reset
        ctx.set_occupancy(**MAP)
        ctx.occupancy_reset()
        assert empty(ctx)
        ref = projected.ProjTree(**MAP)
        for i in range(6):
            ctx.set_transform(POSES[i % 2])
            ref.insert(ctx.process_mono8(synth.s2_scene(480, 752, 40 + (i % 2))), origin_of(POSES[i % 2]))
        same(ctx, ref, "reset")
    finally:
        off(ctx)


def test_grid_outlives_other_exports_until_the_next_projection():
    """d2pc_grid_map's cells stay valid until the next projection: an octomap export that grows its own result buffer
    in between leaves them as they were.  A context of its own, so the octomap buffer starts at its first size."""
    import torch
    import disparity_to_point_cloud_b200 as d2pc
    L = d2pc.lib()
    with d2pc.Context() as ctx:
        ctx.set_occupancy(**MAP)
        pt = np.float32([[1.55, 0.35, 1.05, 1.0]])
        d = torch.from_numpy(pt.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d.data_ptr(), 1, 1, 16, 0, np.float32([[0.0, 0.0, 1.0]]))
        small = ctx.occupancy_octomap()
        assert 0 < len(small) < 1 << 16  # the octomap result buffer holds 64 KiB
        p, g = d2pc.ProjectedMapParams(), d2pc.GridMap()
        L.d2pc_projected_map_params_default(C.byref(p))
        assert L.d2pc_occupancy_projected_map(ctx._h, C.byref(p), C.byref(g)) == 0 and g.width * g.height > 0
        n = g.width * g.height
        want = np.ctypeslib.as_array(g.data, (n,)).copy()
        for i in range(4):
            ctx.set_transform(POSES[i % 2])
            ctx.process_mono8(synth.s2_scene(480, 752, 61 + i))
        assert len(ctx.occupancy_octomap()) > 1 << 16  # the octomap result buffer grew
        assert np.ctypeslib.as_array(g.data, (n,)).tobytes() == want.tobytes()


def test_arguments_and_the_key_range(env):
    import torch
    d2pc, ctx = env
    L = d2pc.lib()
    try:
        ctx.set_occupancy(**MAP)
        ctx.occupancy_reset()
        p, g = d2pc.ProjectedMapParams(), d2pc.GridMap()
        L.d2pc_projected_map_params_default(C.byref(p))
        assert p.struct_size == C.sizeof(p) and p.occupancy_min_z == -np.finfo(np.float64).max
        assert p.occupancy_max_z == np.finfo(np.float64).max and p.min_x_size == 0 == p.min_y_size
        assert L.d2pc_occupancy_projected_map(ctx._h, C.byref(p), C.byref(g)) == 0 and g.width == 0 == g.height
        assert not g.data
        for field, v in (("occupancy_min_z", np.nan), ("occupancy_max_z", np.nan), ("min_x_size", -0.1),
                         ("min_y_size", np.inf), ("min_x_size", np.nan), ("struct_size", 8)):
            q = d2pc.ProjectedMapParams()
            L.d2pc_projected_map_params_default(C.byref(q))
            setattr(q, field, v)
            assert L.d2pc_occupancy_projected_map(ctx._h, C.byref(q), C.byref(g)) == INVALID_ARG, field
        assert L.d2pc_occupancy_projected_map(ctx._h, None, C.byref(g)) == INVALID_ARG
        assert L.d2pc_occupancy_projected_map(ctx._h, C.byref(p), None) == INVALID_ARG
        # infinite z limits are allowed; a map at key 65535 on x has no padded max key at 0.1 m
        ctx.occupancy_projected_map(occupancy_min_z=-np.inf, occupancy_max_z=np.inf)
        ref = projected.ProjTree(**MAP)
        pt = np.float32([[3276.75, 0.0, 0.0, 1.0]])
        o = np.float32([3276.65, 0.0, 0.0])
        d = torch.from_numpy(pt.view(np.uint8).reshape(-1).copy()).cuda()
        ctx.occupancy_insert_device(d.data_ptr(), 1, 1, 16, 0, o.reshape(1, 3))
        ref.insert(pt, o)
        assert ref.projected_map() == "BAD_DIMS"
        assert L.d2pc_occupancy_projected_map(ctx._h, C.byref(p), C.byref(g)) == BAD_DIMS
        with pytest.raises(d2pc.D2pcError):
            ctx.occupancy_projected_map()
    finally:
        off(ctx)


def test_projected_map_fuzz_against_the_pointer_tree(env):
    import torch
    d2pc, ctx = env
    try:
        for case in range(N_FUZZ):
            rng = np.random.default_rng(SEED0 + case)
            res = float(rng.choice([0.05, 0.1, 0.2]))
            p0 = dict(resolution=res, max_range=float(rng.choice([-1.0, 3.0, 8.0])))
            ctx.set_occupancy(**p0)
            ctx.occupancy_reset()
            ref = projected.ProjTree(**p0)
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
            z = float(centre[2])
            kw = dict(occupancy_min_z=z + float(rng.uniform(-2, 0.5)), occupancy_max_z=z + float(rng.uniform(-0.5, 2)),
                      min_x_size=float(rng.choice([0.0, rng.uniform(0, 12)])),
                      min_y_size=float(rng.choice([0.0, rng.uniform(0, 12)])))
            same(ctx, ref, ("fuzz", case), [dict(), kw])
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
        for kw in (dict(), dict(occupancy_min_z=0.4, occupancy_max_z=1.5, min_x_size=30.0, min_y_size=8.0)):
            cells, res, origin = ctx.occupancy_projected_map(**kw)
            want = projected.projected_map(keys, lo, 0.02, 0.5, **kw)
            assert cells.shape == want[0].shape and cells.tobytes() == want[0].tobytes(), kw
            assert np.float64(origin).tobytes() == np.float64(want[2]).tobytes() and np.float32(res) == want[1]
        # and the pointer tree built from the same voxels
        tree = projected.ProjTree(resolution=0.02)
        tree.set_values(keys, lo)
        same(ctx, tree, "720p", [dict()])
    finally:
        off(ctx)


def grid_wire(cells, res, origin, sec, nsec, frame_id):
    f = frame_id.encode()
    h, w = cells.shape
    return (struct.pack("<IIII", 0, sec, nsec, len(f)) + f + struct.pack("<IIfII", 0, 0, res, w, h) +
            struct.pack("<7d", origin[0], origin[1], 0, 0, 0, 0, 0) + struct.pack("<I", w * h) + cells.tobytes())


def test_node_publishes_projected_map(tmp_path):
    """The node mirror with map_enable: /projected_map carries the API's grid with the cloud's header, with the
    map_occupancy_* and map_min_*_size params; /point_cloud is node1map's; with the map off it is not advertised."""
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
              sensor_model_max=0.95, occupancy_thres=0.6, max_range=9.0, max_bricks=100000,
              occupancy_min_z=-0.5, occupancy_max_z=2.0, min_x_size=12.0, min_y_size=4.0)
    fid = "/map"
    params = dict(transform_enable=1, transform_target_frame=fid, map_enable=1,
                  **{f"transform_{k}": v for k, v in NODE_POSE.items()}, **{f"map_{k}": v for k, v in mp.items()})
    t = transform_of((NODE_POSE["roll"], NODE_POSE["pitch"], NODE_POSE["yaw"]),
                     (NODE_POSE["tx"], NODE_POSE["ty"], NODE_POSE["tz"]))
    with d2pc.Context() as ctx:
        ctx.set_transform(t)
        ctx.set_occupancy(resolution=0.1, prob_hit=0.75, prob_miss=0.35, clamp_min=0.15, clamp_max=0.95,
                          occupancy_thres=0.6, max_range=9.0, max_bricks=100000)
        for img in imgs:
            ctx.process_mono8(img)
        api = ctx.occupancy_projected_map(occupancy_min_z=-0.5, occupancy_max_z=2.0, min_x_size=12.0, min_y_size=4.0)
    assert api[0].size > 1000 and (api[0] == 100).any()
    sec = 3 + len(imgs) - 1
    launch = _node_launch(tmp_path, "on", params)
    out = {k: tmp_path / f"{k}.bin" for k in ("c", "g", "n", "c1", "m1")}
    r = subprocess.run([harness, "node1projmap", str(launch), "752", "480", str(out["c"]), str(out["g"]),
                        str(out["n"])] + [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["g"].read_bytes() == grid_wire(api[0], api[1], api[2], sec, 4, fid)
    assert out["n"].read_text().strip() == str(len(imgs))
    r = subprocess.run([harness, "node1map", str(launch), "752", "480", str(out["c1"]), str(out["m1"])] +
                       [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["c"].read_bytes() == out["c1"].read_bytes() and len(out["c"].read_bytes()) > 0
    # map off: /projected_map is not advertised (the harness checks), the cloud is the same
    off_launch = _node_launch(tmp_path, "off", {k: v for k, v in params.items() if k != "map_enable"})
    r = subprocess.run([harness, "node1projmap", str(off_launch), "752", "480", str(out["c1"]), str(out["g"]),
                        str(out["n"])] + [str(p) for p in raws], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out["g"].read_bytes() == b"" and out["n"].read_text().strip() == "0"
    assert out["c1"].read_bytes() == out["c"].read_bytes()
