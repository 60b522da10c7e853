"""GPU: D2PC_FILTER_VOXEL (pcl::VoxelGrid on the CROP cloud) byte for byte against the CPU reference
tests/voxel_ref, through every entry point whose output depends on the filter mode.

The reference is applied to the CROP cloud: the oracle's where the arithmetic is EXACT, the library's own CROP bytes
where it is FAST (the voxel stage consumes whatever the crop produced; the CROP bytes are pinned elsewhere).
D2PC_VOXEL_FUZZ_CASES / D2PC_VOXEL_FUZZ_SEED set the differential fuzz (default 150 cases)."""
import os
import subprocess

import numpy as np
import pytest

import oracle
import voxel_ref
from conftest import ROOT
from disparity_to_point_cloud_b200 import synth
from test_gpu_fuzz import _draw_f32, _draw_q, _draw_u8

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_VOXEL_FUZZ_CASES", "150"))
SEED0 = int(os.environ.get("D2PC_VOXEL_FUZZ_SEED", "31000"))
BUFFER_TOO_SMALL, INVALID_ARG = -9, -1


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


def crop_of(frame, q):
    return oracle.disparity_cb_mono8(frame, q) if frame.dtype == np.uint8 else oracle.disparity_cb_f32(frame, q)


def voxel(ctx, d2pc, leaf, min_points=0, limit=None):
    ctx.set_voxel_grid(leaf, min_points, limit)
    ctx.set_filter_mode(d2pc.FILTER_VOXEL)


def check(got, want, what, cloud=None):
    data, dense = want
    assert got.size == len(data), (what, got.size // 16, len(data) // 16)
    if got.tobytes() != data:
        g, o = np.frombuffer(got.tobytes(), np.uint32), np.frombuffer(data, np.uint32)
        bad = np.nonzero(g != o)[0]
        raise AssertionError(f"{what}: {bad.size} words differ, first at word {bad[0]}: {g[bad[0]]:#x} vs {o[bad[0]]:#x}")
    if cloud is not None:
        assert (cloud.is_dense, cloud.width, cloud.row_step, cloud.height) == (dense, len(data) // 16, len(data), 1), what


def run_entry(d2pc, ctx, pin, reg, frame, entry, cap_bytes=None):
    """One frame through one entry; returns the cloud bytes (and the d2pc_cloud where there is one)."""
    if entry == "library":
        got = ctx.process_mono8(frame) if frame.dtype == np.uint8 else ctx.process_f32(frame)
        return got, ctx.last_cloud
    if entry == "slot":
        ctx.submit(1, frame)
        return ctx.wait(1), ctx.last_cloud
    if entry == "slot_into":
        dst = pin.array[: cap_bytes]
        ctx.submit(2, frame, dst)
        return ctx.wait(2), ctx.last_cloud
    dst = {"pinned": pin.array, "registered": reg.array, "pageable": np.empty(cap_bytes, np.uint8)}[entry][:cap_bytes]
    return ctx.process_into(frame, dst), ctx.last_cloud


ENTRIES = ["library", "pinned", "registered", "pageable", "slot", "slot_into"]


@pytest.mark.parametrize("h,w", [(480, 640), (480, 752), (720, 1280)])
@pytest.mark.parametrize("leaf,limit", [(0.05, None), (0.2, None), (0.05, ("z", 0.0, 10.0)), (0.2, ("z", 0.0, 10.0))])
def test_every_host_entry_matches_the_reference(env, h, w, leaf, limit):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    voxel(ctx, d2pc, leaf, 0, limit)
    try:
        for frame in (synth.s2_scene(h, w, 3), synth.s3_float(h, w, 4)):
            want = voxel_ref.voxel_grid(crop_of(frame, q), leaf, 0, limit)
            for entry in ENTRIES:
                got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, max(len(want[0]), 16) + 64)
                check(got, want, (entry, frame.dtype, h, w, leaf, limit), cl)
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)


def test_too_small_destination_is_reported_at_wait(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 5)
    want = voxel_ref.voxel_grid(crop_of(frame, q), 0.05)
    n = len(want[0])
    assert n > 32
    voxel(ctx, d2pc, 0.05)
    try:
        for dst in (pin.array[: n - 16], np.empty(n - 16, np.uint8)):
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.process_into(frame, dst)
            assert e.value.status == BUFFER_TOO_SMALL
            ctx.submit(0, frame, dst)
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.wait(0)
            assert e.value.status == BUFFER_TOO_SMALL
        # an exact fit is enough
        check(ctx.process_into(frame, pin.array[:n]), want, "exact fit", ctx.last_cloud)
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)


def test_4k_frame(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(2160, 3840, 6)
    crop = crop_of(frame, q)
    voxel(ctx, d2pc, 0.2, 0, ("z", 0.0, 10.0))
    try:
        want = voxel_ref.voxel_grid(crop, 0.2, 0, ("z", 0.0, 10.0))
        for entry in ("library", "pinned", "slot"):
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(want[0]) + 64)
            check(got, want, ("4k", entry), cl)
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)


@pytest.mark.parametrize("leaf", [0.01, 0.05, 0.5, 2.0, 10.0])
def test_leaf_sizes_including_the_overflow_fallback(env, leaf):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    seen_dense = set()
    voxel(ctx, d2pc, leaf)
    try:
        for frame in (synth.s2_scene(480, 752, 7), synth.s3_float(480, 752, 8)):
            want = voxel_ref.voxel_grid(crop_of(frame, q), leaf)
            seen_dense.add(want[1])
            for entry in ("library", "pageable", "slot"):
                got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, max(len(want[0]), 16) + 64)
                check(got, want, (entry, leaf), cl)
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)
    if leaf == 0.01:
        assert 0 in seen_dense  # 1 cm over the whole scene without a limit overflows PCL's int index


def test_generic_q_and_fast_arithmetic(env):
    d2pc, ctx, pin, reg = env
    rng = np.random.default_rng(5)
    q = rng.normal(0, 1, (4, 4))
    q[3, 2] = 3.0
    q0 = ctx.get_q()
    frame = synth.s3_float(480, 640, 9)
    try:
        ctx.set_q(q)
        voxel(ctx, d2pc, 0.5)
        check(ctx.process_f32(frame), voxel_ref.voxel_grid(crop_of(frame, q), 0.5), "generic Q", ctx.last_cloud)
        ctx.set_q(q0)
        ctx.set_arith_mode(d2pc.ARITH_FAST)
        for f in (frame, synth.s2_scene(480, 752, 10)):
            ctx.set_filter_mode(d2pc.FILTER_CROP)
            crop = ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)
            ctx.set_filter_mode(d2pc.FILTER_VOXEL)
            got = ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)
            check(got, voxel_ref.voxel_grid(crop, 0.5), ("FAST", f.dtype), ctx.last_cloud)
    finally:
        ctx.set_arith_mode(d2pc.ARITH_EXACT)
        ctx.set_q(q0)
        ctx.set_filter_mode(d2pc.FILTER_CROP)


def test_stream(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = np.stack([synth.s2_scene(480, 752, 20 + i) for i in range(5)])
    voxel(ctx, d2pc, 0.1, 2, ("z", 0.0, 10.0))
    try:
        got = ctx.process_stream(frames, n_frames=7)
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)
    for i, g in enumerate(got):
        check(g, voxel_ref.voxel_grid(crop_of(frames[i % 5], q), 0.1, 2, ("z", 0.0, 10.0)), ("stream", i))


@pytest.mark.parametrize("mono", [True, False])
def test_device_batch_per_frame_counts(env, mono):
    import torch
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    h, w, nf = 480, 752, 4
    frames = np.stack([synth.s2_scene(h, w, 30 + i) for i in range(nf)])
    if not mono:
        frames = frames.astype(np.float32) * np.float32(0.125)
        frames[3] = synth.s3_float(h, w, 33)
    frames[2] = 0  # a frame with no finite point: the empty cloud
    n = oracle.n_points(w, h)
    stride = n * 16 + 256
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.zeros(nf * stride, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
    grid = (0.1, 0, ("z", 0.0, 10.0))  # the float entry has no median: its salt noise reaches 500 m without a limit
    voxel(ctx, d2pc, *grid)
    try:
        step = w * frames.itemsize
        fn = ctx.reproject_mono8_device if mono else ctx.reproject_f32_device
        with pytest.raises(d2pc.D2pcError):
            fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, 0)  # counts are required
        fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, d_cnt.data_ptr())
        ctx.sync()
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)
    counts = d_cnt.cpu().numpy()
    pts = d_pts.cpu().numpy()
    wants = [voxel_ref.voxel_grid(crop_of(frames[f], q), *grid) for f in range(nf)]
    assert len({len(wv[0]) for wv in wants}) > 2 and counts[2] == 0
    for f in range(nf):
        assert counts[f] * 16 == len(wants[f][0]), f
        check(pts[f * stride: f * stride + counts[f] * 16], wants[f], ("batch", f))


def test_fusion_entries(env):
    """fuse_then_process, submit_fusion and the fusion stream on 4 x 1280x720: the VOXEL cloud is the reference
    applied to the CROP cloud of the same set."""
    d2pc, _, _, _ = env
    h, w = 720, 1280
    sets = np.stack([np.stack([synth.s2_scene(h, w, 40 + 4 * s + i) for i in range(4)]) for s in range(3)])
    with d2pc.Context(offset_x=-7, offset_y=15, n_slots=2) as ctx:
        crops_fused = [ctx.fuse_then_process(*sets[s]) for s in range(3)]
        of = oracle.fuse(*sets[0], -7, 15)[0]
        assert crops_fused[0].tobytes() == oracle.disparity_cb_mono8(of, ctx.get_q()).tobytes()
        crops_pipe = ctx.process_fusion_stream(sets)
        ctx.set_voxel_grid(0.1, 0, ("z", 0.0, 10.0))
        ctx.set_filter_mode(d2pc.FILTER_VOXEL)
        for s in range(3):
            want = voxel_ref.voxel_grid(crops_fused[s], 0.1, 0, ("z", 0.0, 10.0))
            check(ctx.fuse_then_process(*sets[s]), want, ("fuse_then_process", s), ctx.last_cloud)
        for s in range(3):
            ctx.submit_fusion(s % 2, *sets[s])
            check(ctx.wait(s % 2), voxel_ref.voxel_grid(crops_pipe[s], 0.1, 0, ("z", 0.0, 10.0)), ("submit_fusion", s),
                  ctx.last_cloud)
        for s, g in enumerate(ctx.process_fusion_stream(sets, n_sets=5)):
            check(g, voxel_ref.voxel_grid(crops_pipe[s % 3], 0.1, 0, ("z", 0.0, 10.0)), ("fusion stream", s))


def test_switching_back_to_crop_and_argument_checks(env):
    d2pc, _, _, _ = env
    frame = synth.s2_scene(480, 752, 50)
    with d2pc.Context() as ctx:
        q = ctx.get_q()
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.set_filter_mode(d2pc.FILTER_VOXEL)  # no grid yet
        assert e.value.status == INVALID_ARG
        assert ctx.get_voxel_grid().leaf_x == 0 and ctx.get_voxel_grid().limit_field == -1
        for bad in [dict(leaf=0.0), dict(leaf=-1.0), dict(leaf=float("inf")), dict(leaf=float("nan")),
                    dict(leaf=0.1, limit=("z", 2.0, 1.0))]:
            with pytest.raises(d2pc.D2pcError):
                ctx.set_voxel_grid(**bad)
        with pytest.raises(d2pc.D2pcError):
            ctx.set_filter_mode(7)
        crop = ctx.process_mono8(frame)
        assert crop.tobytes() == oracle.disparity_cb_mono8(frame, q).tobytes()
        ctx.set_voxel_grid((0.1, 0.2, 0.3), 3, ("y", -1.0, 1.0))
        g = ctx.get_voxel_grid()
        assert (g.leaf_x, g.leaf_y, g.leaf_z, g.min_points_per_voxel, g.limit_field, g.limit_min, g.limit_max) == (
            np.float32(0.1), np.float32(0.2), np.float32(0.3), 3, 1, -1.0, 1.0)
        ctx.set_filter_mode(d2pc.FILTER_VOXEL)
        check(ctx.process_mono8(frame), voxel_ref.voxel_grid(crop, (0.1, 0.2, 0.3), 3, ("y", -1.0, 1.0)), "aniso",
              ctx.last_cloud)
        ctx.set_filter_mode(d2pc.FILTER_CROP)
        assert ctx.process_mono8(frame).tobytes() == crop.tobytes()
        assert ctx.last_cloud.is_dense == 0


def test_node1_voxel_params_through_the_launch_file(tmp_path):
    from disparity_to_point_cloud_b200 import build
    build.build()
    harness = build.build_harness()
    q = oracle.q_from_intrinsics()
    launch = tmp_path / "voxel.launch"
    launch.write_text('<launch>\n  <node name="disparity_to_point_cloud" pkg="disparity_to_point_cloud" '
                      'type="disparity_to_point_cloud_node">\n'
                      '    <remap from="/disparity" to="/throttled_depth_map"/>\n'
                      '    <param name="voxel_leaf_size" value="0.1"/>\n'
                      '    <param name="voxel_z_min" value="0.5"/>\n'
                      '    <param name="voxel_z_max" value="8"/>\n  </node>\n</launch>\n')
    img = synth.s2_scene(480, 752, 51)
    raw, out = tmp_path / "in.raw", tmp_path / "cloud.bin"
    raw.write_bytes(img.tobytes())
    subprocess.run([harness, "node1", str(launch), "752", "480", str(raw), str(out), "1700000000", "250"], check=True)
    data, dense = voxel_ref.voxel_grid(oracle.disparity_cb_mono8(img, q), 0.1, 0, ("z", 0.5, 8.0))
    want = oracle.serialize_pointcloud2(np.frombuffer(data, np.uint8), seq=0, sec=1700000000, nsec=250, is_dense=dense)
    assert out.read_bytes() == want


def _fuzz_case(case, env):
    d2pc, ctx, pin, reg = env
    rng = np.random.default_rng(SEED0 + case)
    w = int(rng.integers(81, 900)) if rng.random() < 0.9 else int(rng.integers(1, 90))
    h = int(rng.integers(81, 600)) if rng.random() < 0.9 else int(rng.integers(1, 90))
    mono = bool(rng.random() < 0.5)
    qkind, q = _draw_q(rng, d2pc)
    frame = _draw_u8(rng, h, w) if mono else _draw_f32(rng, h, w)
    leaf = float(rng.choice([0.01, 0.03, 0.1, 0.3, 1.0, 5.0, 10.0]))
    if rng.random() < 0.2:
        leaf = tuple(float(v) for v in rng.choice([0.02, 0.1, 0.5, 2.0], 3))
    limit = None
    if rng.random() < 0.5:
        lo = float(rng.choice([-5.0, 0.0, 0.5, 2.0]))
        limit = (str(rng.choice(list("xyz"))), lo, lo + float(rng.choice([0.0, 1.0, 10.0, 100.0])))
    mp = int(rng.choice([0, 0, 1, 2, 3, 10]))
    entry = str(rng.choice(ENTRIES + ["batch"]))
    desc = dict(case=case, w=w, h=h, mono=mono, q=qkind, leaf=leaf, limit=limit, mp=mp, entry=entry)
    ctx.set_q(q)
    crop = crop_of(frame, q)
    want = voxel_ref.voxel_grid(crop, leaf, mp, limit)
    ctx.set_voxel_grid(leaf, mp, limit)
    ctx.set_filter_mode(d2pc.FILTER_VOXEL)
    try:
        if entry == "batch":
            import torch
            frames = np.stack([frame, _draw_u8(rng, h, w) if mono else _draw_f32(rng, h, w)])
            n = oracle.n_points(w, h)
            stride = max(16, n * 16)
            d_in = torch.from_numpy(frames).cuda()
            d_pts = torch.zeros(2 * stride, dtype=torch.uint8, device="cuda")
            d_cnt = torch.zeros(2, dtype=torch.int32, device="cuda")
            step = w * frames.itemsize
            fn = ctx.reproject_mono8_device if mono else ctx.reproject_f32_device
            fn(d_in.data_ptr(), 2, w, h, step, step * h, d_pts.data_ptr(), stride, d_cnt.data_ptr())
            ctx.sync()
            cnt, pts = d_cnt.cpu().numpy(), d_pts.cpu().numpy()
            for f in range(2):
                wf = want if f == 0 else voxel_ref.voxel_grid(crop_of(frames[1], q), leaf, mp, limit)
                check(pts[f * stride: f * stride + cnt[f] * 16], wf, (desc, f))
        else:
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, max(len(want[0]), 16) + 64)
            check(got, want, desc, cl)
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)
    return desc, want[1]


def test_voxel_fuzz_against_reference(env):
    seen, fallbacks = set(), 0
    try:
        for case in range(N_FUZZ):
            d, dense = _fuzz_case(case, env)
            seen.add((d["mono"], d["entry"]))
            fallbacks += dense == 0
    finally:
        env[1].set_q(oracle.q_from_intrinsics())
    if N_FUZZ >= 100:
        assert len(seen) >= 12 and fallbacks > 0, (seen, fallbacks)
    print(f"voxel fuzz: {N_FUZZ} cases from seed {SEED0}, {len(seen)} (entry, kind) classes, {fallbacks} fallbacks")
