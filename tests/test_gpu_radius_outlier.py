"""GPU: the radius outlier stage (pcl::RadiusOutlierRemoval behind the filter mode) byte for byte against the CPU
reference tests/outlier_ref, through every entry point whose output depends on the filter mode, and
d2pc_radius_outlier_device on hand-built clouds.

The reference is applied to the cloud the mode publishes: the CROP cloud of the oracle where the arithmetic is
EXACT, the library's own where it is FAST; CROP_FINITE's is the CROP cloud without its non-finite points (the stage
drops those anyway, so the reference runs on the CROP cloud); VOXEL's is tests/voxel_ref applied to the CROP cloud.
D2PC_ROR_FUZZ_CASES / D2PC_ROR_FUZZ_SEED set the differential fuzz (default 150 cases)."""
import os
import subprocess

import numpy as np
import pytest

import oracle
import outlier_ref
import voxel_ref
from disparity_to_point_cloud_b200 import synth
from test_gpu_fuzz import _draw_f32, _draw_q, _draw_u8
from test_gpu_voxel import ENTRIES, check, crop_of, run_entry

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_ROR_FUZZ_CASES", "150"))
SEED0 = int(os.environ.get("D2PC_ROR_FUZZ_SEED", "47000"))
BUFFER_TOO_SMALL, INVALID_ARG, BAD_DIMS = -9, -1, -3
MODES = ["crop", "finite", "voxel"]
VOXEL_GRID = (0.05, 0, ("z", 0.0, 10.0))


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


def set_mode(d2pc, ctx, mode, grid=VOXEL_GRID):
    if mode == "voxel":
        ctx.set_voxel_grid(*grid)
    ctx.set_filter_mode({"crop": d2pc.FILTER_CROP, "finite": d2pc.FILTER_CROP_FINITE, "voxel": d2pc.FILTER_VOXEL}[mode])


def mode_cloud(crop, mode, grid=VOXEL_GRID):
    """The cloud the mode publishes (for CROP_FINITE: the CROP cloud, whose non-finite points the stage drops)."""
    return voxel_ref.voxel_grid(crop, *grid)[0] if mode == "voxel" else crop


def want(crop, mode, radius, mn, grid=VOXEL_GRID):
    return outlier_ref.radius_outlier(np.frombuffer(mode_cloud(crop, mode, grid), np.uint8), radius, mn), 1


def reset(d2pc, ctx):
    ctx.set_radius_outlier(0.0)
    ctx.set_filter_mode(d2pc.FILTER_CROP)


@pytest.mark.parametrize("h,w", [(480, 640), (480, 752), (720, 1280)])
@pytest.mark.parametrize("mode", MODES)
def test_every_host_entry_matches_the_reference(env, h, w, mode):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    radius, mn = (0.1, 2) if mode == "voxel" else (0.05, 5)
    set_mode(d2pc, ctx, mode)
    ctx.set_radius_outlier(radius, mn)
    try:
        for frame in (synth.s2_scene(h, w, 3), synth.s3_float(h, w, 4)):
            wv = want(crop_of(frame, q), mode, radius, mn)
            assert 0 < len(wv[0])
            for entry in ENTRIES:
                got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                check(got, wv, (entry, frame.dtype, h, w, mode), cl)
    finally:
        reset(d2pc, ctx)


def test_crop_and_crop_finite_give_the_same_bytes(env):
    d2pc, ctx, pin, reg = env
    frames = (synth.s2_scene(480, 752, 11), synth.s3_float(480, 752, 12))
    try:
        for radius, mn in [(0.02, 1), (0.05, 3), (0.2, 10)]:
            ctx.set_radius_outlier(radius, mn)
            for f in frames:
                ctx.set_filter_mode(d2pc.FILTER_CROP)
                a = ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)
                ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
                b = ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)
                assert a.tobytes() == b.tobytes() and ctx.last_cloud.is_dense == 1, (radius, mn, f.dtype)
    finally:
        reset(d2pc, ctx)


def test_too_small_destination_is_reported_at_wait(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 5)
    wv = want(crop_of(frame, q), "crop", 0.05, 2)
    n = len(wv[0])
    assert n > 32
    ctx.set_radius_outlier(0.05, 2)
    try:
        for dst in (pin.array[: n - 16], np.empty(n - 16, np.uint8)):
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.process_into(frame, dst)
            assert e.value.status == BUFFER_TOO_SMALL
            ctx.submit(0, frame, dst)
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.wait(0)
            assert e.value.status == BUFFER_TOO_SMALL
        check(ctx.process_into(frame, pin.array[:n]), wv, "exact fit", ctx.last_cloud)
    finally:
        reset(d2pc, ctx)


def test_4k_frame(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(2160, 3840, 6)
    crop = crop_of(frame, q)
    try:
        for mode, radius, mn in [("crop", 0.05, 5), ("voxel", 0.1, 2)]:
            set_mode(d2pc, ctx, mode)
            ctx.set_radius_outlier(radius, mn)
            wv = want(crop, mode, radius, mn)
            for entry in ("library", "pinned", "slot"):
                got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                check(got, wv, ("4k", mode, entry), cl)
    finally:
        reset(d2pc, ctx)


def test_generic_q_and_fast_arithmetic(env):
    d2pc, ctx, pin, reg = env
    rng = np.random.default_rng(5)
    q = rng.normal(0, 1, (4, 4))
    q[3, 2] = 3.0
    q0 = ctx.get_q()
    frame = synth.s3_float(480, 640, 9)
    try:
        ctx.set_q(q)
        ctx.set_radius_outlier(0.5, 3)
        check(ctx.process_f32(frame), want(crop_of(frame, q), "crop", 0.5, 3), "generic Q", ctx.last_cloud)
        ctx.set_q(q0)
        ctx.set_arith_mode(d2pc.ARITH_FAST)
        for f in (frame, synth.s2_scene(480, 752, 10)):
            ctx.set_radius_outlier(0.0)
            crop = ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)
            ctx.set_radius_outlier(0.05, 3)
            got = ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)
            check(got, want(crop, "crop", 0.05, 3), ("FAST", f.dtype), ctx.last_cloud)
    finally:
        ctx.set_arith_mode(d2pc.ARITH_EXACT)
        ctx.set_q(q0)
        reset(d2pc, ctx)


@pytest.mark.parametrize("mode", MODES)
def test_stream(env, mode):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = np.stack([synth.s2_scene(480, 752, 20 + i) for i in range(5)])
    set_mode(d2pc, ctx, mode)
    ctx.set_radius_outlier(0.1, 2)
    try:
        got = ctx.process_stream(frames, n_frames=7)
    finally:
        reset(d2pc, ctx)
    for i, g in enumerate(got):
        check(g, want(crop_of(frames[i % 5], q), mode, 0.1, 2), ("stream", mode, i))


@pytest.mark.parametrize("mono", [True, False])
@pytest.mark.parametrize("mode", MODES)
def test_device_batch_per_frame_counts(env, mono, mode):
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
    radius, mn = 0.1, 3
    set_mode(d2pc, ctx, mode)
    ctx.set_radius_outlier(radius, mn)
    try:
        step = w * frames.itemsize
        fn = ctx.reproject_mono8_device if mono else ctx.reproject_f32_device
        with pytest.raises(d2pc.D2pcError) as e:
            fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, 0)  # counts are required
        assert e.value.status == INVALID_ARG
        fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, d_cnt.data_ptr())
        ctx.sync()
    finally:
        reset(d2pc, ctx)
    counts = d_cnt.cpu().numpy()
    pts = d_pts.cpu().numpy()
    wants = [want(crop_of(frames[f], q), mode, radius, mn) for f in range(nf)]
    assert counts[2] == 0 and len(wants[0][0]) > 0
    for f in range(nf):
        assert counts[f] * 16 == len(wants[f][0]), f
        check(pts[f * stride: f * stride + counts[f] * 16], wants[f], ("batch", mode, f))


def test_fusion_entries(env):
    """fuse_then_process, submit_fusion and the fusion stream on 4 x 1280x720: the stage applied to the CROP cloud
    of the same set."""
    d2pc, _, _, _ = env
    h, w = 720, 1280
    sets = np.stack([np.stack([synth.s2_scene(h, w, 40 + 4 * s + i) for i in range(4)]) for s in range(3)])
    with d2pc.Context(offset_x=-7, offset_y=15, n_slots=2) as ctx:
        crops_fused = [ctx.fuse_then_process(*sets[s]) for s in range(3)]
        crops_pipe = ctx.process_fusion_stream(sets)
        for mode in ("crop", "finite", "voxel"):
            set_mode(d2pc, ctx, mode, (0.1, 0, ("z", 0.0, 10.0)))
            ctx.set_radius_outlier(0.15, 2)
            wf = [want(c, mode, 0.15, 2, (0.1, 0, ("z", 0.0, 10.0))) for c in crops_fused]
            wp = [want(c, mode, 0.15, 2, (0.1, 0, ("z", 0.0, 10.0))) for c in crops_pipe]
            for s in range(3):
                check(ctx.fuse_then_process(*sets[s]), wf[s], ("fuse_then_process", mode, s), ctx.last_cloud)
            for s in range(3):
                ctx.submit_fusion(s % 2, *sets[s])
                check(ctx.wait(s % 2), wp[s], ("submit_fusion", mode, s), ctx.last_cloud)
            for s, g in enumerate(ctx.process_fusion_stream(sets, n_sets=5)):
                check(g, wp[s % 3], ("fusion stream", mode, s))


def cloud_of(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    pts = np.zeros((len(xyz), 4), np.float32)
    pts[:, :3] = xyz
    pts[:, 3] = np.arange(len(xyz), dtype=np.float32)  # the pad word travels unchanged
    return pts


def adversarial_clouds(rng):
    """(name, cloud, radius, min_neighbors): boundary pairs across cell edges, duplicates, non-finite points,
    coarsening spans, empty frames."""
    out = []
    r = 0.25
    base = np.array([-3.0, -7.0, -1.0], np.float32)
    edge = [base, base - np.float32([r, 0, 0]), base + np.float32([0, r, 0]), base - np.float32([0, 0, r])]
    far = np.nextafter(np.float32(r), np.float32(1))
    edge += [base + np.float32([5, 0, 0]), base + np.float32([5, 0, 0]) + np.float32([far, 0, 0])]
    out.append(("boundary pairs", cloud_of(edge), r, 1))
    grid = rng.integers(-40, 40, (3000, 3)).astype(np.float32) * np.float32(r)  # every pair on a cell edge
    out.append(("lattice at the radius", cloud_of(grid), r, 2))
    dup = rng.uniform(-1, 1, (50, 3))
    out.append(("duplicates", cloud_of(dup[rng.integers(0, 50, 4000)]), 1e-7, 3))
    pts = cloud_of(rng.normal(0, 1, (5000, 3)))
    k = 700
    pts[rng.integers(0, 5000, k), rng.integers(0, 3, k)] = rng.choice([np.nan, np.inf, -np.inf], k)
    out.append(("non-finite", pts, 0.1, 2))
    span = cloud_of(np.concatenate([rng.normal(0, 0.05, (2000, 3)), [[1e30, 0, 0], [1e30, 0, 0], [-3e38, 3e38, 0]]]))
    out.append(("1e30 span", span, 0.02, 1))
    out.append(("huge radius", cloud_of(rng.uniform(-1e3, 1e3, (3000, 3))), 1e200, 2999))
    out.append(("tiny radius", cloud_of(np.concatenate([np.zeros((3, 3)), [[1e-30, 0, 0], [1e-20, 0, 0]]])), 1e-40, 2))
    out.append(("empty", cloud_of(np.empty((0, 3))), 0.1, 1))
    out.append(("all non-finite", cloud_of(np.full((100, 3), np.nan)), 0.1, 0))
    out.append(("min 0", pts, 0.01, 0))
    out.append(("min above n", cloud_of(np.zeros((64, 3))), 1.0, 64))
    return out


def test_device_entry_on_adversarial_clouds(env):
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(77)
    cases = adversarial_clouds(rng)
    try:
        for name, pts, radius, mn in cases:  # one frame each
            ctx.set_radius_outlier(radius, mn)
            n = max(len(pts), 1)
            d_in = torch.from_numpy(np.ascontiguousarray(pts).view(np.uint8).reshape(-1)).cuda() if len(pts) else \
                torch.zeros(16, dtype=torch.uint8, device="cuda")
            d_out = torch.zeros(n * 16, dtype=torch.uint8, device="cuda")
            d_cnt = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
            ctx.radius_outlier_device(d_in.data_ptr(), 1, len(pts), n * 16, 0, d_out.data_ptr(), n * 16,
                                      d_cnt.data_ptr())
            ctx.sync()
            c = int(d_cnt.cpu()[0])
            wv = outlier_ref.radius_outlier(pts, radius, mn)
            assert wv == outlier_ref.radius_outlier(pts, radius, mn, "brute") or len(pts) > 3500
            check(d_out.cpu().numpy()[: c * 16], (wv, 1), name)
        # several frames with per-frame counts (positions past the count hold garbage that must not be read)
        n_max, nf = 5200, len(cases)
        stride = n_max * 16 + 64
        host = np.full(nf * stride // 4, np.nan, np.float32)
        host.view(np.uint32)[1::7] = 0x7f800001  # signalling-NaN garbage past the counts
        counts = np.zeros(nf, np.uint32)
        for f, (_, pts, _, _) in enumerate(cases):
            m = min(len(pts), n_max)
            host.view(np.uint8)[f * stride: f * stride + m * 16] = pts[:m].view(np.uint8).reshape(-1)
            counts[f] = m
        counts[-1] = n_max * 3  # above n_max counts as n_max
        radius, mn = 0.05, 2
        ctx.set_radius_outlier(radius, mn)
        d_in = torch.from_numpy(host.view(np.uint8)).cuda()
        d_cnt_in = torch.from_numpy(counts.view(np.int32)).cuda()
        d_out = torch.zeros(nf * stride, dtype=torch.uint8, device="cuda")
        d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
        ctx.radius_outlier_device(d_in.data_ptr(), nf, n_max, stride, d_cnt_in.data_ptr(), d_out.data_ptr(), stride,
                                  d_cnt.data_ptr())
        ctx.sync()
        got_c, got = d_cnt.cpu().numpy(), d_out.cpu().numpy()
        for f in range(nf):
            m = min(int(counts[f]), n_max)
            frame = host.view(np.uint8)[f * stride: f * stride + m * 16]
            wv = outlier_ref.radius_outlier(frame, radius, mn)
            check(got[f * stride: f * stride + got_c[f] * 16], (wv, 1), ("batch", cases[f][0] if f < nf - 1 else f))
        # argument checks
        with pytest.raises(d2pc.D2pcError) as e:  # counts out are required
            ctx.radius_outlier_device(d_in.data_ptr(), nf, n_max, stride, 0, d_out.data_ptr(), stride, 0)
        assert e.value.status == INVALID_ARG
        with pytest.raises(d2pc.D2pcError) as e:  # input and output overlap
            ctx.radius_outlier_device(d_in.data_ptr(), 2, n_max, stride, 0, d_in.data_ptr() + stride, stride,
                                      d_cnt.data_ptr())
        assert e.value.status == INVALID_ARG
        with pytest.raises(d2pc.D2pcError) as e:  # stride below a frame
            ctx.radius_outlier_device(d_in.data_ptr(), 2, n_max, n_max * 8, 0, d_out.data_ptr(), stride,
                                      d_cnt.data_ptr())
        assert e.value.status == BAD_DIMS
        with pytest.raises(d2pc.D2pcError) as e:  # misaligned
            ctx.radius_outlier_device(d_in.data_ptr() + 4, 1, 10, stride, 0, d_out.data_ptr(), stride,
                                      d_cnt.data_ptr())
        assert e.value.status == BAD_DIMS
        ctx.set_radius_outlier(0.0)
        with pytest.raises(d2pc.D2pcError) as e:  # the stage is off
            ctx.radius_outlier_device(d_in.data_ptr(), 1, 10, stride, 0, d_out.data_ptr(), stride, d_cnt.data_ptr())
        assert e.value.status == INVALID_ARG
    finally:
        reset(d2pc, ctx)


def test_voxel_overflow_fallback_feeds_the_crop_cloud_to_the_stage(env):
    """A VOXEL frame that takes the overflow fallback publishes its CROP cloud (+-inf points, is_dense 0); behind the
    stage it is that cloud filtered, is_dense 1 -- the same bytes as CROP + stage."""
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s3_float(480, 752, 8)  # uniform disparities: hundreds of metres, no limit -> PCL's int overflow
    crop = crop_of(frame, q)
    grid = (0.05, 0, None)
    assert voxel_ref.voxel_grid(crop, *grid)[1] == 0
    wv = want(crop, "voxel", 0.5, 2, grid)
    assert wv[0] == want(crop, "crop", 0.5, 2)[0] and 0 < len(wv[0]) < len(crop)
    try:
        set_mode(d2pc, ctx, "voxel", grid)
        ctx.set_radius_outlier(0.0)
        ctx.process_f32(frame)
        assert ctx.last_cloud.is_dense == 0  # the fallback really is taken
        ctx.set_radius_outlier(0.5, 2)
        for entry in ("library", "pinned", "slot"):
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
            check(got, wv, ("fallback", entry), cl)
    finally:
        reset(d2pc, ctx)


def test_device_entry_with_more_than_65535_frames(env):
    """70 000 clouds of at most 3 points in one call: the frame count has no launch-geometry limit."""
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(78)
    nf, n_max, radius, mn = 70000, 3, 0.2, 1
    pts = np.full((nf, n_max, 4), np.nan, np.float32)
    pts[..., :3] = rng.uniform(0, 0.3, (nf, n_max, 3)).astype(np.float32)
    pts[..., 3] = 1.0
    pts[rng.random((nf, n_max)) < 0.1, int(rng.integers(0, 3))] = np.inf
    counts = rng.integers(0, n_max + 2, nf).astype(np.uint32)  # n_max + 1 counts as n_max
    # the rule, vectorised over frames: float32 distances, double compare, only finite points below the count
    valid = (np.arange(n_max)[None, :] < np.minimum(counts, n_max)[:, None]) & np.isfinite(pts[..., :3]).all(-1)
    with np.errstate(invalid="ignore", over="ignore"):  # inf - inf and overflows belong to dropped points
        d = pts[:, :, None, :3] - pts[:, None, :, :3]
        s = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    keep = valid & (((s.astype(np.float64) <= radius * radius) & valid[:, None, :]).sum(-1) >= mn + 1)
    want_cnt = keep.sum(1)
    assert 0 < want_cnt.sum() < valid.sum()
    d_in = torch.from_numpy(pts.reshape(-1).view(np.uint8).copy()).cuda()
    d_cnt_in = torch.from_numpy(counts.view(np.int32)).cuda()
    d_out = torch.zeros(nf * n_max * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.full((nf,), -1, dtype=torch.int32, device="cuda")
    try:
        ctx.set_radius_outlier(radius, mn)
        ctx.radius_outlier_device(d_in.data_ptr(), nf, n_max, n_max * 16, d_cnt_in.data_ptr(), d_out.data_ptr(),
                                  n_max * 16, d_cnt.data_ptr())
        ctx.sync()
    finally:
        reset(d2pc, ctx)
    got_cnt = d_cnt.cpu().numpy()
    np.testing.assert_array_equal(got_cnt, want_cnt)
    got = d_out.cpu().numpy().view(np.uint32).reshape(nf, n_max, 4)
    order = np.argsort(~keep, axis=1, kind="stable")  # kept points first, in input order
    want_pts = np.take_along_axis(pts.view(np.uint32), order[..., None], axis=1)
    head = np.arange(n_max)[None, :] < want_cnt[:, None]
    np.testing.assert_array_equal(got[head], want_pts[head])


def test_radius_zero_restores_crop_and_argument_checks(env):
    d2pc, _, _, _ = env
    frame = synth.s2_scene(480, 752, 50)
    with d2pc.Context() as ctx:
        q = ctx.get_q()
        p = ctx.get_radius_outlier()
        assert (p.radius, p.min_neighbors, p.struct_size) == (0.0, 1, 24)
        crop = ctx.process_mono8(frame)
        assert crop.tobytes() == oracle.disparity_cb_mono8(frame, q).tobytes() and ctx.last_cloud.is_dense == 0
        for bad in [-1.0, float("nan"), float("inf"), -float("inf")]:
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.set_radius_outlier(bad, 2)
            assert e.value.status == INVALID_ARG
        assert ctx.get_radius_outlier().radius == 0.0  # the previous setting is kept
        for bad in (-1, 2**32):
            with pytest.raises(ValueError):
                ctx.set_radius_outlier(0.05, bad)
        assert ctx.get_radius_outlier().radius == 0.0
        ctx.set_radius_outlier(0.05, 7)
        p = ctx.get_radius_outlier()
        assert (p.radius, p.min_neighbors) == (0.05, 7)
        check(ctx.process_mono8(frame), want(crop, "crop", 0.05, 7), "on", ctx.last_cloud)
        ctx.set_radius_outlier(0.0, 7)
        assert ctx.process_mono8(frame).tobytes() == crop.tobytes()
        assert ctx.last_cloud.is_dense == 0 and ctx.last_cloud.width == len(crop) // 16


def test_node1_radius_outlier_params_through_the_launch_file(tmp_path):
    from disparity_to_point_cloud_b200 import build
    build.build()
    harness = build.build_harness()
    q = oracle.q_from_intrinsics()
    launch = tmp_path / "ror.launch"
    launch.write_text('<launch>\n  <node name="disparity_to_point_cloud" pkg="disparity_to_point_cloud" '
                      'type="disparity_to_point_cloud_node">\n'
                      '    <remap from="/disparity" to="/throttled_depth_map"/>\n'
                      '    <param name="voxel_leaf_size" value="0.05"/>\n'
                      '    <param name="radius_outlier_radius" value="0.1"/>\n'
                      '    <param name="radius_outlier_min_neighbors" value="3"/>\n  </node>\n</launch>\n')
    img = synth.s2_scene(480, 752, 51)
    raw, out = tmp_path / "in.raw", tmp_path / "cloud.bin"
    raw.write_bytes(img.tobytes())
    subprocess.run([harness, "node1", str(launch), "752", "480", str(raw), str(out), "1700000000", "250"], check=True)
    data, _ = want(oracle.disparity_cb_mono8(img, q), "voxel", 0.1, 3, (0.05, 0, None))
    assert len(data) > 0
    wire = oracle.serialize_pointcloud2(np.frombuffer(data, np.uint8), seq=0, sec=1700000000, nsec=250, is_dense=1)
    assert out.read_bytes() == wire


def _radius_from_pairs(rng, cloud):
    """A radius equal to an actual pair distance of the cloud (rule 3), so the boundary is hit."""
    xyz = np.frombuffer(cloud, np.uint8).view(np.float32).reshape(-1, 4)[:, :3]
    xyz = xyz[np.isfinite(xyz).all(axis=1)]
    if len(xyz) < 2:
        return float(rng.choice([0.02, 0.1]))
    i = int(rng.integers(0, len(xyz)))
    d = xyz[i] - xyz[np.argsort(np.abs(xyz - xyz[i]).sum(axis=1))[int(rng.integers(1, min(len(xyz), 40)))]]
    s = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
    return float(np.sqrt(np.float64(s))) or float(rng.choice([0.02, 0.1]))


def _fuzz_case(case, env):
    d2pc, ctx, pin, reg = env
    rng = np.random.default_rng(SEED0 + case)
    w = int(rng.integers(81, 900)) if rng.random() < 0.9 else int(rng.integers(1, 90))
    h = int(rng.integers(81, 600)) if rng.random() < 0.9 else int(rng.integers(1, 90))
    mono = bool(rng.random() < 0.5)
    qkind, q = _draw_q(rng, d2pc)
    frame = _draw_u8(rng, h, w) if mono else _draw_f32(rng, h, w)
    mode = str(rng.choice(MODES))
    grid = (float(rng.choice([0.02, 0.1, 0.5])), 0, ("z", 0.0, 10.0) if rng.random() < 0.5 else None)
    mn = int(rng.choice([0, 1, 2, 5, 50]))
    entry = str(rng.choice(ENTRIES + ["batch"]))
    ctx.set_q(q)
    crop = crop_of(frame, q)
    cloud = mode_cloud(crop, mode, grid)
    radius = _radius_from_pairs(rng, cloud) if rng.random() < 0.8 else float(rng.choice([0.01, 0.1, 1.0, 100.0]))
    desc = dict(case=case, w=w, h=h, mono=mono, q=qkind, mode=mode, grid=grid, radius=radius, mn=mn, entry=entry)
    wv = (outlier_ref.radius_outlier(np.frombuffer(cloud, np.uint8), radius, mn), 1)
    set_mode(d2pc, ctx, mode, grid)
    ctx.set_radius_outlier(radius, mn)
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
                wf = wv if f == 0 else want(crop_of(frames[1], q), mode, radius, mn, grid)
                check(pts[f * stride: f * stride + cnt[f] * 16], wf, (desc, f))
        else:
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, max(len(wv[0]), 16) + 64)
            check(got, wv, desc, cl)
    finally:
        reset(d2pc, ctx)
    return desc, len(wv[0]) // 16, len(cloud) // 16


def test_radius_outlier_fuzz_against_reference(env):
    seen, partial = set(), 0
    try:
        for case in range(N_FUZZ):
            d, kept, n_in = _fuzz_case(case, env)
            seen.add((d["mode"], d["entry"]))
            partial += 0 < kept < n_in
    finally:
        env[1].set_q(oracle.q_from_intrinsics())
    if N_FUZZ >= 100:
        assert len(seen) >= 15 and partial > N_FUZZ // 4, (seen, partial)
    print(f"radius outlier fuzz: {N_FUZZ} cases from seed {SEED0}, {len(seen)} (mode, entry) classes, "
          f"{partial} with some points kept and some dropped")
