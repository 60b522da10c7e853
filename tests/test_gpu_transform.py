"""GPU: the cloud transform (pcl::transformPointCloud, the first cloud stage) byte for byte against the CPU reference
tests/transform_ref, composed with tests/box_ref, tests/voxel_ref and tests/outlier_ref where those stages run,
through every entry point whose output depends on the filter plan, and d2pc_cloud_transform_device on hand-built
clouds.

The transform is applied to the reproject step's cloud: the oracle's where the arithmetic is EXACT, the library's own
CROP bytes where it is FAST.  D2PC_TRANSFORM_FUZZ_CASES / D2PC_TRANSFORM_FUZZ_SEED set the differential fuzz (default
150 cases)."""
import os
import subprocess

import numpy as np
import pytest

import box_ref
import oracle
import outlier_ref
import transform_ref
import voxel_ref
from disparity_to_point_cloud_b200 import synth
from test_gpu_crop_box import box_for, cloud_of, library_crop, set_mode, transform_of
from test_gpu_fuzz import _draw_f32, _draw_q, _draw_u8
from test_gpu_voxel import ENTRIES, check, crop_of, run_entry

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_TRANSFORM_FUZZ_CASES", "150"))
SEED0 = int(os.environ.get("D2PC_TRANSFORM_FUZZ_SEED", "61000"))
BUFFER_TOO_SMALL, INVALID_ARG, BAD_DIMS = -9, -1, -3
MODES = ["crop", "finite", "voxel"]
VOXEL_GRID = (0.05, 0, ("z", 0.0, 10.0))
ROR = (0.1, 2)
# camera optical frame -> a body frame: z forward becomes x forward, plus a small tilt and an offset
OPTICAL_TO_BODY = np.float32([[0, 0, 1], [-1, 0, 0], [0, -1, 0]])
POSE = np.concatenate([OPTICAL_TO_BODY @ transform_of((0.05, -0.1, 0.2), (0, 0, 0))[:, :3], [[0.1], [0.02], [-0.05]]],
                      axis=1).astype(np.float32)


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


def u8(data) -> np.ndarray:
    return np.frombuffer(data, np.uint8) if isinstance(data, bytes) else np.ascontiguousarray(data).view(np.uint8)


def want(crop, mode, xf=None, box=None, ror=None, grid=VOXEL_GRID):
    """The published cloud and its is_dense: reproject -> transform -> crop box -> VOXEL -> outlier stage."""
    data, dense = u8(crop).tobytes(), 0
    if mode == "finite":
        data, dense = oracle.filter_finite(u8(data)).tobytes(), 1
    if xf is not None:
        data = transform_ref.transform(u8(data), xf)
    if box is not None:
        data, dense = box_ref.crop_box(u8(data), *box), 1
    if mode == "voxel":
        data, vd = voxel_ref.voxel_grid(u8(data), *grid)
        dense = 1 if box is not None else vd
    if ror is not None:
        data, dense = outlier_ref.radius_outlier(u8(data), *ror), 1
    return data, dense


def reset(d2pc, ctx):
    ctx.set_transform(None)
    ctx.set_crop_box(None)
    ctx.set_radius_outlier(0.0)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ctx.set_arith_mode(d2pc.ARITH_EXACT)


def frame_crop(d2pc, ctx, frame, q, arith):
    if arith == "exact":
        return crop_of(frame, q)
    ctx.set_transform(None)
    return library_crop(d2pc, ctx, frame)


@pytest.mark.parametrize("arith", ["exact", "fast"])
@pytest.mark.parametrize("ror", [False, True])
@pytest.mark.parametrize("box", [False, True])
@pytest.mark.parametrize("mode", MODES)
def test_every_host_entry_matches_the_reference(env, mode, box, ror, arith):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    rr = ROR if ror else None
    try:
        ctx.set_arith_mode(d2pc.ARITH_FAST if arith == "fast" else d2pc.ARITH_EXACT)
        for frame in (synth.s2_scene(480, 752, 3), synth.s3_float(480, 752, 4)):
            crop = frame_crop(d2pc, ctx, frame, q, arith)
            # the box lies in the target frame: quantiles of the transformed cloud
            bx = box_for(u8(transform_ref.transform(crop, POSE)), 0.4, None) if box else None
            wv = want(crop, mode, POSE, bx, rr)
            assert 0 < len(wv[0])
            set_mode(d2pc, ctx, mode)
            ctx.set_radius_outlier(*(rr or (0.0,)))
            ctx.set_crop_box(*(bx or (None,)))
            ctx.set_transform(POSE)
            for entry in ENTRIES:
                got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                check(got, wv, (entry, frame.dtype, mode, box, ror, arith), cl)
    finally:
        reset(d2pc, ctx)


def test_crop_stays_uncounted_and_each_batch_gains_one_launch(env):
    """The transform alone keeps CROP uncounted: BUFFER_TOO_SMALL at submit, is_dense 0, d_counts optional; every
    mode makes exactly one launch more per call."""
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 9)
    crop = crop_of(frame, q)
    try:
        for mode in MODES:
            set_mode(d2pc, ctx, mode)
            launches = []
            for xf in (None, POSE):
                ctx.set_transform(xf)
                n0 = ctx.launch_count()
                got = ctx.process_mono8(frame)
                launches.append(ctx.launch_count() - n0)
                check(got, want(crop, mode, xf), (mode, xf is None), ctx.last_cloud)
            assert launches[1] == launches[0] + 1, (mode, launches)
        set_mode(d2pc, ctx, "crop")
        n = len(crop)
        with pytest.raises(d2pc.D2pcError) as e:  # CROP: the size is known at submit
            ctx.submit(0, frame, pin.array[: n - 16])
        assert e.value.status == BUFFER_TOO_SMALL
        check(ctx.process_into(frame, pin.array[:n]), want(crop, "crop", POSE), "exact fit", ctx.last_cloud)
        for direct in (1, -1):  # the transform kernel storing into page-locked memory, and never
            ctx.set_tuning("direct_out", direct)
            check(ctx.process_mono8(frame), want(crop, "crop", POSE), ("direct_out", direct), ctx.last_cloud)
    finally:
        ctx.set_tuning("direct_out", 0)
        reset(d2pc, ctx)


@pytest.mark.parametrize("mode", MODES)
def test_stream_and_4k(env, mode):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = np.stack([synth.s2_scene(480, 752, 20 + i) for i in range(5)])
    bx = box_for(u8(transform_ref.transform(crop_of(frames[0], q), POSE)), 0.5, None)
    set_mode(d2pc, ctx, mode)
    ctx.set_transform(POSE)
    try:
        for b in (None, bx):
            ctx.set_crop_box(*(b or (None,)))
            got = ctx.process_stream(frames, n_frames=7)
            for i, g in enumerate(got):
                check(g, want(crop_of(frames[i % 5], q), mode, POSE, b), ("stream", mode, b is None, i))
        ctx.set_crop_box(None)
        big = synth.s2_scene(2160, 3840, 6)
        wv = want(crop_of(big, q), mode, POSE)
        for entry in ("library", "pinned", "slot"):
            got, cl = run_entry(d2pc, ctx, pin, reg, big, entry, len(wv[0]) + 64)
            check(got, wv, ("4k", mode, entry), cl)
    finally:
        reset(d2pc, ctx)


@pytest.mark.parametrize("box", [False, True])
@pytest.mark.parametrize("mono", [True, False])
@pytest.mark.parametrize("mode", MODES)
def test_device_batch(env, mono, mode, box):
    import torch
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    h, w, nf = 480, 752, 4
    frames = np.stack([synth.s2_scene(h, w, 30 + i) for i in range(nf)])
    if not mono:
        frames = frames.astype(np.float32) * np.float32(0.125)
        frames[3] = synth.s3_float(h, w, 33)
    frames[2] = 0  # a frame with no finite point
    n = oracle.n_points(w, h)
    stride = n * 16 + 256
    d_in = torch.from_numpy(frames).cuda()
    d_pts = torch.zeros(nf * stride, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
    bx = box_for(u8(transform_ref.transform(crop_of(frames[0], q), POSE)), 0.5, None) if box else None
    set_mode(d2pc, ctx, mode)
    ctx.set_crop_box(*(bx or (None,)))
    step = w * frames.itemsize
    fn = ctx.reproject_mono8_device if mono else ctx.reproject_f32_device
    uncounted = mode == "crop" and not box
    try:
        n0 = ctx.launch_count()
        fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, d_cnt.data_ptr())
        ctx.sync()
        base = ctx.launch_count() - n0
        ctx.set_transform(POSE)
        if uncounted:  # CROP + transform: d_counts may be NULL
            d_pts.zero_()
            fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, 0)
            ctx.sync()
            for f in range(nf):
                check(d_pts.cpu().numpy()[f * stride: f * stride + n * 16], want(crop_of(frames[f], q), mode, POSE),
                      ("batch, no counts", f))
        else:
            with pytest.raises(d2pc.D2pcError) as e:
                fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, 0)
            assert e.value.status == INVALID_ARG
        d_cnt.fill_(-1)
        n0 = ctx.launch_count()
        fn(d_in.data_ptr(), nf, w, h, step, step * h, d_pts.data_ptr(), stride, d_cnt.data_ptr())
        ctx.sync()
        assert ctx.launch_count() - n0 == base + 1
    finally:
        reset(d2pc, ctx)
    counts, pts = d_cnt.cpu().numpy(), d_pts.cpu().numpy()
    for f in range(nf):
        wv = want(crop_of(frames[f], q), mode, POSE, bx)
        c = n if uncounted else counts[f]
        if uncounted:
            assert counts[f] == n  # the transform passes the reproject step's count on
        check(pts[f * stride: f * stride + c * 16], wv, ("batch", mode, box, f))


def test_fusion_entries(env):
    """fuse_then_process, submit_fusion and the fusion stream on 4 x 1280x720 with the transform, alone and in front
    of the box, VOXEL and the outlier stage."""
    d2pc, _, _, _ = env
    h, w = 720, 1280
    sets = np.stack([np.stack([synth.s2_scene(h, w, 40 + 4 * s + i) for i in range(4)]) for s in range(3)])
    grid = (0.1, 0, ("z", 0.0, 10.0))
    with d2pc.Context(offset_x=-7, offset_y=15, n_slots=2) as ctx:
        crops_fused = [ctx.fuse_then_process(*sets[s]) for s in range(3)]
        crops_pipe = ctx.process_fusion_stream(sets)
        bx = box_for(u8(transform_ref.transform(crops_fused[0], POSE)), 0.5, None)
        ctx.set_transform(POSE)
        for mode in MODES:
            for b, rr in ((None, None), (bx, (0.15, 2))):
                set_mode(d2pc, ctx, mode, grid)
                ctx.set_radius_outlier(*(rr or (0.0,)))
                ctx.set_crop_box(*(b or (None,)))
                wf = [want(c, mode, POSE, b, rr, grid) for c in crops_fused]
                wp = [want(c, mode, POSE, b, rr, grid) for c in crops_pipe]
                what = (mode, b is None, rr)
                for s in range(3):
                    check(ctx.fuse_then_process(*sets[s]), wf[s], ("fuse_then_process", what, s), ctx.last_cloud)
                for s in range(3):
                    ctx.submit_fusion(s % 2, *sets[s])
                    check(ctx.wait(s % 2), wp[s], ("submit_fusion", what, s), ctx.last_cloud)
                for s, g in enumerate(ctx.process_fusion_stream(sets, n_sets=5)):
                    check(g, wp[s % 3], ("fusion stream", what, s))


def test_voxel_overflow_fallback_behind_the_transform(env):
    """A VOXEL frame that takes the overflow fallback publishes the transformed CROP cloud, with is_dense 0."""
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s3_float(480, 752, 8)  # uniform disparities: hundreds of metres -> PCL's int overflow
    grid = (0.05, 0, None)
    moved = transform_ref.transform(crop_of(frame, q), POSE)
    assert voxel_ref.voxel_grid(u8(moved), *grid)[1] == 0  # the fallback is taken
    try:
        set_mode(d2pc, ctx, "voxel", grid)
        ctx.set_transform(POSE)
        for entry in ("library", "pinned", "pageable", "slot"):
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(moved) + 64)
            check(got, (moved, 0), ("fallback", entry), cl)
    finally:
        reset(d2pc, ctx)


def test_box_behind_the_transform_keeps_what_the_box_with_that_transform_keeps(env):
    """With T p finite for every point: box(identity) behind transform(T) keeps the points box(T) keeps, in the same
    order; only the bytes differ (transformed against original coordinates)."""
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    try:
        for seed in (90, 91):
            frame = synth.s2_scene(480, 752, seed)
            crop = crop_of(frame, q)
            mn, mx, _ = box_for(crop, 0.3, POSE)
            ctx.set_crop_box(mn, mx, POSE)
            kept_original = ctx.process_mono8(frame)
            ctx.set_crop_box(mn, mx, None)
            ctx.set_transform(POSE)
            kept_moved = ctx.process_mono8(frame)
            ctx.set_transform(None)
            assert 0 < len(kept_moved) == len(kept_original) < len(crop)
            assert kept_moved.tobytes() == transform_ref.transform(kept_original, POSE)
    finally:
        reset(d2pc, ctx)


def test_two_slots_submitted_under_different_poses(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = [synth.s2_scene(480, 752, 70 + i) for i in range(3)]
    poses = [transform_of((0.1 * i, -0.2, 0.3 * i), (i, -i, 0.5)) for i in range(3)]
    try:
        for mode in ("crop", "finite"):
            set_mode(d2pc, ctx, mode)
            for i in range(3):
                ctx.set_transform(poses[i])
                ctx.submit(i, frames[i])
            ctx.set_transform(None)
            for i in range(3):
                check(ctx.wait(i), want(crop_of(frames[i], q), mode, poses[i]), ("pending", mode, i), ctx.last_cloud)
    finally:
        reset(d2pc, ctx)


def hand_built_cases(rng):
    """(name, cloud, matrix)."""
    inf, nan = np.inf, np.nan
    nan_payload = cloud_of([[1, 2, 3], [4, 5, 6], [7, 8, 9]])
    nan_payload.view(np.uint32)[0, 0] = 0x7FC12345
    nan_payload.view(np.uint32)[1, 2] = 0xFFA00001
    zeros = cloud_of([[-0.0, 0.0, -0.0], [1e-45, -1e-45, 0.0]])
    return [("rotated", cloud_of(rng.normal(0, 2, (6000, 3))), POSE),
            ("affine", cloud_of(rng.normal(0, 2, (3000, 3))), rng.normal(0, 1, (3, 4)).astype(np.float32)),
            ("non-finite", cloud_of([[0, 0, 0], [nan, 0, 0], [0, inf, 0], [0, 0, -inf], [0.5, 0.5, 0.5]]), POSE),
            ("nan payloads", nan_payload, POSE),
            ("identity on zeros", zeros, np.eye(3, 4, dtype=np.float32)),
            ("quarter turn", cloud_of(rng.uniform(-3, 3, (5000, 3))),
             np.float32([[0, 1, 0, 0], [-1, 0, 0, 0], [0, 0, 1, 0]])),
            ("overflow", cloud_of([[3e38, 3e38, 0], [-3e38, 3e38, 1], [1, 1, 1]]),
             np.float32([[10, 0, 0, 0], [1e3, 1e3, 0, 0], [0, 0, 1, 0]]))]


def test_device_entry_on_hand_built_clouds(env):
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(81)
    cases = hand_built_cases(rng)
    try:
        for name, pts, m in cases:  # one frame each, the context's setting, counts out optional
            ctx.set_transform(m)
            d_in = torch.from_numpy(pts.view(np.uint8).reshape(-1).copy()).cuda()
            d_out = torch.zeros(len(pts) * 16, dtype=torch.uint8, device="cuda")
            n0 = ctx.launch_count()
            ctx.transform_device(d_in.data_ptr(), 1, len(pts), len(pts) * 16, 0, d_out.data_ptr(), len(pts) * 16)
            ctx.sync()
            assert ctx.launch_count() - n0 == 1
            assert d_out.cpu().numpy().tobytes() == transform_ref.transform(pts, m), name
            ctx.transform_device(d_in.data_ptr(), 1, len(pts), 0, 0, d_in.data_ptr(), 0)  # in place
            ctx.sync()
            assert d_in.cpu().numpy().tobytes() == transform_ref.transform(pts, m), (name, "in place")
        # several frames, per-frame counts below n_max and per-frame matrices; positions past a count are neither
        # read nor written
        n_max, nf = 6000, len(cases)
        stride = n_max * 16 + 64
        host = np.zeros(nf * stride // 4, np.float32)
        host.view(np.uint32)[1::7] = 0x3F000000
        counts = np.zeros(nf, np.uint32)
        mats = np.stack([m for _, _, m in cases]).astype(np.float32)
        for f, (_, pts, _) in enumerate(cases):
            k = min(len(pts), n_max)
            host.view(np.uint8)[f * stride: f * stride + k * 16] = pts[:k].view(np.uint8).reshape(-1)
            counts[f] = k
        counts[0] = 1234  # below the frame's points
        counts[-1] = n_max * 3  # above n_max counts as n_max
        ctx.set_transform(None)
        d_in = torch.from_numpy(host.view(np.uint8).copy()).cuda()
        d_cnt_in = torch.from_numpy(counts.view(np.int32)).cuda()
        d_mats = torch.from_numpy(mats.reshape(-1)).cuda()
        sentinel = 0xA5
        d_out = torch.full((nf * stride,), sentinel, dtype=torch.uint8, device="cuda")
        d_cnt = torch.full((nf,), -1, dtype=torch.int32, device="cuda")
        ctx.transform_device(d_in.data_ptr(), nf, n_max, stride, d_cnt_in.data_ptr(), d_out.data_ptr(), stride,
                             d_cnt.data_ptr(), d_mats.data_ptr())
        ctx.sync()
        got_c, got = d_cnt.cpu().numpy(), d_out.cpu().numpy()
        for f in range(nf):
            k = min(int(counts[f]), n_max)
            assert got_c[f] == k
            src = host.view(np.uint8)[f * stride: f * stride + k * 16]
            assert got[f * stride: f * stride + k * 16].tobytes() == transform_ref.transform(src, mats[f]), f
            assert (got[f * stride + k * 16: (f + 1) * stride] == sentinel).all(), f
        # the same batch in place, without counts out
        ctx.transform_device(d_in.data_ptr(), nf, n_max, stride, d_cnt_in.data_ptr(), d_in.data_ptr(), stride, 0,
                             d_mats.data_ptr())
        ctx.sync()
        inplace = d_in.cpu().numpy()
        for f in range(nf):
            k = min(int(counts[f]), n_max)
            src = host.view(np.uint8)[f * stride: (f + 1) * stride]
            assert inplace[f * stride: f * stride + k * 16].tobytes() == transform_ref.transform(src[: k * 16], mats[f])
            assert inplace[f * stride + k * 16: (f + 1) * stride].tobytes() == src[k * 16:].tobytes(), f
        # n_max 0: every count is 0
        d_cnt.fill_(7)
        ctx.transform_device(d_in.data_ptr(), nf, 0, 0, 0, d_out.data_ptr(), 0, d_cnt.data_ptr(), d_mats.data_ptr())
        ctx.sync()
        assert not d_cnt.cpu().numpy().any()
    finally:
        reset(d2pc, ctx)


def test_device_entry_on_70000_frames(env):
    """70 000 frames of 5 points with per-frame matrices in one call."""
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(82)
    nf, n = 70000, 5
    pts = rng.normal(0, 3, (nf, n, 4)).astype(np.float32)
    pts[..., 3] = 1.0
    pts[rng.random((nf, n)) < 0.1, 0] = np.nan
    mats = rng.normal(0, 1, (nf, 3, 4)).astype(np.float32)
    counts = rng.integers(0, n + 1, nf).astype(np.uint32)
    d_in = torch.from_numpy(pts.reshape(-1)).cuda()
    d_out = torch.zeros(nf * n * 4, dtype=torch.float32, device="cuda")
    d_cnt_in = torch.from_numpy(counts.view(np.int32)).cuda()
    d_cnt = torch.full((nf,), -1, dtype=torch.int32, device="cuda")
    d_mats = torch.from_numpy(mats.reshape(-1)).cuda()
    n0 = ctx.launch_count()
    ctx.transform_device(d_in.data_ptr(), nf, n, n * 16, d_cnt_in.data_ptr(), d_out.data_ptr(), n * 16,
                         d_cnt.data_ptr(), d_mats.data_ptr())
    ctx.sync()
    assert ctx.launch_count() - n0 == 1
    got = d_out.cpu().numpy().reshape(nf, n, 4)
    assert np.array_equal(d_cnt.cpu().numpy(), counts.astype(np.int32))
    for f in range(nf):
        k = int(counts[f])
        assert got[f, :k].tobytes() == transform_ref.transform(pts[f, :k], mats[f]), f
        assert not got[f, k:].any(), f


def test_refused_arguments_and_settings(env):
    import torch
    d2pc, _, _, _ = env
    with d2pc.Context() as ctx:
        t = ctx.get_transform()
        assert (t.struct_size, t.enabled, list(t.matrix)) == (56, 0, list(np.eye(3, 4).reshape(12)))
        n_max, stride = 100, 1600
        d = torch.zeros(4 * stride, dtype=torch.uint8, device="cuda")
        p = d.data_ptr()
        with pytest.raises(d2pc.D2pcError) as e:  # NULL matrices and the setting off
            ctx.transform_device(p, 1, n_max, stride, 0, p + stride, stride)
        assert e.value.status == INVALID_ARG
        ctx.set_transform(POSE)
        for out, out_stride in ((p + 16, stride), (p + stride, stride), (p, stride + 16)):  # partial overlaps
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.transform_device(p, 2, n_max, stride, 0, out, out_stride)
            assert e.value.status == INVALID_ARG, (out - p, out_stride)
        with pytest.raises(d2pc.D2pcError) as e:  # misaligned
            ctx.transform_device(p + 4, 1, n_max, stride, 0, p + 2 * stride, stride)
        assert e.value.status == BAD_DIMS
        with pytest.raises(d2pc.D2pcError) as e:  # stride below a frame
            ctx.transform_device(p, 2, n_max, n_max * 8, 0, p + 2 * stride, stride)
        assert e.value.status == BAD_DIMS
        ctx.transform_device(p, 2, n_max, stride, 0, p, stride)  # exact in place is allowed
        ctx.transform_device(p, 2, n_max, stride, 0, p + 2 * stride, stride)  # adjacent, no overlap
        ctx.sync()
        for v in (np.nan, np.inf, -np.inf):
            bad = POSE.copy()
            bad[2, 1] = v
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.set_transform(bad)
            assert e.value.status == INVALID_ARG
        raw = d2pc.CloudTransform()
        d2pc.lib().d2pc_cloud_transform_default(raw)
        raw.struct_size = 52
        assert d2pc.lib().d2pc_set_cloud_transform(ctx._h, raw) == INVALID_ARG
        g = ctx.get_transform()  # the previous setting is kept
        assert g.enabled == 1 and np.array_equal(np.float32(g.matrix), POSE.reshape(12))
        ctx.set_transform(np.vstack([POSE, [0, 0, 0, 1]]))  # 4x4
        assert np.array_equal(np.float32(ctx.get_transform().matrix), POSE.reshape(12))
        with pytest.raises(ValueError):
            ctx.set_transform(np.eye(4) * 2)
        frame = synth.s2_scene(480, 752, 50)
        crop = oracle.disparity_cb_mono8(frame, ctx.get_q())
        check(ctx.process_mono8(frame), want(crop, "crop", POSE), "on", ctx.last_cloud)
        ctx.set_transform(None)
        assert ctx.get_transform().enabled == 0
        check(ctx.process_mono8(frame), (crop.tobytes(), 0), "off", ctx.last_cloud)


def test_node1_transform_params_and_frame_id(tmp_path):
    from disparity_to_point_cloud_b200 import build
    build.build()
    harness = build.build_harness()
    q = oracle.q_from_intrinsics()
    pose = dict(tx=0.2, ty=-0.1, tz=0.05, roll=-1.5707963, pitch=0.05, yaw=-1.5707963)
    box = dict(min_x=0.5, min_y=-1.0, min_z=-0.5, max_x=4.0, max_y=1.0, max_z=0.8)
    img = synth.s2_scene(480, 752, 51)
    crop = oracle.disparity_cb_mono8(img, q)
    t = transform_of((pose["roll"], pose["pitch"], pose["yaw"]), (pose["tx"], pose["ty"], pose["tz"]))
    for with_box in (False, True):
        params = "".join(f'    <param name="transform_{k}" value="{v}"/>\n' for k, v in pose.items())
        if with_box:
            params += '    <param name="crop_box_enable" value="1"/>\n'
            params += "".join(f'    <param name="crop_box_{k}" value="{v}"/>\n' for k, v in box.items())
        launch = tmp_path / f"xf{with_box}.launch"
        launch.write_text('<launch>\n  <node name="disparity_to_point_cloud" pkg="disparity_to_point_cloud" '
                          'type="disparity_to_point_cloud_node">\n'
                          '    <remap from="/disparity" to="/throttled_depth_map"/>\n'
                          '    <param name="transform_enable" value="1"/>\n'
                          '    <param name="transform_target_frame" value="/body"/>\n' + params +
                          '  </node>\n</launch>\n')
        raw, out = tmp_path / "in.raw", tmp_path / "cloud.bin"
        raw.write_bytes(img.tobytes())
        subprocess.run([harness, "node1", str(launch), "752", "480", str(raw), str(out), "1700000000", "250"],
                       check=True)
        bx = ([box["min_x"], box["min_y"], box["min_z"]], [box["max_x"], box["max_y"], box["max_z"]], None)
        data, dense = want(crop, "crop", t, bx if with_box else None)
        assert len(data) > 0
        wire = oracle.serialize_pointcloud2(u8(data), seq=0, sec=1700000000, nsec=250, frame_id="/body",
                                            is_dense=dense)
        assert out.read_bytes() == wire, with_box


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
    rr = (float(rng.choice([0.02, 0.1, 0.5])), int(rng.choice([0, 1, 3]))) if rng.random() < 0.3 else None
    entry = str(rng.choice(ENTRIES + ["batch"]))
    ctx.set_q(q)
    crop = crop_of(frame, q)
    xf = transform_of(rng.uniform(-np.pi, np.pi, 3), rng.normal(0, 1, 3))
    if rng.random() < 0.2:  # a general affine map
        xf = rng.normal(0, 1.5, (3, 4)).astype(np.float32)
    bx = None
    if rng.random() < 0.4:
        bx = box_for(u8(transform_ref.transform(crop, xf)), float(rng.choice([0.5, 0.1])), None, rng)
    desc = dict(case=case, w=w, h=h, mono=mono, q=qkind, mode=mode, grid=grid, ror=rr, box=bx is not None,
                entry=entry)
    wv = want(crop, mode, xf, bx, rr, grid)
    set_mode(d2pc, ctx, mode, grid)
    ctx.set_radius_outlier(*(rr or (0.0,)))
    ctx.set_crop_box(*(bx or (None,)))
    ctx.set_transform(xf)
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
                wf = wv if f == 0 else want(crop_of(frames[1], q), mode, xf, bx, rr, grid)
                check(pts[f * stride: f * stride + cnt[f] * 16], wf, (desc, f))
        else:
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, max(len(wv[0]), 16) + 64)
            check(got, wv, desc, cl)
    finally:
        reset(d2pc, ctx)
    return desc


def test_transform_fuzz_against_reference(env):
    seen = set()
    try:
        for case in range(N_FUZZ):
            d = _fuzz_case(case, env)
            seen.add((d["mode"], d["entry"], d["box"]))
    finally:
        env[1].set_q(oracle.q_from_intrinsics())
    if N_FUZZ >= 100:
        assert len(seen) >= 25, seen
    print(f"transform fuzz: {N_FUZZ} cases from seed {SEED0}, {len(seen)} (mode, entry, box) classes")
