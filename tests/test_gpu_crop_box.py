"""GPU: the crop box (pcl::CropBox with setTransform, in front of VOXEL and the radius outlier stage) byte for byte
against the CPU reference tests/box_ref, composed with tests/voxel_ref and tests/outlier_ref where those stages run,
through every entry point whose output depends on the filter plan, and d2pc_crop_box_device on hand-built clouds.

The box is applied to the CROP cloud: the oracle's where the arithmetic is EXACT, the library's own CROP bytes where
it is FAST.  D2PC_BOX_FUZZ_CASES / D2PC_BOX_FUZZ_SEED set the differential fuzz (default 150 cases)."""
import os
import subprocess

import numpy as np
import pytest

import box_ref
import oracle
import outlier_ref
import voxel_ref
from disparity_to_point_cloud_b200 import synth
from test_gpu_fuzz import _draw_f32, _draw_q, _draw_u8
from test_gpu_voxel import ENTRIES, check, crop_of, run_entry

pytestmark = pytest.mark.gpu

N_FUZZ = int(os.environ.get("D2PC_BOX_FUZZ_CASES", "150"))
SEED0 = int(os.environ.get("D2PC_BOX_FUZZ_SEED", "53000"))
BUFFER_TOO_SMALL, INVALID_ARG, BAD_DIMS = -9, -1, -3
MODES = ["crop", "finite", "voxel"]
VOXEL_GRID = (0.05, 0, ("z", 0.0, 10.0))
ROR = (0.1, 2)


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


def rot(roll, pitch, yaw) -> np.ndarray:
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    return np.array([[cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr],
                     [sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr],
                     [-sp, cp * sr, cp * cr]])


def transform_of(rpy, t) -> np.ndarray:
    return np.concatenate([rot(*rpy), np.reshape(t, (3, 1))], axis=1).astype(np.float32)


ROTATED = transform_of((0.3, -0.2, 0.5), (0.1, -0.2, 0.3))


def box_for(cloud, frac, t=None, rng=None):
    """A box (min_pt, max_pt, t) that keeps about `frac` of the cloud's finite points: per-axis quantiles of T p."""
    pts = np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4)[:, :3]
    pts = pts[np.isfinite(pts).all(1)]
    tt = box_ref.IDENTITY if t is None else t
    if len(pts) == 0:
        return np.float32([-1] * 3), np.float32([1] * 3), t
    with np.errstate(over="ignore", invalid="ignore"):
        loc = pts.astype(np.float64) @ tt[:, :3].T.astype(np.float64) + tt[:, 3]
    side = frac ** (1 / 3)
    lo = (1 - side) / 2 if rng is None else float(rng.uniform(0, 1 - side))
    mn = np.nanquantile(loc, lo, axis=0).astype(np.float32)
    mx = np.nanquantile(loc, lo + side, axis=0).astype(np.float32)
    return mn, mx, t


def set_mode(d2pc, ctx, mode, grid=VOXEL_GRID):
    if mode == "voxel":
        ctx.set_voxel_grid(*grid)
    ctx.set_filter_mode({"crop": d2pc.FILTER_CROP, "finite": d2pc.FILTER_CROP_FINITE, "voxel": d2pc.FILTER_VOXEL}[mode])


def want(crop, box, mode, ror=None, grid=VOXEL_GRID):
    """The published cloud: VoxelGrid / outlier stage of CropBox(CROP cloud); is_dense is always 1."""
    data = box_ref.crop_box(np.frombuffer(crop, np.uint8) if isinstance(crop, bytes) else crop, *box)
    if mode == "voxel":
        data = voxel_ref.voxel_grid(np.frombuffer(data, np.uint8), *grid)[0]
    if ror is not None:
        data = outlier_ref.radius_outlier(np.frombuffer(data, np.uint8), *ror)
    return data, 1


def reset(d2pc, ctx):
    ctx.set_crop_box(None)
    ctx.set_radius_outlier(0.0)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    ctx.set_arith_mode(d2pc.ARITH_EXACT)


def library_crop(d2pc, ctx, frame):
    """The library's own CROP cloud of a frame with the context's Q and arithmetic."""
    ctx.set_crop_box(None)
    ctx.set_radius_outlier(0.0)
    ctx.set_filter_mode(d2pc.FILTER_CROP)
    return ctx.process_f32(frame) if frame.dtype == np.float32 else ctx.process_mono8(frame)


@pytest.mark.parametrize("arith", ["exact", "fast"])
@pytest.mark.parametrize("ror", [False, True])
@pytest.mark.parametrize("mode", MODES)
def test_every_host_entry_matches_the_reference(env, mode, ror, arith):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    rr = ROR if ror else None
    try:
        ctx.set_arith_mode(d2pc.ARITH_FAST if arith == "fast" else d2pc.ARITH_EXACT)
        for frame in (synth.s2_scene(480, 752, 3), synth.s3_float(480, 752, 4)):
            crop = crop_of(frame, q) if arith == "exact" else library_crop(d2pc, ctx, frame)
            for t in (None, ROTATED):
                box = box_for(crop, 0.4, t)
                wv = want(crop, box, mode, rr)
                assert 0 < len(wv[0])
                set_mode(d2pc, ctx, mode)
                ctx.set_radius_outlier(*(rr or (0.0,)))
                ctx.set_crop_box(*box)
                for entry in ENTRIES:
                    got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(wv[0]) + 64)
                    check(got, wv, (entry, frame.dtype, mode, ror, arith, t is None), cl)
    finally:
        reset(d2pc, ctx)


def test_crop_and_crop_finite_give_the_same_bytes_and_launches(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    try:
        for f in (synth.s2_scene(480, 752, 11), synth.s3_float(480, 752, 12)):
            crop = crop_of(f, q)
            for frac, t in ((1.0, None), (0.5, ROTATED), (0.1, None)):
                box = box_for(crop, frac, t)
                ctx.set_crop_box(*box)
                out = []
                for m in (d2pc.FILTER_CROP, d2pc.FILTER_CROP_FINITE):
                    ctx.set_filter_mode(m)
                    n0 = ctx.launch_count()
                    got = (ctx.process_f32(f) if f.dtype == np.float32 else ctx.process_mono8(f)).tobytes()
                    out.append((got, ctx.launch_count() - n0, ctx.last_cloud.is_dense))
                assert out[0] == out[1], (frac, f.dtype)
                assert out[0][0] == want(crop, box, "crop")[0] and out[0][2] == 1
    finally:
        reset(d2pc, ctx)


def test_too_small_destination_is_reported_at_wait(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s2_scene(480, 752, 5)
    crop = crop_of(frame, q)
    box = box_for(crop, 0.3, ROTATED)
    wv = want(crop, box, "crop")
    n = len(wv[0])
    assert n > 32
    ctx.set_crop_box(*box)
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


@pytest.mark.parametrize("mode", MODES)
def test_stream_and_4k(env, mode):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = np.stack([synth.s2_scene(480, 752, 20 + i) for i in range(5)])
    box = box_for(crop_of(frames[0], q), 0.5, ROTATED)
    set_mode(d2pc, ctx, mode)
    ctx.set_crop_box(*box)
    try:
        got = ctx.process_stream(frames, n_frames=7)
        for i, g in enumerate(got):
            check(g, want(crop_of(frames[i % 5], q), box, mode), ("stream", mode, i))
        big = synth.s2_scene(2160, 3840, 6)
        crop = crop_of(big, q)
        box = box_for(crop, 0.2, ROTATED)
        ctx.set_crop_box(*box)
        wv = want(crop, box, mode)
        for entry in ("library", "pinned", "slot"):
            got, cl = run_entry(d2pc, ctx, pin, reg, big, entry, len(wv[0]) + 64)
            check(got, wv, ("4k", mode, entry), cl)
    finally:
        reset(d2pc, ctx)


@pytest.mark.parametrize("ror", [False, True])
@pytest.mark.parametrize("mono", [True, False])
@pytest.mark.parametrize("mode", MODES)
def test_device_batch_per_frame_counts(env, mono, mode, ror):
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
    box = box_for(crop_of(frames[0], q), 0.5, ROTATED)
    rr = ROR if ror else None
    set_mode(d2pc, ctx, mode)
    ctx.set_radius_outlier(*(rr or (0.0,)))
    ctx.set_crop_box(*box)
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
    counts, pts = d_cnt.cpu().numpy(), d_pts.cpu().numpy()
    wants = [want(crop_of(frames[f], q), box, mode, rr) for f in range(nf)]
    assert counts[2] == 0 and len(wants[0][0]) > 0
    for f in range(nf):
        check(pts[f * stride: f * stride + counts[f] * 16], wants[f], ("batch", mode, ror, f))


def test_device_batch_of_more_than_65535_voxel_frames(env):
    """70 000 tiny frames (border 0, 4 x 2 pixels) through VOXEL + box in one device call: the batch runs in chunks."""
    import torch
    d2pc, _, _, _ = env
    rng = np.random.default_rng(60)
    nf, h, w = 70000, 2, 4
    frames = rng.uniform(0.5, 60, (nf, h, w)).astype(np.float32)
    frames[rng.random((nf, h, w)) < 0.1] = 0.0  # zero disparity: non-finite points
    n = h * w
    with d2pc.Context() as ctx:
        ctx.set_tuning("border", 0)
        d_in = torch.from_numpy(frames).cuda()
        d_crop = torch.zeros(nf * n * 16, dtype=torch.uint8, device="cuda")
        ctx.reproject_f32_device(d_in.data_ptr(), nf, w, h, w * 4, w * h * 4, d_crop.data_ptr(), n * 16, 0)
        ctx.sync()
        crops = d_crop.cpu().numpy().reshape(nf, n * 16)
        box = (np.float32([-50, -50, 0.0]), np.float32([50, 50, 300.0]), ROTATED)
        grid = (2.0, 0, None)
        set_mode(d2pc, ctx, "voxel", grid)
        ctx.set_crop_box(*box)
        d_pts = torch.zeros(nf * n * 16, dtype=torch.uint8, device="cuda")
        d_cnt = torch.full((nf,), -1, dtype=torch.int32, device="cuda")
        ctx.reproject_f32_device(d_in.data_ptr(), nf, w, h, w * 4, w * h * 4, d_pts.data_ptr(), n * 16,
                                 d_cnt.data_ptr())
        ctx.sync()
        counts, pts = d_cnt.cpu().numpy(), d_pts.cpu().numpy()
    merged = 0
    for f in range(nf):
        wv = want(crops[f], box, "voxel", None, grid)
        check(pts[f * n * 16: f * n * 16 + counts[f] * 16], wv, ("70k", f))
        merged += len(wv[0]) < len(box_ref.crop_box(crops[f], *box))
    assert merged > 1000


def test_fusion_entries(env):
    """fuse_then_process, submit_fusion and the fusion stream on 4 x 1280x720: the box applied to the CROP cloud of
    the same set, then VOXEL / the outlier stage."""
    d2pc, _, _, _ = env
    h, w = 720, 1280
    sets = np.stack([np.stack([synth.s2_scene(h, w, 40 + 4 * s + i) for i in range(4)]) for s in range(3)])
    grid = (0.1, 0, ("z", 0.0, 10.0))
    with d2pc.Context(offset_x=-7, offset_y=15, n_slots=2) as ctx:
        crops_fused = [ctx.fuse_then_process(*sets[s]) for s in range(3)]
        crops_pipe = ctx.process_fusion_stream(sets)
        box = box_for(crops_fused[0], 0.5, ROTATED)
        for mode in MODES:
            for rr in (None, (0.15, 2)):
                set_mode(d2pc, ctx, mode, grid)
                ctx.set_radius_outlier(*(rr or (0.0,)))
                ctx.set_crop_box(*box)
                wf = [want(c, box, mode, rr, grid) for c in crops_fused]
                wp = [want(c, box, mode, rr, grid) for c in crops_pipe]
                for s in range(3):
                    check(ctx.fuse_then_process(*sets[s]), wf[s], ("fuse_then_process", mode, rr, s), ctx.last_cloud)
                for s in range(3):
                    ctx.submit_fusion(s % 2, *sets[s])
                    check(ctx.wait(s % 2), wp[s], ("submit_fusion", mode, rr, s), ctx.last_cloud)
                for s, g in enumerate(ctx.process_fusion_stream(sets, n_sets=5)):
                    check(g, wp[s % 3], ("fusion stream", mode, rr, s))


def test_voxel_overflow_fallback_behind_the_box_is_dense(env):
    """A VOXEL frame that takes the overflow fallback publishes the box's cloud, with is_dense 1."""
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frame = synth.s3_float(480, 752, 8)  # uniform disparities: hundreds of metres -> PCL's int overflow
    crop = crop_of(frame, q)
    grid = (0.05, 0, None)
    box = (np.float32([0, -1e4, -1e4]), np.float32([1e4] * 3), ROTATED)  # about half the points
    inside = box_ref.crop_box(crop, *box)
    assert voxel_ref.voxel_grid(np.frombuffer(inside, np.uint8), *grid)[1] == 0  # the fallback is taken
    assert 0 < len(inside) < np.isfinite(crop.view(np.float32).reshape(-1, 4)[:, :3]).all(1).sum() * 16
    try:
        set_mode(d2pc, ctx, "voxel", grid)
        ctx.set_crop_box(*box)
        for entry in ("library", "pinned", "pageable", "slot"):
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, len(inside) + 64)
            check(got, (inside, 1), ("fallback", entry), cl)
    finally:
        reset(d2pc, ctx)


def cloud_of(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    pts = np.zeros((len(xyz), 4), np.float32)
    pts[:, :3] = xyz
    pts[:, 3] = np.arange(len(xyz), dtype=np.float32)  # the pad word travels unchanged
    return pts


def hand_built_cases(rng):
    """(name, cloud, min_pt, max_pt, transform)."""
    mn, mx = np.float32([-1.5, -0.25, 0.0]), np.float32([2.0, 0.75, 10.0])
    faces = []
    for a in range(3):
        for v in (mn[a], mx[a], np.nextafter(mn[a], np.float32(-np.inf)), np.nextafter(mx[a], np.float32(np.inf))):
            p = (mn + mx) / 2
            p[a] = v
            faces.append(p)
    inf, nan = np.inf, np.nan
    out = [("faces", cloud_of(faces), mn, mx, None),
           ("signed zeros", cloud_of([[0, 0, 0], [-0.0, -0.0, -0.0], [-1e-45, 0, 0], [0, 1e-45, 0]]), [0, -0.0, 0],
            [0.0, 0, 0], None),
           ("non-finite", cloud_of([[0, 0, 0], [nan, 0, 0], [0, inf, 0], [0, 0, -inf], [0.5, 0.5, 0.5]]), [-1] * 3,
            [1] * 3, ROTATED),
           ("infinite bounds", cloud_of(rng.normal(0, 1e30, (3000, 3))), [-inf, -inf, 0], [inf, inf, inf], None),
           ("quarter turn", cloud_of(rng.uniform(-3, 3, (5000, 3))), [0, -2, -1], [1, 0, 1],
            np.float32([[0, 1, 0, 0.5], [-1, 0, 0, 0], [0, 0, 1, 0]])),
           ("rotated", cloud_of(rng.normal(0, 2, (6000, 3))), [-1, -2, -0.5], [1.5, 0.5, 2], ROTATED),
           ("overflowing transform", cloud_of([[3e38, 3e38, 0], [1, 1, 1]]), [-inf] * 3, [inf] * 3,
            np.float32([[1e3, -1e3, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]])),  # inf - inf: a NaN l is dropped
           ("empty result", cloud_of(rng.uniform(-1, 1, (100, 3))), [2] * 3, [3] * 3, None),
           ("empty", cloud_of(np.empty((0, 3))), [-1] * 3, [1] * 3, None)]
    return out


def test_device_entry_on_hand_built_clouds(env):
    import torch
    d2pc, ctx, _, _ = env
    rng = np.random.default_rng(81)
    cases = hand_built_cases(rng)
    try:
        for name, pts, mn, mx, t in cases:  # one frame each
            ctx.set_crop_box(mn, mx, t)
            n = max(len(pts), 1)
            d_in = torch.from_numpy(np.ascontiguousarray(pts).view(np.uint8).reshape(-1)).cuda() if len(pts) else \
                torch.zeros(16, dtype=torch.uint8, device="cuda")
            d_out = torch.zeros(n * 16, dtype=torch.uint8, device="cuda")
            d_cnt = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
            ctx.crop_box_device(d_in.data_ptr(), 1, len(pts), n * 16, 0, d_out.data_ptr(), n * 16, d_cnt.data_ptr())
            ctx.sync()
            c = int(d_cnt.cpu()[0])
            check(d_out.cpu().numpy()[: c * 16], (box_ref.crop_box(pts, mn, mx, t), 1), name)
        # several frames with per-frame counts (positions past the count hold garbage that must not be read)
        n_max, nf = 6000, len(cases)
        stride = n_max * 16 + 64
        host = np.zeros(nf * stride // 4, np.float32)
        host.view(np.uint32)[1::7] = 0x3f000000  # 0.5: inside most boxes, so a read past the count would show
        counts = np.zeros(nf, np.uint32)
        for f, (_, pts, _, _, _) in enumerate(cases):
            m = min(len(pts), n_max)
            host.view(np.uint8)[f * stride: f * stride + m * 16] = pts[:m].view(np.uint8).reshape(-1)
            counts[f] = m
        counts[-1] = n_max * 3  # above n_max counts as n_max
        box = (np.float32([-1, -1, -1]), np.float32([1, 1, 1]), ROTATED)
        ctx.set_crop_box(*box)
        d_in = torch.from_numpy(host.view(np.uint8)).cuda()
        d_cnt_in = torch.from_numpy(counts.view(np.int32)).cuda()
        d_out = torch.zeros(nf * stride, dtype=torch.uint8, device="cuda")
        d_cnt = torch.zeros(nf, dtype=torch.int32, device="cuda")
        ctx.crop_box_device(d_in.data_ptr(), nf, n_max, stride, d_cnt_in.data_ptr(), d_out.data_ptr(), stride,
                            d_cnt.data_ptr())
        ctx.sync()
        got_c, got = d_cnt.cpu().numpy(), d_out.cpu().numpy()
        for f in range(nf):
            m = min(int(counts[f]), n_max)
            wv = box_ref.crop_box(host.view(np.uint8)[f * stride: f * stride + m * 16], *box)
            check(got[f * stride: f * stride + got_c[f] * 16], (wv, 1), ("batch", f))
        assert len(box_ref.crop_box(host.view(np.uint8)[(nf - 1) * stride: nf * stride - 64], *box)) > 0
        # n_max 0: every count is 0
        d_cnt.fill_(7)
        ctx.crop_box_device(d_in.data_ptr(), nf, 0, 0, 0, d_out.data_ptr(), 0, d_cnt.data_ptr())
        ctx.sync()
        assert not d_cnt.cpu().numpy().any()
        # argument checks
        with pytest.raises(d2pc.D2pcError) as e:  # counts out are required
            ctx.crop_box_device(d_in.data_ptr(), nf, n_max, stride, 0, d_out.data_ptr(), stride, 0)
        assert e.value.status == INVALID_ARG
        with pytest.raises(d2pc.D2pcError) as e:  # input and output overlap
            ctx.crop_box_device(d_in.data_ptr(), 2, n_max, stride, 0, d_in.data_ptr() + stride, stride,
                                d_cnt.data_ptr())
        assert e.value.status == INVALID_ARG
        with pytest.raises(d2pc.D2pcError) as e:  # stride below a frame
            ctx.crop_box_device(d_in.data_ptr(), 2, n_max, n_max * 8, 0, d_out.data_ptr(), stride, d_cnt.data_ptr())
        assert e.value.status == BAD_DIMS
        for off_in, off_out in ((4, 0), (0, 8)):  # misaligned
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.crop_box_device(d_in.data_ptr() + off_in, 1, 10, stride, 0, d_out.data_ptr() + off_out, stride,
                                    d_cnt.data_ptr())
            assert e.value.status == BAD_DIMS
        ctx.set_crop_box(None)
        with pytest.raises(d2pc.D2pcError) as e:  # the box is off
            ctx.crop_box_device(d_in.data_ptr(), 1, 10, stride, 0, d_out.data_ptr(), stride, d_cnt.data_ptr())
        assert e.value.status == INVALID_ARG
    finally:
        reset(d2pc, ctx)


def test_settings_are_checked_and_off_restores_crop(env):
    d2pc, _, _, _ = env
    frame = synth.s2_scene(480, 752, 50)
    with d2pc.Context() as ctx:
        q = ctx.get_q()
        b = ctx.get_crop_box()
        assert (b.struct_size, b.enabled, list(b.min_pt), list(b.max_pt)) == (80, 0, [-1.0] * 3, [1.0] * 3)
        assert list(b.transform) == list(np.eye(3, 4).reshape(12))
        crop = ctx.process_mono8(frame)
        assert crop.tobytes() == oracle.disparity_cb_mono8(frame, q).tobytes() and ctx.last_cloud.is_dense == 0
        n_crop = ctx.launch_count()
        box = box_for(crop, 0.3, ROTATED)
        ctx.set_crop_box(*box)
        nan, inf = float("nan"), float("inf")
        bad_t = ROTATED.copy()
        for args in (([nan, 0, 0], [1, 1, 1]), ([0, 0, 0], [1, nan, 1]), ([0, 2, 0], [1, 1, 1]),
                     ([1, 0, 0], [-inf, 1, 1])):
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.set_crop_box(*args)
            assert e.value.status == INVALID_ARG
        for v in (nan, inf, -inf):
            bad_t[1, 2] = v
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.set_crop_box([0] * 3, [1] * 3, bad_t)
            assert e.value.status == INVALID_ARG
        raw = d2pc.CropBox()
        d2pc.lib().d2pc_crop_box_default(raw)
        raw.struct_size = 76
        assert d2pc.lib().d2pc_set_crop_box(ctx._h, raw) == INVALID_ARG
        g = ctx.get_crop_box()  # the previous setting is kept
        assert g.enabled == 1 and np.array_equal(np.float32(g.min_pt), box[0]) and np.array_equal(np.float32(g.transform),
                                                                                                ROTATED.reshape(12))
        check(ctx.process_mono8(frame), want(crop, box, "crop"), "on", ctx.last_cloud)
        ctx.set_crop_box([-inf, -inf, 0.0], [inf, inf, inf], np.vstack([ROTATED, [0, 0, 0, 1]]))  # half-open, 4x4
        check(ctx.process_mono8(frame), want(crop, ([-inf, -inf, 0.0], [inf, inf, inf], ROTATED), "crop"), "half-open",
              ctx.last_cloud)
        with pytest.raises(ValueError):
            ctx.set_crop_box([0] * 3, [1] * 3, np.eye(4) * 2)
        ctx.set_crop_box(None)
        assert ctx.get_crop_box().enabled == 0
        n0 = ctx.launch_count()
        assert ctx.process_mono8(frame).tobytes() == crop.tobytes()
        assert ctx.last_cloud.is_dense == 0
        assert ctx.launch_count() - n0 == n_crop  # the same launches as before the box was ever set


def test_a_setting_changed_after_submit_does_not_reach_the_pending_slot(env):
    d2pc, ctx, pin, reg = env
    q = ctx.get_q()
    frames = [synth.s2_scene(480, 752, 70 + i) for i in range(3)]
    crops = [crop_of(f, q) for f in frames]
    boxes = [box_for(crops[0], frac, ROTATED) for frac in (0.8, 0.4, 0.1)]
    try:
        for i in range(3):
            ctx.set_crop_box(*boxes[i])
            ctx.submit(i, frames[i])
        ctx.set_crop_box(None)
        for i in range(3):
            check(ctx.wait(i), want(crops[i], boxes[i], "crop"), ("pending", i), ctx.last_cloud)
    finally:
        reset(d2pc, ctx)


def test_node1_crop_box_params_through_the_launch_file(tmp_path):
    from disparity_to_point_cloud_b200 import build
    build.build()
    harness = build.build_harness()
    q = oracle.q_from_intrinsics()
    pose = dict(tx=0.1, ty=-0.3, tz=-1.0, roll=0.05, pitch=-0.1, yaw=0.2)
    lims = dict(min_x=-1.0, min_y=-0.6, min_z=0.0, max_x=1.2, max_y=0.4, max_z=2.5)
    params = "".join(f'    <param name="crop_box_{k}" value="{v}"/>\n' for k, v in {**pose, **lims}.items())
    launch = tmp_path / "box.launch"
    launch.write_text('<launch>\n  <node name="disparity_to_point_cloud" pkg="disparity_to_point_cloud" '
                      'type="disparity_to_point_cloud_node">\n'
                      '    <remap from="/disparity" to="/throttled_depth_map"/>\n'
                      '    <param name="crop_box_enable" value="1"/>\n' + params +
                      '    <param name="radius_outlier_radius" value="0.1"/>\n  </node>\n</launch>\n')
    img = synth.s2_scene(480, 752, 51)
    raw, out = tmp_path / "in.raw", tmp_path / "cloud.bin"
    raw.write_bytes(img.tobytes())
    subprocess.run([harness, "node1", str(launch), "752", "480", str(raw), str(out), "1700000000", "250"], check=True)
    t = transform_of((pose["roll"], pose["pitch"], pose["yaw"]), (pose["tx"], pose["ty"], pose["tz"]))
    box = ([lims["min_x"], lims["min_y"], lims["min_z"]], [lims["max_x"], lims["max_y"], lims["max_z"]], t)
    data, _ = want(oracle.disparity_cb_mono8(img, q), box, "crop", (0.1, 1))
    assert len(data) > 0
    wire = oracle.serialize_pointcloud2(np.frombuffer(data, np.uint8), seq=0, sec=1700000000, nsec=250, is_dense=1)
    assert out.read_bytes() == wire


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
    t = None if rng.random() < 0.3 else transform_of(rng.uniform(-np.pi, np.pi, 3), rng.normal(0, 1, 3))
    frac = float(rng.choice([1.0, 0.5, 0.1, 0.01]))
    box = box_for(crop, frac, t, rng)
    if rng.random() < 0.15:  # half-open along one axis
        a = int(rng.integers(0, 3))
        box[0][a] = -np.inf if rng.random() < 0.5 else box[0][a]
        box[1][a] = np.inf
    desc = dict(case=case, w=w, h=h, mono=mono, q=qkind, mode=mode, grid=grid, ror=rr, frac=frac,
                rotated=t is not None, entry=entry)
    wv = want(crop, box, mode, rr, grid)
    set_mode(d2pc, ctx, mode, grid)
    ctx.set_radius_outlier(*(rr or (0.0,)))
    ctx.set_crop_box(*box)
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
                wf = wv if f == 0 else want(crop_of(frames[1], q), box, mode, rr, grid)
                check(pts[f * stride: f * stride + cnt[f] * 16], wf, (desc, f))
        else:
            got, cl = run_entry(d2pc, ctx, pin, reg, frame, entry, max(len(wv[0]), 16) + 64)
            check(got, wv, desc, cl)
    finally:
        reset(d2pc, ctx)
    n_fin = int(np.isfinite(crop.view(np.float32).reshape(-1, 4)[:, :3]).all(1).sum())
    return desc, len(box_ref.crop_box(crop, *box)) // 16, n_fin


def test_crop_box_fuzz_against_reference(env):
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
    print(f"crop box fuzz: {N_FUZZ} cases from seed {SEED0}, {len(seen)} (mode, entry) classes, "
          f"{partial} with some points kept and some dropped")
