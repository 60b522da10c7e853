"""GPU parity: the whole DisparityCb on mono8 frames (median 11 -> x1/8 -> reproject -> crop -> pack),
the median kernel on its own, the slot pipeline and the wire serialisation."""
import numpy as np
import pytest

import oracle
from conftest import assert_same_bits, golden
from disparity_to_point_cloud_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import disparity_to_point_cloud_b200 as d2pc
    with d2pc.Context() as c:
        yield c


@pytest.fixture(scope="module")
def q():
    return golden("q_golden.npz")["q"][0]


def test_callback_golden_fixtures(ctx):
    g = golden("callback_golden.npz")
    ctx.set_q(g["q"])
    for i in range(3):
        assert_same_bits(ctx.process_mono8(g[f"img{i}"]), g[f"cloud{i}"], f"cv2 fixture #{i}")


@pytest.mark.parametrize("w,h,kind", [(752, 480, "s2"), (640, 480, "s1"), (1280, 720, "s2"), (665, 665, "s1"),
                                      (81, 81, "s1"), (131, 203, "s2"), (80, 80, "s1")])
@pytest.mark.parametrize("fuse", [0, -1])
def test_mono8_callback_bit_exact(ctx, q, w, h, kind, fuse):
    """fuse 0: the default, median + x 1/8 + reproject + pack as ONE launch (the default Q allows it); -1: the
    two-launch form (median image, then the reprojection kernel) every other Q / filter mode takes."""
    img = synth.s2_scene(h, w, 11) if kind == "s2" else synth.s1_uniform(h, w, 11)
    ctx.set_tuning("fuse_median", fuse)
    try:
        n0 = ctx.launch_count()
        assert_same_bits(ctx.process_mono8(img), oracle.disparity_cb_mono8(img, q), f"{w}x{h} {kind}")
        if (w - 80) * (h - 80) > 0:
            assert ctx.launch_count() - n0 == (1 if fuse == 0 else 2)
    finally:
        ctx.set_tuning("fuse_median", 0)


def test_fused_callback_other_q_and_knobs(ctx, q):
    """The fused launch only exists for the plain rectified arithmetic; anything else must quietly take two launches
    and give the same bytes: q33 != 0, a generic Q, the Markstein variant, CROP_FINITE (a Q with an integral principal
    point stays fused: X == 0 on the column u == 250, Y == 0 on the row v == 150, 0 / 0 where the byte is 0 too).  Plus the fused path itself on bytes whose disparity is 0 (W = +0:
    +-inf and, on the row v == 240 of the default Q, NaN) and with a narrow border."""
    import disparity_to_point_cloud_b200 as d2pc
    img = synth.s2_scene(300, 500, 21)
    img[120:130, :] = 0
    img[:, 250] = 0
    for ks in (5, 11, 15):
        ctx.set_tuning("median_ksize", ks)
        try:
            want = oracle.crop_pack(oracle.reproject_image_to_3d(oracle.convert_u8_f32(oracle.median_blur(img, ks)), q))
            assert_same_bits(ctx.process_mono8(img), want, f"fused, ksize {ks}")
        finally:
            ctx.set_tuning("median_ksize", 11)
    ctx.set_tuning("border", 2)
    try:
        want = oracle.crop_pack(oracle.reproject_image_to_3d(oracle.convert_u8_f32(oracle.median_blur(img, 11)), q), 2)
        assert_same_bits(ctx.process_mono8(img), want, "fused, border 2 (replicate edge inside the window)")
    finally:
        ctx.set_tuning("border", 40)
    qi = np.array([[1, 0, 0, -250.0], [0, 1, 0, -150.0], [0, 0, 0, 713.5], [0, 0, 1 / 0.09, 0.0]])
    qw = q.copy()
    qw[3, 3] = 0.37
    qg = golden("reproject_golden.npz")["q_generic"]
    try:
        for name, qq, knobs, launches in (("integral principal point", qi, {}, 1), ("q33 != 0", qw, {}, 2),
                                          ("integral principal point, ordinary kernels", qi, {"zero_numer": -1}, 1),
                                          ("generic", qg, {}, 2), ("Markstein", q, {"exact_variant": 1}, 2),
                                          ("forced generic", q, {"force_generic": 1}, 2)):
            ctx.set_q(qq)
            for k, v in knobs.items():
                ctx.set_tuning(k, v)
            try:
                n0 = ctx.launch_count()
                assert_same_bits(ctx.process_mono8(img), oracle.disparity_cb_mono8(img, qq), name)
                assert ctx.launch_count() - n0 == launches, name
            finally:
                for k in knobs:
                    ctx.set_tuning(k, 0)
        ctx.set_q(q)
        ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
        assert_same_bits(ctx.process_mono8(img), oracle.filter_finite(oracle.disparity_cb_mono8(img, q)), "CROP_FINITE")
    finally:
        ctx.set_filter_mode(d2pc.FILTER_CROP)
        ctx.set_q(q)


def test_mono8_strided_message(ctx, q):
    """sensor_msgs/Image.step larger than width (A1: honour step)."""
    buf = synth.s2_scene(300, 512, 12)
    view = buf[:, 7:407]
    assert_same_bits(ctx.process_mono8(view), oracle.disparity_cb_mono8(np.ascontiguousarray(view), q), "step")


def test_mono8_4k(ctx, q):
    img = synth.s2_scene(2160, 3840, 13)
    assert_same_bits(ctx.process_mono8(img), oracle.disparity_cb_mono8(img, q), "4K mono8")


@pytest.mark.parametrize("variant", [0, 2])
@pytest.mark.parametrize("ksize", [3, 5, 7, 9, 11, 13, 15])
@pytest.mark.parametrize("w,h", [(96, 64), (7, 5), (333, 222), (32, 300), (1, 40), (40, 1), (700, 37)])
def test_median_kernel_full_frame(ctx, ksize, w, h, variant):
    """variant 0: the default (window histogram per output column; 19-exchange selection network for ksize 3);
    2: the window histogram for ksize 3 as well."""
    import torch
    ctx.set_tuning("median_variant", variant)
    img = synth.s1_uniform(h, w, 14 + ksize)
    d_src = torch.from_numpy(img).cuda()
    d_dst = torch.zeros_like(d_src)
    torch.cuda.synchronize()
    ctx.median_u8_device(d_src.data_ptr(), w, h, w, d_dst.data_ptr(), w, ksize)
    ctx.sync()
    ctx.set_tuning("median_variant", 0)
    assert_same_bits(d_dst.cpu().numpy(), oracle.median_blur(img, ksize), f"median {ksize} {w}x{h}")


def test_median_golden_cv2(ctx):
    import torch
    g = golden("median_golden.npz")
    for i in range(4):
        img = g[f"img{i}"]
        h, w = img.shape
        for k in (11, 3):
            d_src = torch.from_numpy(img).cuda()
            d_dst = torch.zeros_like(d_src)
            torch.cuda.synchronize()
            ctx.median_u8_device(d_src.data_ptr(), w, h, w, d_dst.data_ptr(), w, k)
            ctx.sync()
            assert_same_bits(d_dst.cpu().numpy(), g[f"m{k}_{i}"], f"cv2 median {k} #{i}")


@pytest.mark.parametrize("variant", [0, 2])
def test_median_smooth_and_constant(ctx, variant):
    import torch
    ctx.set_tuning("median_variant", variant)
    for img in (np.full((100, 100), 255, np.uint8), np.zeros((64, 64), np.uint8),
                np.tile(np.arange(200, dtype=np.uint8), (120, 1)), synth.s2_scene(480, 752, 15)):
        h, w = img.shape
        d_src = torch.from_numpy(np.ascontiguousarray(img)).cuda()
        d_dst = torch.zeros_like(d_src)
        torch.cuda.synchronize()
        ctx.median_u8_device(d_src.data_ptr(), w, h, w, d_dst.data_ptr(), w, 11)
        ctx.sync()
        assert_same_bits(d_dst.cpu().numpy(), oracle.median_blur(np.ascontiguousarray(img), 11), "median")
    ctx.set_tuning("median_variant", 0)


def test_mono8_device_batch(ctx, q):
    import torch
    f, h, w = 3, 240, 376
    frames = np.stack([synth.s2_scene(h, w, 40 + i) for i in range(f)])
    n = oracle.n_points(w, h)
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.zeros((f, n * 16), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.reproject_mono8_device(d_in.data_ptr(), f, w, h, w, w * h, d_out.data_ptr(), n * 16)
    ctx.sync()
    got = d_out.cpu().numpy()
    for i in range(f):
        assert_same_bits(got[i], oracle.disparity_cb_mono8(frames[i], q), f"frame {i}")


def test_slot_pipeline_and_stream(ctx, q):
    """Config 2 shape: a 752x480 mono8 stream through the 3-slot H2D|kernel|D2H pipeline, order preserved."""
    import disparity_to_point_cloud_b200 as d2pc
    f, h, w = 12, 480, 752
    pin = d2pc.PinnedArray((f, h, w), np.uint8)
    for i in range(f):
        pin.array[i] = synth.s2_scene(h, w, 50 + i)
    clouds = ctx.process_stream(pin.array)
    assert len(clouds) == f
    for i in (0, 1, 5, 11):
        assert_same_bits(clouds[i], oracle.disparity_cb_mono8(pin.array[i], q), f"stream frame {i}")
    # explicit slots, pageable input, out-of-order wait
    a, b = synth.s2_scene(h, w, 70), synth.s1_uniform(h, w, 71)
    ctx.submit(0, a)
    ctx.submit(1, b)
    got_b = ctx.wait(1)
    got_a = ctx.wait(0)
    assert_same_bits(got_a, oracle.disparity_cb_mono8(a, q), "slot 0")
    assert_same_bits(got_b, oracle.disparity_cb_mono8(b, q), "slot 1")
    with pytest.raises(d2pc.D2pcError):
        ctx.wait(2)  # nothing submitted
    pin.free()


def test_caller_supplied_destination(ctx, q):
    """d2pc_process_*_into / d2pc_submit_*_into (SURVEY 8(b) Ownership): the cloud lands in the caller's buffer --
    by DMA when it is page-locked (d2pc_host_alloc or d2pc_host_register), through the library's pinned buffer
    when it is pageable -- and nothing is written past the cloud."""
    import ctypes as C
    import disparity_to_point_cloud_b200 as d2pc
    h, w = 480, 752
    img = synth.s2_scene(h, w, 60)
    want = oracle.disparity_cb_mono8(img, q)
    nb = want.size
    pin = d2pc.PinnedArray((nb + 64,), np.uint8)
    own = np.empty(nb + 64, np.uint8)
    reg = d2pc.RegisteredArray(np.empty(nb + 64, np.uint8))
    try:
        for name, dst in (("pinned", pin.array), ("pageable", own), ("registered", reg.array)):
            dst[:] = 0xAB
            got = ctx.process_into(img, dst)
            assert got.ctypes.data == dst.ctypes.data and got.size == nb
            assert ctx.last_cloud.width == nb // 16 and C.addressof(ctx.last_cloud.data.contents) == dst.ctypes.data
            assert_same_bits(got, want, name)
            assert (dst[nb:] == 0xAB).all(), name
        d = synth.s3_float(h, w, 61)
        assert_same_bits(ctx.process_into(d, pin.array), oracle.disparity_cb_f32(d, q), "float entry")
        # too small: refused at submit in CROP mode, nothing written
        small = np.full(nb - 16, 0xCD, np.uint8)
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.process_into(img, small)
        assert e.value.status == -9 and (small == 0xCD).all()
        # slots: two frames in flight into two caller buffers, waited out of order
        a, b = synth.s2_scene(h, w, 62), synth.s1_uniform(h, w, 63)
        da, db = pin.array[:nb], reg.array[:nb]
        ctx.submit(0, a, dst=da)
        ctx.submit(1, b, dst=db)
        assert_same_bits(ctx.wait(1), oracle.disparity_cb_mono8(b, q), "slot 1")
        assert_same_bits(ctx.wait(0), oracle.disparity_cb_mono8(a, q), "slot 0")
        # CROP_FINITE: the count is only known afterwards; a buffer that holds the kept points is enough
        ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
        try:
            kept = oracle.filter_finite(want)
            assert 0 < kept.size < nb
            own[:] = 0xAB
            got = ctx.process_into(img, own[:kept.size])
            assert_same_bits(got, kept, "compacted into a caller buffer")
            assert (own[kept.size:] == 0xAB).all()
            with pytest.raises(d2pc.D2pcError) as e:
                ctx.process_into(img, own[:kept.size - 16])
            assert e.value.status == -9
        finally:
            ctx.set_filter_mode(d2pc.FILTER_CROP)
        # the library-owned path still works after caller-owned submissions on the same slot
        assert_same_bits(ctx.process_mono8(img), want, "library-owned after into")
    finally:
        pin.free()
        reg.free()


@pytest.mark.parametrize("direct", [-1, 0, 1])
def test_direct_output_modes(ctx, q, direct):
    """direct_out: a CROP cloud is written by the kernel straight into the page-locked host buffer (no D2H copy
    behind the kernel): 0 = synchronous single-frame mono8 entries only (default), 1 = every CROP submission (float
    frames, slots, streams, fusion sets), -1 = never.  Same bytes in every mode, every destination kind, nothing written
    past the cloud."""
    import disparity_to_point_cloud_b200 as d2pc
    ctx.set_tuning("direct_out", direct)
    pin = reg = None
    try:
        for (w, h, seed) in [(752, 480, 80), (640, 480, 81), (131, 203, 82), (81, 81, 83), (80, 80, 84)]:
            img = synth.s2_scene(h, w, seed)
            d = synth.s3_float(h, w, seed)
            assert_same_bits(ctx.process_mono8(img), oracle.disparity_cb_mono8(img, q), f"mono8 {w}x{h}")
            assert_same_bits(ctx.process_f32(d), oracle.disparity_cb_f32(d, q), f"f32 {w}x{h}")
        h, w = 480, 752
        img = synth.s2_scene(h, w, 85)
        want = oracle.disparity_cb_mono8(img, q)
        nb = want.size
        pin = d2pc.PinnedArray((nb + 64,), np.uint8)
        reg = d2pc.RegisteredArray(np.empty(nb + 80, np.uint8))
        own = np.empty(nb + 64, np.uint8)
        # a registered buffer that is not 16-byte aligned takes the copy path whatever the mode
        off = (-reg.array.ctypes.data) % 16 + 4
        for name, dst in (("pinned", pin.array), ("registered", reg.array[:nb + 64]), ("pageable", own),
                          ("registered, unaligned", reg.array[off:off + nb + 32])):
            dst[:] = 0xAB
            got = ctx.process_into(img, dst)
            assert_same_bits(got, want, name)
            assert (dst[nb:] == 0xAB).all(), name
        # slots and a stream (direct only when direct_out = 1), then the two-launch callback and CROP_FINITE
        a, b = synth.s2_scene(h, w, 86), synth.s1_uniform(h, w, 87)
        ctx.submit(0, a, dst=pin.array[:nb])
        ctx.submit(1, b)
        assert_same_bits(ctx.wait(1), oracle.disparity_cb_mono8(b, q), "slot 1")
        assert_same_bits(ctx.wait(0), oracle.disparity_cb_mono8(a, q), "slot 0")
        frames = d2pc.PinnedArray((6, h, w), np.uint8)
        for i in range(6):
            frames.array[i] = synth.s2_scene(h, w, 90 + i)
        clouds = ctx.process_stream(frames.array)
        for i in (0, 3, 5):
            assert_same_bits(clouds[i], oracle.disparity_cb_mono8(frames.array[i], q), f"stream frame {i}")
        frames.free()
        # fusion sets on a slot and in a stream: DisparityCb on the fused map (the context's offsets are 0, 0)
        rng = np.random.default_rng(88)
        sets = np.stack([np.stack([synth.s2_scene(h, w, 96 + i), synth.s2_scene(h, w, 98 + i),
                                   rng.integers(0, 256, (h, w), dtype=np.uint8),
                                   rng.integers(0, 256, (h, w), dtype=np.uint8)]) for i in range(2)])
        fused = [oracle.disparity_cb_mono8(oracle.fuse(*sets[i], 0, 0)[0], q) for i in range(2)]
        ctx.submit_fusion(2, *sets[1], preprocess_scores=False)
        assert_same_bits(ctx.wait(2), fused[1], "fusion slot")
        for i, c in enumerate(ctx.process_fusion_stream(sets, preprocess_scores=False, n_sets=5)):
            assert_same_bits(c, fused[i % 2], f"fusion stream set {i}")
        ctx.set_tuning("fuse_median", -1)
        assert_same_bits(ctx.process_mono8(img), want, "two-launch callback")
        ctx.set_tuning("fuse_median", 0)
        ctx.set_filter_mode(d2pc.FILTER_CROP_FINITE)
        assert_same_bits(ctx.process_mono8(img), oracle.filter_finite(want), "CROP_FINITE is never direct")
        ctx.set_filter_mode(d2pc.FILTER_CROP)
    finally:
        ctx.set_tuning("direct_out", 0)
        ctx.set_tuning("fuse_median", 0)
        ctx.set_filter_mode(d2pc.FILTER_CROP)
        if pin:
            pin.free()
        if reg:
            reg.free()


def test_per_call_timing(q):
    """d2pc_set_timing / d2pc_slot_timing: the device-side spans of one submission (H2D, kernels, D2H) are positive,
    add up to the total, and the call still produces the same bytes; without timing enabled the query says so."""
    import disparity_to_point_cloud_b200 as d2pc
    img = synth.s2_scene(480, 752, 33)
    want = oracle.disparity_cb_mono8(img, q)
    with d2pc.Context() as c:
        c.process_mono8(img)
        with pytest.raises(d2pc.D2pcError) as e:
            c.slot_timing(0)
        assert e.value.status == -8
        c.set_timing(True)
        for _ in range(3):
            assert_same_bits(c.process_mono8(img), want, "timed call")
        t = c.slot_timing(0)
        assert t.points == want.size // 16
        # a synchronous mono8 call stores its cloud from the kernel (direct_out): the transfer is inside the kernel span
        assert t.h2d_us > 0 and t.kernels_us > 40 and 0 <= t.d2h_us < 20 and t.total_us < 5000
        assert abs(t.h2d_us + t.kernels_us + t.d2h_us - t.total_us) < 0.05 * t.total_us + 2
        c.set_tuning("direct_out", -1)  # the three-stage form: H2D, kernels, D2H copy
        for _ in range(2):
            assert_same_bits(c.process_mono8(img), want, "timed call, copy after the kernel")
        t = c.slot_timing(0)
        assert t.h2d_us > 0 and t.kernels_us > 5 and t.d2h_us > 20 and t.total_us < 5000
        assert abs(t.h2d_us + t.kernels_us + t.d2h_us - t.total_us) < 0.05 * t.total_us + 2
        c.set_tuning("direct_out", 0)
        c.submit(1, img)
        c.wait(1)
        assert c.slot_timing(1).kernels_us > 5
        four = [synth.s2_scene(240, 320, 2 + i) for i in range(4)]
        c.submit_fusion(2, *four)
        c.wait(2)
        assert c.slot_timing(2).total_us > 0
        c.set_timing(False)
        assert_same_bits(c.process_mono8(img), want, "after timing was switched off")


def test_float_stream_matches_single_calls(ctx, q):
    f, h, w = 7, 300, 420
    frames = np.stack([synth.s4_stress(h, w, 80 + i) for i in range(f)])
    clouds = ctx.process_stream(frames)
    for i in range(f):
        assert_same_bits(clouds[i], oracle.disparity_cb_f32(frames[i], q), f"frame {i}")


def test_pointcloud2_wire_bytes(ctx, q):
    img = synth.s2_scene(120, 136, 90)
    ctx.process_mono8(img)
    got = ctx.serialize_pointcloud2(ctx.last_cloud, seq=3, sec=1700000000, nsec=123456789)
    want = oracle.serialize_pointcloud2(oracle.disparity_cb_mono8(img, q), seq=3, sec=1700000000, nsec=123456789)
    assert got == want


def test_bad_arguments(ctx):
    import disparity_to_point_cloud_b200 as d2pc
    import ctypes as C
    cl = d2pc.Cloud()
    L = d2pc.lib()
    img = np.zeros((10, 10), np.uint8)
    assert L.d2pc_process_mono8(ctx._h, None, 10, 10, 10, C.byref(cl)) == -1
    assert L.d2pc_process_mono8(ctx._h, img.ctypes.data, 10, 10, 5, C.byref(cl)) == -3   # step < width
    assert L.d2pc_process_mono8(ctx._h, img.ctypes.data, 0, 10, 10, C.byref(cl)) == -3
    assert L.d2pc_submit_mono8(ctx._h, 99, img.ctypes.data, 10, 10, 10) == -1
    assert L.d2pc_set_filter_mode(ctx._h, 7) == -1
    assert L.d2pc_process_mono8_into(ctx._h, img.ctypes.data, 10, 10, 10, None, 0, C.byref(cl)) == -1
    assert L.d2pc_host_register(None, 16) == -1
    # a frame whose cloud would not fit PointCloud2's uint32 width / row_step is refused before anything is touched
    assert L.d2pc_process_mono8(ctx._h, img.ctypes.data, 60000, 60000, 60000, C.byref(cl)) == -3
    assert L.d2pc_reproject_mono8_device(ctx._h, 0x1000, 1, 60000, 60000, 60000, 3600000000, 0x2000, 0, None) == -3
    # an empty batch is a no-op, not an allocation of (0 - 1) frames
    n0 = ctx.launch_count()
    assert L.d2pc_reproject_mono8_device(ctx._h, 0x1000, 0, 752, 480, 752, 752 * 480, 0x2000, 4300800, None) == 0
    assert ctx.launch_count() == n0
    # d2pc_reproject_f32_device: a float pointer that is not 4-byte aligned is refused, not dereferenced
    assert L.d2pc_reproject_f32_device(ctx._h, 0x1001, 1, 100, 100, 400, 40000, 0x2000, 0, None) == -3
