"""GPU parity: depth_map_fusion's merge (rotate + crop + gradFilter + median 3 + trim) vs the oracle and
the cv2-generated fixtures, the exhaustive gradFilter table, and config 5's fuse -> reproject chain."""
import numpy as np
import pytest

import oracle
from conftest import assert_same_bits, golden
from disparity_to_point_cloud_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import disparity_to_point_cloud_b200 as d2pc
    with d2pc.Context(offset_x=-7, offset_y=15) as c:
        yield c


def _four(h, w, seed):
    rng = np.random.default_rng(seed)
    d1 = synth.s2_scene(h, w, seed)
    d2 = synth.s2_scene(h, w, seed + 100)
    s1 = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    s2 = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    return d1, d2, s1, s2


def test_geometry_table(ctx):
    # SURVEY.md A.6
    st, r1, r2, rc, dims = ctx.fuse_geometry(1280, 720)
    assert st == 0 and r1 == (277, 15, 705, 705) and r2 == (7, 261, 705, 705) and rc == (280, 0, 705, 705)
    assert dims == (705, 665, 665)
    st, r1, r2, rc, dims = ctx.fuse_geometry(640, 480)
    assert st == 0 and r1 == (77, 15, 465, 465) and r2 == (7, 61, 465, 465) and rc == (80, 0, 465, 465)


def test_fusion_cv2_fixtures(ctx):
    g = golden("fusion_golden.npz")
    for i in range(3):
        ox, oy = (int(v) for v in g[f"off_{i}"])
        ctx.set_tuning("offset_x", ox)
        ctx.set_tuning("offset_y", oy)
        fused, combined = ctx.fuse(g[f"d1_{i}"], g[f"d2_{i}"], g[f"s1_{i}"], g[f"s2_{i}"])
        assert_same_bits(fused, g[f"fused_{i}"], f"fused #{i}")
        assert_same_bits(combined, g[f"combined_{i}"], f"combined #{i}")
    ctx.set_tuning("offset_x", -7)
    ctx.set_tuning("offset_y", 15)


@pytest.mark.parametrize("w,h", [(1280, 720), (640, 480), (752, 480), (300, 333)])
def test_fusion_vs_oracle(ctx, w, h):
    d1, d2, s1, s2 = _four(h, w, 3)
    fused, combined = ctx.fuse(d1, d2, s1, s2)
    of, oc = oracle.fuse(d1, d2, s1, s2, -7, 15)
    assert_same_bits(fused, of, "fused")
    assert_same_bits(combined, oc, "combined")


def test_exhaustive_grad_filter_over_d1_d2(ctx):
    """All 65,536 (d1,d2) pairs x several score pairs through the kernel, against the oracle's scalar
    gradFilter -- covers the (4k,5k) ratio quirk (SURVEY.md A.5) and division by zero.  The median and the
    border trim are switched off so that every raw merge output is visible."""
    keys = {"offset_x": 0, "offset_y": 0, "fuse_median_ksize": 1, "fuse_crop_right": 0, "fuse_crop_top": 0,
            "fuse_crop_bottom": 0}
    restore = {"offset_x": -7, "offset_y": 15, "fuse_median_ksize": 3, "fuse_crop_right": 40, "fuse_crop_top": 30,
               "fuse_crop_bottom": 10}
    for k, v in keys.items():
        ctx.set_tuning(k, v)
    try:
        n = 256
        dd1, dd2 = np.meshgrid(np.arange(n, dtype=np.uint8), np.arange(n, dtype=np.uint8), indexing="ij")
        src2 = np.ascontiguousarray(np.rot90(dd2, 1))   # the kernel reads map 2 rotated clockwise: cropped_2 == dd2
        # gradFilter sees the scores only through s1<s2, s2<s1, s<100, s<125: these 36 pairs hit every class
        levels = [0, 99, 100, 124, 125, 255]
        for sc1, sc2 in [(a, b) for a in levels for b in levels] + [(110, 110), (10, 20), (20, 10)]:
            s1 = np.full((n, n), sc1, np.uint8)
            s2 = np.full((n, n), sc2, np.uint8)
            want = oracle.grad_filter_table(sc1, sc2)
            fused, combined = ctx.fuse(dd1, src2, s1, s2)
            assert_same_bits(fused, want, f"scores {sc1},{sc2}")
            assert np.all(combined == min(sc1, sc2))
        # and with the reference's median 3 + trim on top
        for k in ("fuse_median_ksize", "fuse_crop_right", "fuse_crop_top", "fuse_crop_bottom"):
            ctx.set_tuning(k, restore[k])
        s1 = np.full((n, n), 110, np.uint8)
        want = oracle.grad_filter_table(110, 110)
        fused, _ = ctx.fuse(dd1, src2, s1, s1)
        assert_same_bits(fused, oracle.median_blur(want, 3)[30:n - 10, 0:n - 40], "median + trim")
    finally:
        for k, v in restore.items():
            ctx.set_tuning(k, v)


@pytest.mark.parametrize("rule", range(1, 8))
def test_alternate_rules(ctx, rule):
    d1, d2, s1, s2 = _four(240, 320, 4)
    ctx.set_tuning("fuse_rule", rule)
    try:
        fused, _ = ctx.fuse(d1, d2, s1, s2)
    finally:
        ctx.set_tuning("fuse_rule", 0)
    of, _ = oracle.fuse(d1, d2, s1, s2, -7, 15, mode=rule)
    assert_same_bits(fused, of, f"rule {rule}")


def test_bad_geometry_is_an_error(ctx):
    import ctypes as C
    import disparity_to_point_cloud_b200 as d2pc
    ctx.set_tuning("offset_y", 400)
    try:
        with pytest.raises(d2pc.D2pcError) as e:
            ctx.fuse(*_four(100, 120, 5))
        assert e.value.status == -7
    finally:
        ctx.set_tuning("offset_y", 15)
    # 20000 x 20000 frames fuse into a 19865^2-point cloud, more bytes than PointCloud2's uint32 row_step holds: both
    # slot entries refuse it before they read an input (all four pointers name one 64-byte buffer) or allocate
    tiny = np.zeros(64, np.uint8)
    p = tiny.ctypes.data
    assert d2pc.lib().d2pc_submit_fusion(ctx._h, 0, p, p, p, p, 20000, 20000, 20000, 1) == -3
    assert d2pc.lib().d2pc_fuse_then_process(ctx._h, p, p, p, p, 20000, 20000, 20000, C.byref(d2pc.Cloud())) == -3


def _expected_cloud(crop, mode):
    """The cloud the filter mode publishes from the CROP cloud, and its is_dense."""
    return (crop, 0) if mode == "crop" else (oracle.filter_finite(crop), 1)


@pytest.fixture(params=["crop", "finite"])
def mode(request, ctx):
    import disparity_to_point_cloud_b200 as d2pc
    ctx.set_filter_mode({"crop": d2pc.FILTER_CROP, "finite": d2pc.FILTER_CROP_FINITE}[request.param])
    yield request.param
    ctx.set_filter_mode(d2pc.FILTER_CROP)


@pytest.mark.parametrize("direct", [0, -1])
def test_config5_fuse_then_reproject(ctx, mode, direct):
    """BASELINE config 5: four 1280x720 maps -> 665x665 fused -> DisparityCb -> 585x585 points (direct 0: the
    callback kernel stores the cloud into the pinned buffer itself; -1: device buffer + D2H copy), in CROP and
    CROP_FINITE mode."""
    q = golden("q_golden.npz")["q"][0]
    d1, d2, s1, s2 = _four(720, 1280, 6)
    ctx.set_tuning("direct_out", direct)
    try:
        got = ctx.fuse_then_process(d1, d2, s1, s2)
    finally:
        ctx.set_tuning("direct_out", 0)
    fused, _ = oracle.fuse(d1, d2, s1, s2, -7, 15)
    assert fused.shape == (665, 665)
    crop = oracle.disparity_cb_mono8(fused, q)
    assert crop.size == 342225 * 16
    want, dense = _expected_cloud(crop, mode)
    assert_same_bits(got, want, f"config 5 {mode}")
    assert ctx.last_cloud.is_dense == dense


def _node_pass_oracle(d1, d2, s1, s2, q, preprocess):
    """MatchingScoreCb1/2 (when preprocess) -> DisparityCb1/2 -> publishFusedDepthMap -> DisparityCb, by the oracle."""
    from oracle import nodes
    if not preprocess:
        fused, _ = oracle.fuse(d1, d2, s1, s2, -7, 15)
    else:
        o = nodes.FusionNodeOracle(-7, 15)
        o.callback(3, s1), o.callback(4, s2), o.callback(1, d1)
        fused = [m for m in o.callback(2, d2) if m[0] == "/fused_depth_map"][0][2]
    return oracle.disparity_cb_mono8(np.ascontiguousarray(fused), q)


@pytest.mark.parametrize("h,w", [(480, 752), (330, 430)])   # rows that are / are not 16-byte multiples
@pytest.mark.parametrize("preprocess", [True, False])
def test_fusion_pipeline_slots_and_stream(ctx, mode, preprocess, h, w):
    """d2pc_submit_fusion / d2pc_process_fusion_stream: whole node passes (the four callbacks + DisparityCb on the
    fused map) overlapped on the slot pipeline; clouds in order, bit-identical to the oracle's node, in CROP and
    CROP_FINITE mode."""
    import disparity_to_point_cloud_b200 as d2pc
    q = golden("q_golden.npz")["q"][0]
    n_sets = 5
    pin = d2pc.PinnedArray((n_sets, 4, h, w), np.uint8)
    rng = np.random.default_rng(77)
    for i in range(n_sets):
        pin.array[i, 0], pin.array[i, 1] = synth.s2_scene(h, w, 300 + i), synth.s2_scene(h, w, 400 + i)
        pin.array[i, 2] = rng.integers(0, 256, (h, w), dtype=np.uint8)
        pin.array[i, 3] = rng.integers(0, 256, (h, w), dtype=np.uint8)
    want = [_expected_cloud(_node_pass_oracle(*pin.array[i], q, preprocess), mode) for i in range(n_sets)]
    dense = []
    clouds = ctx.process_fusion_stream(pin.array, preprocess_scores=preprocess, n_sets=2 * n_sets,
                                       sink=lambda i, c: dense.append(c.is_dense))
    assert len(clouds) == 2 * n_sets
    for i, c in enumerate(clouds):
        assert_same_bits(c, want[i % n_sets][0], f"stream set {i}")
        assert dense[i] == want[i % n_sets][1], f"stream set {i}"
    # explicit slots, pageable frames, waited out of order
    a = [np.array(pin.array[0, k]) for k in range(4)]
    b = [np.array(pin.array[3, k]) for k in range(4)]
    ctx.submit_fusion(0, *a, preprocess_scores=preprocess)
    ctx.submit_fusion(1, *b, preprocess_scores=preprocess)
    assert_same_bits(ctx.wait(1), want[3][0], "slot 1")
    assert ctx.last_cloud.is_dense == want[3][1]
    assert_same_bits(ctx.wait(0), want[0][0], "slot 0")
    assert ctx.last_cloud.is_dense == want[0][1]
    pin.free()


def test_debug_colouriser(ctx):
    """DepthMapFusion::colorizeDepth: every gray level, and a scene."""
    ramp = np.tile(np.arange(256, dtype=np.uint8), (3, 1))
    assert_same_bits(ctx.colorize_depth(ramp), oracle.colorize_depth(ramp), "all gray levels")
    img = synth.s2_scene(211, 333, 8)
    got = ctx.colorize_depth(img)
    assert_same_bits(got, oracle.colorize_depth(img), "scene")
    assert np.all(got[img == 0] == 0)     # black stays black
