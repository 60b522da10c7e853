"""The oracle against the reference's OWN code: oracle/_ref/libd2pc_ref.so is the original project's
src/depth_map_fusion.cpp and src/disparity_to_point_cloud.cpp compiled unmodified against stand-in headers
(oracle/ref_stubs/ref_stubs.hpp says what is reference code and what is a stand-in).  These tests pin the C restatement
(oracle/d2pc_oracle.c) and the sequence oracle (oracle/nodes.py) to that compiled code: gradFilter and the seven
alternate rules, cropToSquare (offset_y_ quirk included), cropMat, rotateMat, colorizeDepth, the callback state machine
with its cv::Mat aliasing, and DisparityCb's crop loop / cloud metadata.  CPU only.

The original project's sources are not part of this repository, so every answer the oracle gives here is also pinned by
digest in tests/golden/ref_compiled.json.  Without oracle/_ref the oracle is held to those digests; with it, the
compiled reference is compared with the oracle as well.  D2PC_RECORD_REF_GOLDEN=1 rewrites the file from the oracle's
answers, and records whether the compiled reference was there to agree with them."""
import contextlib
import hashlib
import json
import os

import numpy as np
import pytest

import oracle
from conftest import GOLDEN
from oracle import nodes, ref

REF = ref.build() is not None
needs_ref = pytest.mark.skipif(not REF, reason="the original project's sources are absent and oracle/_ref is not prebuilt")

STORE = os.path.join(GOLDEN, "ref_compiled.json")
RECORD = os.environ.get("D2PC_RECORD_REF_GOLDEN") == "1"
_digests = {} if RECORD else json.load(open(STORE))["digests"]


def digest(*parts):
    """SHA-256 over the dtype, shape and bytes of each part (arrays, tuples of ints, str, bytes)."""
    h = hashlib.sha256()
    for p in parts:
        a = np.frombuffer(p.encode() if isinstance(p, str) else p, np.uint8) if isinstance(p, (str, bytes)) \
            else np.ascontiguousarray(p)
        h.update(f"{a.dtype.str}{a.shape};".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def expect(key, *parts):
    """The oracle's answer for `key` is the one the compiled reference gave (stored in ref_compiled.json)."""
    d = digest(*parts)
    if RECORD:
        _digests[key] = d
    else:
        assert d == _digests[key], f"{key}: the oracle's answer differs from the one stored in {STORE}"


@pytest.fixture(scope="module", autouse=True)
def _record():
    yield
    if RECORD:
        with open(STORE, "w") as f:
            json.dump({"checked_against_compiled_reference": REF, "digests": dict(sorted(_digests.items()))}, f,
                      indent=1)
            f.write("\n")


@pytest.fixture(scope="module")
def fusion():
    """The reference's DepthMapFusion at the launch offsets, or None where oracle/_ref is absent."""
    if not REF:
        yield None
        return
    with ref.FusionNode(-7, 15) as n:
        yield n


@needs_ref
def test_constructor_topics_queues_and_params(fusion):
    """depth_map_fusion.hpp:97-124 as the reference's constructor registers them."""
    assert fusion.offsets() == (-7, 15) and fusion.warnings == 0
    assert fusion.subscribed == [("/disparity_1", 1, False), ("/disparity_2", 1, False), ("/matching_score_1", 1, False),
                                 ("/matching_score_2", 1, False)]
    assert fusion.advertised == [(t, 5, False) for t in ("/cropped_depth_1", "/cropped_depth_2", "/cropped_score_1",
                                                         "/cropped_score_2", "/fused_depth_map", "/combined_score",
                                                         "/gradient")]
    with ref.FusionNode() as bare:  # no params on the server: two ROS_WARNs, offsets stay 0 (hpp:76-77, :119-124)
        assert bare.offsets() == (0, 0) and bare.warnings == 2


@pytest.mark.parametrize("s1,s2", [(0, 0), (99, 100), (100, 99), (100, 100), (110, 110), (124, 124), (125, 124),
                                   (124, 125), (125, 125), (50, 200), (200, 50), (255, 255), (99, 99)])
def test_grad_filter_exhaustive_against_the_reference(fusion, s1, s2):
    """All 65,536 (d1, d2) per score pair, src/depth_map_fusion.cpp:219-235 (the (4k, 5k) float quirk included)."""
    tab = oracle.grad_filter_table(s1, s2)
    expect(f"grad_filter {s1} {s2}", tab)
    if fusion is not None:
        L = ref.lib()
        got = np.array([[L.ref_grad_filter(fusion._h, a, b, s1, s2, s1, s2) for b in range(256)] for a in range(0, 256, 1)],
                       dtype=np.int64)
        assert np.array_equal(got & 255, tab)
        assert got.min() >= 0 and got.max() <= 255


def test_numpy_grad_filter_is_the_c_oracle():
    """oracle/nodes.py vectorises gradFilter in numpy; it must be the same function as the C table."""
    dd1, dd2 = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    for s1, s2 in [(0, 0), (99, 100), (100, 99), (110, 110), (124, 124), (125, 124), (124, 125), (50, 200), (200, 50), (255, 0)]:
        got = nodes.grad_filter_np(dd1, dd2, np.full_like(dd1, s1), np.full_like(dd1, s2))
        assert np.array_equal(got, oracle.grad_filter_table(s1, s2)), (s1, s2)


def test_alternate_rules_against_the_reference(fusion):
    """src/depth_map_fusion.cpp:169-217, modes 1..7 of d2pc_fuse_rule."""
    rng = np.random.default_rng(3)
    cases = [(a, b, c, d) for a in (0, 1, 37, 128, 229, 230, 255) for b in (0, 1, 99, 150, 255) for c in (0, 19, 20, 49, 50, 99, 100, 255)
             for d in (0, 19, 20, 49, 50, 99, 100, 255)]
    cases += [tuple(int(v) for v in rng.integers(0, 256, 4)) for _ in range(3000)]
    for mode in range(1, 8):
        want = [oracle.fuse_rule(mode, a, b, c, d) for a, b, c, d in cases]
        expect(f"fuse_rule {mode}", np.array(want, dtype=np.int64))
        if fusion is not None:
            for (a, b, c, d), w in zip(cases, want):
                assert fusion.fuse_rule(mode, a, b, c, d) == w, (mode, a, b, c, d)


def test_crop_to_square_sweep(fusion):
    """src/depth_map_fusion.cpp:247-265 incl. the member offset_y_ (= 15 here) read at :252-253, and the cases
    where cv::Mat::operator()(Rect) throws."""
    answers, n_bad = [], 0
    for cols, rows in [(1280, 720), (720, 1280), (752, 480), (480, 752), (640, 480), (200, 150), (150, 200), (100, 100),
                       (31, 90), (90, 31)]:
        for ox in (-40, -7, 0, 5, 7, 33):
            for oy in (-30, -15, 0, 9, 15, 28):
                orc, orr = oracle.crop_to_square(cols, rows, ox, oy, 15)
                answers.append((orc == 0,) + (orr if orc == 0 else (0, 0, 0, 0)))
                n_bad += orc != 0
                if fusion is not None:
                    rc, r = fusion.crop_to_square(cols, rows, ox, oy)
                    assert (rc == 0) == (orc == 0), (cols, rows, ox, oy, rc, orc)
                    if rc == 0:
                        assert r == orr, (cols, rows, ox, oy)
    expect("crop_to_square", np.array(answers, dtype=np.int64))
    assert n_bad > 0  # the sweep does reach rectangles that leave the image


def test_crop_mat_and_rotate(fusion):
    if fusion is not None:
        assert fusion.crop_mat(705, 705, 0, 40, 30, 10) == (0, (0, 30, 665, 665))  # :130
        assert fusion.crop_mat(50, 40, 3, 4, 5, 6) == (0, (3, 5, 43, 29))
        assert fusion.crop_mat(30, 30, 0, 40, 30, 10)[0] != 0
    rng = np.random.default_rng(5)
    for h, w in [(5, 9), (64, 48), (33, 33)]:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        want = oracle.rotate_cw(img)
        expect(f"rotate {h}x{w}", want)
        if fusion is not None:
            assert np.array_equal(fusion.rotate(img), want)  # :268-273


def test_colorize_depth_every_gray_level(fusion):
    gray = np.arange(256, dtype=np.uint8).reshape(16, 16)
    want = oracle.colorize_depth(gray)
    expect("colorize_depth", want)
    if fusion is not None:
        assert np.array_equal(fusion.colorize(gray), want)  # :304-358


def _same(pubs, want):
    if len(pubs) != len(want):
        return False
    for p, (topic, enc, arr, hdr) in zip(pubs, want):
        if p.topic != topic or p.encoding != enc or (p.seq, p.sec, p.nsec) != hdr or not np.array_equal(p.image(), arr):
            return False
    return True


@pytest.mark.parametrize("h,w,ox,oy", [(150, 200, -7, 15), (160, 120, 5, -9), (130, 130, 0, 0)])
def test_callback_sequences_with_aliased_score_state(h, w, ox, oy):
    """Every message of a 16-callback run, the reference's class vs oracle/nodes.py.  The run fires DisparityCb2
    before the caches are full (no fused publish), twice in a row (the second pass reads score 1 = min(score 1,
    score 2) left behind by the first, :77, :113, :118-121), and again after fresh scores."""
    rng = np.random.default_rng(h * 1000 + w)
    seq = [2, 1, 3, 2, 4, 2, 2, 2, 3, 2, 4, 4, 2, 1, 2, 3]
    parts = []
    with (ref.FusionNode(ox, oy) if REF else contextlib.nullcontext()) as n:
        o = nodes.FusionNodeOracle(ox, oy)
        n_fused = 0
        for step, which in enumerate(seq):
            base = rng.integers(0, 256, (h, w), dtype=np.uint8)
            img = base if which in (3, 4) else (base // 2 + 40).astype(np.uint8)
            hdr = (step, 100 + step, 7 * step)
            want = o.callback(which, img, hdr)
            for topic, enc, arr, hd in want:
                parts += [topic, enc, hd, arr]
            if n is not None:
                rc, pubs = n.callback(which, img, *hdr)
                assert rc == 0
                assert _same(pubs, want), (step, which, [p.topic for p in pubs])
            n_fused += sum(topic == "/fused_depth_map" for topic, *_ in want)
        assert n_fused == 6
    expect(f"callback sequence {h}x{w} {ox} {oy}", *parts)


def test_score_chain_blur_path_follows_the_submatrix_flag():
    """A square frame with zero offsets makes cropToSquare return the whole image: not a submatrix, so the first
    GaussianBlur takes OpenCV's fixed-point path; any real crop takes sepFilter2D (ADVICE r1).  The compiled
    reference decides through cv::Mat's flag, the oracle through its rectangle test: they must agree."""
    rng = np.random.default_rng(11)
    parts = []
    for h, w, ox, oy in [(96, 96, 0, 0), (96, 96, 3, 0), (96, 128, 0, 0)]:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        rc0, r = oracle.crop_to_square(w, h, ox, oy, oy)
        want = oracle.score_preprocess(img, r, False)
        parts.append(want)
        if REF:
            with ref.FusionNode(ox, oy) as n:
                rc, pubs = n.callback(3, img)
                assert rc == 0
                assert np.array_equal(pubs[0].image(), want)
    expect("score chain blur path", *parts)


@needs_ref
def test_bad_encoding_is_the_uncaught_cv_bridge_exception(fusion):
    rc, pubs = fusion.callback(1, np.zeros((50, 60), np.uint8), encoding="32FC1")
    assert rc == -2 and pubs == []


@pytest.mark.parametrize("params", [{}, {"fx_": 700.0, "fy_": 650.5, "cx_": 300.25, "cy_": 250.0, "base_line_": 0.043}])
def test_disparity_cb_of_the_reference_node(params):
    """src/disparity_to_point_cloud.cpp:46-92 compiled from the reference: crop loop, PointXYZ packing, cloud
    metadata, header; disparity_to_point_cloud.hpp:77-81 topics (the publisher is latched: `this` as the flag)."""
    from disparity_to_point_cloud_b200 import synth
    q = oracle.q_from_intrinsics(*(params.get(k, d) for k, d in (("fx_", 714.24), ("fy_", 713.5), ("cx_", 376.0),
                                                                   ("cy_", 240.0), ("base_line_", 0.09))))
    wires = []
    with (ref.D2pcNode(**params) if REF else contextlib.nullcontext()) as n:
        if n is not None:
            assert n.subscribed == [("/disparity", 1, False)] and n.advertised == [("/point_cloud", 1, True)]
        for h, w, seed in [(120, 136, 1), (97, 101, 2), (80, 200, 3), (81, 81, 4)]:
            img = synth.s2_scene(h, w, seed)
            want = oracle.disparity_cb_mono8(img, q)
            # the wire image of the cloud the reference publishes for this frame
            wire = oracle.serialize_pointcloud2(want, seq=0, sec=1700000000, nsec=42)
            wires.append(wire)
            if n is None:
                continue
            rc, pubs = n.callback(img, seq=5, sec=1700000000, nsec=42)
            assert rc == 0 and len(pubs) == 1
            c = pubs[0]
            assert c.topic == "/point_cloud" and c.is_cloud and c.latched and c.queue == 1
            assert c.data.tobytes() == want.tobytes()
            npts = oracle.n_points(w, h)
            assert (c.width, c.height, c.point_step, c.row_step, c.is_dense) == (npts, 1, 16, 16 * npts, 0)
            assert c.fields == [("x", 0, 7, 1), ("y", 4, 7, 1), ("z", 8, 7, 1)]
            assert c.frame_id == "/camera_optical_frame" and (c.sec, c.nsec) == (1700000000, 42)
            assert wire == oracle.serialize_pointcloud2(c.data, seq=0, sec=1700000000, nsec=42, frame_id=c.frame_id,
                                                        is_dense=c.is_dense)
    expect("disparity_cb " + ("custom intrinsics" if params else "default intrinsics"), *wires)
