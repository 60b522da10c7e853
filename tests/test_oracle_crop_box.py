"""CPU: the crop box reference tests/box_ref against a numpy float32 restatement of the recipe in
include/d2pc_b200.h, against PCL's CropBox loop restated literally, and against known answers."""
import numpy as np
import pytest

import box_ref


def cloud_of(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    pts = np.zeros((len(xyz), 4), np.float32)
    pts[:, :3] = xyz
    pts[:, 3] = np.arange(len(xyz), dtype=np.float32)  # the pad word travels unchanged
    return pts


def numpy_box(pts, mn, mx, t=None) -> bytes:
    """The recipe with numpy float32: every operation rounded on its own, in the order of rule 2."""
    pts = np.asarray(pts, np.float32).reshape(-1, 4)
    t = box_ref.IDENTITY if t is None else np.asarray(t, np.float32).reshape(3, 4)
    mn, mx = np.asarray(mn, np.float32), np.asarray(mx, np.float32)
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    keep = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
    with np.errstate(invalid="ignore", over="ignore"):
        for a in range(3):
            l = ((t[a, 0] * x + t[a, 1] * y) + t[a, 2] * z) + t[a, 3]
            keep &= (mn[a] <= l) & (l <= mx[a])
    return pts[keep].tobytes()


def rotation(rng) -> np.ndarray:
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    q *= np.sign(np.diag(r))
    return q * np.sign(np.linalg.det(q))


def random_case(rng):
    n = int(rng.integers(0, 4000))
    pts = cloud_of(rng.normal(0, 3, (n, 3)))
    if n:
        k = n // 10
        pts[rng.integers(0, n, k), rng.integers(0, 3, k)] = rng.choice([np.nan, np.inf, -np.inf], k)
    lo = rng.uniform(-4, 2, 3)
    mn, mx = lo, lo + rng.uniform(0.1, 6, 3)
    t = None
    if rng.random() < 0.8:
        t = np.concatenate([rotation(rng), rng.normal(0, 2, (3, 1))], axis=1).astype(np.float32)
    return pts, mn.astype(np.float32), mx.astype(np.float32), t


def test_reference_matches_numpy_and_pcl_on_random_clouds():
    rng = np.random.default_rng(2024)
    partial = 0
    for case in range(300):
        pts, mn, mx, t = random_case(rng)
        want = numpy_box(pts, mn, mx, t)
        assert box_ref.crop_box(pts, mn, mx, t) == want, case
        assert box_ref.pcl(pts, mn, mx, t) == want, case
        partial += 0 < len(want) < 16 * np.isfinite(pts[:, :3]).all(1).sum()
    assert partial > 200


def test_points_on_every_face_are_inside():
    mn, mx = np.float32([-1.5, -0.25, 0.0]), np.float32([2.0, 0.75, 10.0])
    faces = []
    for a in range(3):
        for v in (mn[a], mx[a]):
            p = (mn + mx) / 2
            p[a] = v
            faces.append(p)
    just_out = []
    for a in range(3):
        lo, hi = ((mn + mx) / 2).copy(), ((mn + mx) / 2).copy()
        lo[a] = np.nextafter(mn[a], np.float32(-np.inf))
        hi[a] = np.nextafter(mx[a], np.float32(np.inf))
        just_out += [lo, hi]
    pts = cloud_of(faces + just_out)
    got = box_ref.crop_box(pts, mn, mx)
    assert got == pts[:6].tobytes()
    assert box_ref.pcl(pts, mn, mx) == got == numpy_box(pts, mn, mx)


def test_both_signs_of_zero_on_a_zero_face():
    pts = cloud_of([[0.0, 0.0, 0.0], [-0.0, -0.0, -0.0], [0.0, -0.0, 0.5], [-1e-45, 0.0, 0.0]])
    for mn, mx in (([0, 0, 0], [1, 1, 1]), ([-0.0, -0.0, -0.0], [1, 1, 1]), ([-1, -1, -1], [-0.0, 0.0, 0.0])):
        got = box_ref.crop_box(pts, mn, mx)
        want = pts[:3].tobytes() if mx[0] == 1 else pts[[0, 1, 3]].tobytes()
        assert got == want and box_ref.pcl(pts, mn, mx) == got, (mn, mx)


def test_infinite_bounds_make_a_half_open_box():
    rng = np.random.default_rng(3)
    pts = cloud_of(rng.normal(0, 1e30, (1000, 3)))
    inf = np.inf
    assert box_ref.crop_box(pts, [-inf] * 3, [inf] * 3) == pts.tobytes()
    got = box_ref.crop_box(pts, [-inf, -inf, 0.0], [inf, inf, inf])
    assert got == pts[pts[:, 2] >= 0].tobytes() and 0 < len(got) < pts.nbytes
    assert box_ref.pcl(pts, [-inf, -inf, 0.0], [inf, inf, inf]) == got


def test_non_finite_points_are_dropped():
    pts = cloud_of([[0, 0, 0], [np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.5, 0.5, 0.5]])
    inf = np.inf
    for mn, mx in (([-1] * 3, [1] * 3), ([-inf] * 3, [inf] * 3)):
        assert box_ref.crop_box(pts, mn, mx) == pts[[0, 4]].tobytes()
        assert box_ref.pcl(pts, mn, mx) == pts[[0, 4]].tobytes()


def test_identity_is_the_same_as_no_transform():
    rng = np.random.default_rng(4)
    pts = cloud_of(rng.normal(0, 1, (5000, 3)))
    pts[::7, 1] = -0.0
    a = box_ref.crop_box(pts, [-0.5, -1, 0], [1, 0.0, 2])
    assert a == box_ref.crop_box(pts, [-0.5, -1, 0], [1, 0.0, 2], np.eye(3, 4)) == numpy_box(pts, [-0.5, -1, 0],
                                                                                               [1, 0.0, 2])
    assert 0 < len(a) < pts.nbytes


def test_a_quarter_turn_permutes_the_axes_exactly():
    rng = np.random.default_rng(5)
    pts = cloud_of(rng.uniform(-3, 3, (4000, 3)))
    # l = (y, -x, z) + (0.5, 0, 0): x_l in [0, 1] <=> y in [-0.5, 0.5]; y_l in [-2, 0] <=> x in [0, 2]
    t = np.float32([[0, 1, 0, 0.5], [-1, 0, 0, 0], [0, 0, 1, 0]])
    got = box_ref.crop_box(pts, [0, -2, -1], [1, 0, 1], t)
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    keep = (y + np.float32(0.5) >= 0) & (y + np.float32(0.5) <= 1) & (x >= 0) & (x <= 2) & (np.abs(z) <= 1)
    assert got == pts[keep].tobytes() and keep.sum() > 50
    assert box_ref.pcl(pts, [0, -2, -1], [1, 0, 1], t) == got


def test_input_order_is_kept_and_points_are_unchanged():
    rng = np.random.default_rng(6)
    pts = cloud_of(rng.uniform(-1, 1, (3000, 3)))
    t = np.concatenate([rotation(rng), [[5.0], [-3.0], [0.25]]], axis=1).astype(np.float32)
    got = np.frombuffer(box_ref.crop_box(pts, [4, -4, -0.5], [6, -2, 1], t), np.float32).reshape(-1, 4)
    idx = got[:, 3].astype(np.int64)
    assert len(idx) > 100 and np.all(np.diff(idx) > 0)
    assert got.tobytes() == pts[idx].tobytes()


def test_an_empty_result():
    pts = cloud_of(np.random.default_rng(7).uniform(-1, 1, (100, 3)))
    assert box_ref.crop_box(pts, [2, 2, 2], [3, 3, 3]) == b""
    assert box_ref.crop_box(cloud_of(np.empty((0, 3))), [-1] * 3, [1] * 3) == b""
    assert box_ref.pcl(pts, [2, 2, 2], [3, 3, 3]) == b""


@pytest.mark.parametrize("eps", [1e-6, 5e-6])
def test_pcl_skips_a_near_identity_transform_that_the_recipe_applies(eps):
    """The one documented difference on finite transforms: PCL's fuzzy isIdentity() skips a transform within 1e-5 of
    the identity, the recipe applies it; a point on a face sees the difference."""
    t = np.eye(3, 4, dtype=np.float32)
    t[0, 3] = eps
    pts = cloud_of([[1.0, 0.0, 0.0], [0.5, 0.0, 0.0]])
    assert box_ref.pcl(pts, [-1] * 3, [1] * 3, t) == pts.tobytes()
    assert box_ref.crop_box(pts, [-1] * 3, [1] * 3, t) == pts[1:].tobytes() == numpy_box(pts, [-1] * 3, [1] * 3, t)
