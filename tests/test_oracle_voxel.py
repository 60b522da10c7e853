"""CPU: the voxel-grid reference (tests/voxel_ref) that the GPU's D2PC_FILTER_VOXEL is checked against.

It is pinned three ways: against an independent numpy restatement of the recipe in include/d2pc_b200.h (np.lexsort
plus a sequential float32 fold), against hand-built clouds with known answers, and against a literal restatement of
PCL's applyFilter that keeps PCL's own std::sort order -- same voxels, same order, centroids within the rounding
that the summation order can move.  Also: the binding's VoxelGrid has the header's layout."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import voxel_ref
from conftest import ROOT

INT32_MAX = 2147483647


def cloud_of(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    pts = np.zeros((len(xyz), 4), np.float32)
    pts[:, :3] = xyz
    return pts


def np_voxel(pts, leaf, min_points=0, limit=None):
    """The recipe again, in numpy: float32 element-wise arithmetic, np.lexsort for the stable order."""
    pts = np.asarray(pts, np.float32).reshape(-1, 4)
    leaf = np.broadcast_to(np.asarray(leaf, np.float32), (3,))
    inv = np.float32(1.0) / leaf
    xyz = pts[:, :3]
    inc = np.isfinite(xyz).all(axis=1)
    if limit is not None:
        field, lo, hi = limit
        v = xyz[:, "xyz".index(field)].astype(np.float64)
        with np.errstate(invalid="ignore"):
            inc &= (v >= lo) & (v <= hi)
    if not inc.any():
        return b"", 1
    mn, mx = xyz[inc].min(axis=0), xyz[inc].max(axis=0)
    with np.errstate(over="ignore", invalid="ignore"):
        d = np.trunc(((mx - mn) * inv).astype(np.float64)) + 1.0
        fallback = not (d[0] * d[1] * d[2] <= INT32_MAX)
        lo_b, hi_b = np.floor(mn * inv), np.floor(mx * inv)
    if not fallback and not ((lo_b >= -2.0 ** 31).all() and (hi_b < 2.0 ** 31).all()):
        fallback = True
    if not fallback:
        div = hi_b.astype(np.float64) - lo_b.astype(np.float64) + 1.0
        span = (hi_b - lo_b).astype(np.float64)
        fallback = not (span[0] + span[1] * div[0] + span[2] * div[0] * div[1] < INT32_MAX)
    if fallback:
        return pts.tobytes(), 0
    min_b = lo_b.astype(np.int64)
    mul = np.array([1, int(div[0]), int(div[0]) * int(div[1])], np.int64)
    sel = np.nonzero(inc)[0]
    ijk = (np.floor(xyz[sel] * inv) - min_b.astype(np.float32)).astype(np.int64)
    idx = ijk @ mul
    order = np.lexsort((sel, idx))
    idx, sel = idx[order], sel[order]
    out = []
    a = 0
    while a < len(sel):
        b = a
        while b < len(sel) and idx[b] == idx[a]:
            b += 1
        if b - a >= min_points:
            s = np.zeros(3, np.float32)
            for m in range(a, b):
                s = s + xyz[sel[m]]  # float32 + float32: one rounding per add, left to right
            out.append(np.append(s / np.float32(b - a), np.float32(1.0)).astype(np.float32))
        a = b
    return (np.array(out, np.float32).tobytes() if out else b""), 1


def points(b) -> np.ndarray:
    return np.frombuffer(b, np.float32).reshape(-1, 4)


def random_cloud(rng, n, scale):
    pts = cloud_of(rng.normal(0, scale, (n, 3)) + rng.uniform(-scale, scale, 3))
    k = rng.integers(0, max(1, n // 10))
    pts[rng.integers(0, n, k), rng.integers(0, 3, k)] = rng.choice([np.nan, np.inf, -np.inf], k)
    if rng.random() < 0.3:  # exact voxel boundaries
        pts[: n // 4, :3] = np.round(pts[: n // 4, :3] * 4) / 4
    return pts


@pytest.mark.parametrize("seed", range(40))
def test_reference_matches_numpy_restatement(seed):
    rng = np.random.default_rng(7000 + seed)
    n = int(rng.integers(1, 600))
    pts = random_cloud(rng, n, float(rng.choice([0.1, 1.0, 10.0, 1000.0])))
    leaf = float(rng.choice([0.01, 0.05, 0.2, 1.0, 10.0])) if rng.random() < 0.7 else tuple(rng.uniform(0.05, 2, 3))
    mp = int(rng.choice([0, 0, 1, 2, 5]))
    limit = None
    if rng.random() < 0.5:
        lo = float(rng.normal(0, 2))
        limit = (str(rng.choice(list("xyz"))), lo, lo + float(rng.uniform(0, 6)))
    got = voxel_ref.voxel_grid(pts, leaf, mp, limit)
    want = np_voxel(pts, leaf, mp, limit)
    assert got[1] == want[1] and got[0] == want[0], (seed, len(got[0]) // 16, len(want[0]) // 16)


def test_points_on_voxel_boundaries_open_the_upper_voxel():
    # 0.5 / 0.5 = 1 exactly: floor puts 0.5 into voxel 1, not 0; 1.0 into voxel 2
    pts = cloud_of([[0.0, 0, 0], [0.25, 0, 0], [0.5, 0, 0], [1.0, 0, 0]])
    out, dense = voxel_ref.voxel_grid(pts, 0.5)
    assert dense == 1
    np.testing.assert_array_equal(points(out), [[0.125, 0, 0, 1], [0.5, 0, 0, 1], [1.0, 0, 0, 1]])


def test_negative_coordinates_floor_not_truncate():
    # -0.1 and 0.1 must land in different voxels (floorf(-0.2) = -1); -0.6 one voxel further down
    pts = cloud_of([[-0.1, 0, 0], [0.1, 0, 0], [-0.6, 0, 0], [-0.9, 0, 0]])
    out, _ = voxel_ref.voxel_grid(pts, 0.5)
    np.testing.assert_array_equal(points(out)[:, 0], np.array([-0.75, -0.1, 0.1], np.float32))


def test_limit_endpoints_are_inclusive():
    z = [0.0, 1.0, 2.0, 3.0, 4.0]
    pts = cloud_of([[0, 0, v] for v in z])
    out, _ = voxel_ref.voxel_grid(pts, 10.0, limit=("z", 1.0, 3.0))
    np.testing.assert_array_equal(points(out), [[0, 0, 2.0, 1]])
    # a float just below the lower limit in double is out
    below = np.nextafter(np.float32(1.0), np.float32(0))
    out, _ = voxel_ref.voxel_grid(cloud_of([[0, 0, below], [0, 0, 2.0]]), 10.0, limit=("z", 1.0, 3.0))
    np.testing.assert_array_equal(points(out), [[0, 0, 2.0, 1]])


def test_non_finite_points_are_excluded():
    pts = cloud_of([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [1.0, 1.0, 1.0], [1.5, 1.5, 1.5]])
    out, dense = voxel_ref.voxel_grid(pts, 1.0)
    assert dense == 1
    np.testing.assert_array_equal(points(out), [[1.25, 1.25, 1.25, 1]])


def test_min_points_per_voxel_drops_small_voxels():
    pts = cloud_of([[0.1, 0, 0], [0.2, 0, 0], [0.3, 0, 0], [5.1, 0, 0], [5.2, 0, 0], [9.5, 0, 0]])
    for mp, want in [(0, 3), (1, 3), (2, 2), (3, 1), (4, 0)]:
        out, dense = voxel_ref.voxel_grid(pts, 1.0, mp)
        assert len(out) // 16 == want and dense == 1, mp
        assert out == np_voxel(pts, 1.0, mp)[0]


def test_overflow_guard_returns_the_input_unchanged():
    pts = cloud_of([[0, 0, 0], [100.0, 100.0, 100.0], [np.nan, 1, 2], [3, 4, 5]])
    # 100 / 0.01 + 1 = 10001 voxels per axis: 1e12 > INT32_MAX
    out, dense = voxel_ref.voxel_grid(pts, 0.01)
    assert dense == 0 and out == pts.tobytes()
    # just inside: 1290^3 < 2^31 - 1 < 1291^3
    ok, dense = voxel_ref.voxel_grid(cloud_of([[0, 0, 0], [1289.0, 1289.0, 1289.0]]), 1.0)
    assert dense == 1 and len(ok) == 32
    bad, dense = voxel_ref.voxel_grid(cloud_of([[0, 0, 0], [1290.0, 1290.0, 1290.0]]), 1.0)
    assert dense == 0 and len(bad) == 32


def test_empty_result():
    for pts, kw in [(cloud_of(np.empty((0, 3))), {}), (cloud_of([[np.nan, 0, 0]]), {}),
                    (cloud_of([[0, 0, 5.0]]), {"limit": ("z", 0.0, 1.0)})]:
        out, dense = voxel_ref.voxel_grid(pts, 0.1, **kw)
        assert out == b"" and dense == 1


def test_pcl_sort_order_differs_only_in_the_last_bits():
    """PCL's std::sort leaves a voxel's order unspecified: same voxels in the same order, centroids within
    count * 2^-23 * max|coord| of the stable-order ones (what the stable order costs, and all it costs)."""
    rng = np.random.default_rng(11)
    moved = 0
    for case in range(20):
        n = int(rng.integers(200, 5000))
        pts = random_cloud(rng, n, float(rng.choice([1.0, 10.0])))
        leaf = float(rng.choice([0.5, 2.0, 8.0]))
        mp = int(rng.choice([0, 2]))
        ours, d1 = voxel_ref.voxel_grid(pts, leaf, mp)
        pcl, d2 = voxel_ref.voxel_pcl_order(pts, leaf, mp)
        assert d1 == d2 == 1 and len(ours) == len(pcl) > 0, case
        a, b = points(ours), points(pcl)
        xyz = pts[:, :3][np.isfinite(pts[:, :3]).all(axis=1)]
        bound = len(xyz) * 2.0 ** -23 * float(np.abs(xyz).max())
        assert np.abs(a - b).max() <= bound, case
        moved += int((a != b).any())
    assert moved > 0  # the two orders really do round differently somewhere


def test_binding_voxel_grid_matches_the_header_layout(tmp_path):
    import disparity_to_point_cloud_b200 as d2pc
    hdr = open(os.path.join(ROOT, "include", "d2pc_b200.h")).read()
    body = re.search(r"typedef struct d2pc_voxel_grid \{(.*?)\} d2pc_voxel_grid;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"([a-z_]+)(?=[,;])", body)
    assert names == [f[0] for f in d2pc.VoxelGrid._fields_]
    src = tmp_path / "layout.c"
    fields = ", ".join(f'(unsigned)offsetof(d2pc_voxel_grid, {n})' for n in names)
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "d2pc_b200.h"\n'
                   f'int main(void) {{ unsigned o[] = {{{fields}}}; printf("%u", (unsigned)sizeof(d2pc_voxel_grid));'
                   ' for (unsigned i = 0; i < sizeof o / sizeof o[0]; ++i) printf(" %u", o[i]); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(d2pc.VoxelGrid)] + [getattr(d2pc.VoxelGrid, n).offset for n in names]
    assert got == want
