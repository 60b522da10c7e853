"""CPU: the radius outlier references (tests/outlier_ref) that the GPU stage is checked against.

The grid reference is pinned three ways: against the literal O(N^2) rule in the same C file, against an independent
numpy float32 restatement of the recipe in include/d2pc_b200.h, and against hand-built clouds with known answers.
PCL's two branches, restated literally, are compared with the rule: the k-NN branch (is_dense input) agrees
everywhere, the radiusSearch branch (strict < against the float radius squared) only differs on a pair exactly at
the boundary.  Also: the binding's RadiusOutlier has the header's layout."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import outlier_ref
from conftest import ROOT


def cloud_of(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    pts = np.zeros((len(xyz), 4), np.float32)
    pts[:, :3] = xyz
    pts[:, 3] = 1.0
    return pts


def np_ror(pts, radius, min_neighbors=1) -> bytes:
    """The recipe again, in numpy: float32 element-wise arithmetic (one rounding per operation), double compare."""
    pts = np.asarray(pts, np.float32).reshape(-1, 4)
    xyz = pts[:, :3]
    fin = np.isfinite(xyz).all(axis=1)
    f = xyz[fin]
    r2 = float(radius) * float(radius)
    keep = np.zeros(len(pts), bool)
    idx = np.nonzero(fin)[0]
    for a in range(0, len(f), 512):
        p = f[a: a + 512]
        dx, dy, dz = (p[:, None, k] - f[None, :, k] for k in range(3))
        with np.errstate(over="ignore"):  # an infinite distance is simply not <= r2
            s = (dx * dx + dy * dy) + dz * dz
        keep[idx[a: a + 512]] = (s.astype(np.float64) <= r2).sum(axis=1) >= min_neighbors + 1
    return pts[keep].tobytes()


def points(b) -> np.ndarray:
    return np.frombuffer(b, np.float32).reshape(-1, 4)


def pair_distance(pts, rng) -> float:
    """sqrt of the squared distance of a random finite pair (rule 3), so that the radius hits a boundary."""
    xyz = pts[:, :3][np.isfinite(pts[:, :3]).all(axis=1)]
    if len(xyz) < 2:
        return 0.5
    i, j = rng.choice(len(xyz), 2, replace=False)
    d = xyz[i] - xyz[j]
    s = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
    return float(np.sqrt(np.float64(s))) or 0.5


def draw_cloud(rng, n, kind):
    if kind == "random":
        pts = cloud_of(rng.uniform(-5, 5, (n, 3)))
    elif kind == "clustered":
        centres = rng.uniform(-20, 20, (max(1, n // 50), 3))
        pts = cloud_of(centres[rng.integers(0, len(centres), n)] + rng.normal(0, 0.05, (n, 3)))
    elif kind == "duplicated":
        base = rng.uniform(-2, 2, (max(1, n // 3), 3))
        pts = cloud_of(base[rng.integers(0, len(base), n)])
    else:  # a stereo-like cloud: a surface with salt, flying pixels and non-finite points
        u, v = rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)
        z = 2.0 + 0.5 * u + rng.normal(0, 0.002, n)
        pts = cloud_of(np.stack([u * z, v * z, z], 1))
        k = n // 20
        pts[rng.integers(0, n, k), :3] = rng.uniform(-50, 300, (k, 3))
    k = int(rng.integers(0, max(1, n // 8)))
    pts[rng.integers(0, max(n, 1), k), rng.integers(0, 3, k)] = rng.choice([np.nan, np.inf, -np.inf], k)
    return pts


@pytest.mark.parametrize("seed", range(40))
def test_grid_equals_brute_force_and_numpy(seed):
    rng = np.random.default_rng(9100 + seed)
    n = [0, 1, 2, 3][seed] if seed < 4 else int(rng.integers(4, 3000))
    pts = draw_cloud(rng, n, ["random", "clustered", "duplicated", "stereo"][seed % 4])
    radius = pair_distance(pts, rng) if rng.random() < 0.6 else float(rng.choice([0.01, 0.05, 0.2, 1.0, 5.0]))
    mn = int(rng.choice([0, 1, 2, 5, 50]))
    got = outlier_ref.radius_outlier(pts, radius, mn)
    assert got == outlier_ref.radius_outlier(pts, radius, mn, "brute"), seed
    assert got == np_ror(pts, radius, mn), seed


def test_grid_equals_numpy_at_20k_points():
    rng = np.random.default_rng(9200)
    pts = draw_cloud(rng, 20000, "stereo")
    for radius, mn in [(0.02, 2), (pair_distance(pts, rng), 5), (0.1, 10)]:
        got = outlier_ref.radius_outlier(pts, radius, mn)
        assert got == np_ror(pts, radius, mn), (radius, mn)
        assert 0 < len(got) < len(pts) * 16


def test_a_pair_exactly_r_apart_is_kept_and_one_ulp_further_is_not():
    out = outlier_ref.radius_outlier(cloud_of([[0, 0, 0], [0.5, 0, 0]]), 0.5, 1)
    assert len(out) == 32
    far = np.nextafter(np.float32(0.5), np.float32(1.0))
    assert outlier_ref.radius_outlier(cloud_of([[0, 0, 0], [far, 0, 0]]), 0.5, 1) == b""
    # in 3-D the sum is rounded too: (0.3, 0.4, 0) is 0.5 apart when its float32 sum says so
    p = cloud_of([[0, 0, 0], [0.3, 0.4, 0.0]])
    s = (np.float32(0.3) * np.float32(0.3) + np.float32(0.4) * np.float32(0.4)) + np.float32(0)
    r = float(np.sqrt(np.float64(s)))
    assert len(outlier_ref.radius_outlier(p, r, 1)) == (32 if float(r) * float(r) >= float(s) else 0)


def test_duplicates_count_and_min_zero_keeps_every_finite_point():
    pts = cloud_of([[1, 1, 1], [1, 1, 1], [1, 1, 1], [5, 5, 5], [np.nan, 0, 0], [0, np.inf, 0]])
    assert points(outlier_ref.radius_outlier(pts, 1e-6, 2))[:, 0].tolist() == [1, 1, 1]
    assert outlier_ref.radius_outlier(pts, 1e-6, 3) == b""
    assert points(outlier_ref.radius_outlier(pts, 1e-6, 0))[:, 0].tolist() == [1, 1, 1, 5]


def test_min_above_n_drops_everything():
    pts = cloud_of(np.zeros((10, 3)))
    assert len(outlier_ref.radius_outlier(pts, 1.0, 9)) == 160
    assert outlier_ref.radius_outlier(pts, 1.0, 10) == b""
    assert outlier_ref.radius_outlier(pts, 1.0, 2**32 - 1) == b""


def test_pairs_straddling_cell_edges_on_negative_coordinates():
    # pairs whose two points lie in neighbouring cells of any grid with cells near r, below zero on every axis
    r = 0.25
    base = np.array([-3.0, -7.0, -1.0], np.float32)
    xyz = []
    for k, axis in enumerate(np.eye(3, dtype=np.float32)):
        a = base - np.float32(10 * k)
        xyz += [a, a - axis * np.float32(r)]
    xyz.append(base + np.float32(5))  # isolated
    pts = cloud_of(xyz)
    got = outlier_ref.radius_outlier(pts, r, 1)
    assert got == outlier_ref.radius_outlier(pts, r, 1, "brute") == np_ror(pts, r, 1)
    assert len(got) == 6 * 16


def test_a_1e30_span_forces_coarsening():
    pts = cloud_of([[0, 0, 0], [0.09, 0, 0], [0.5, 0, 0], [1e30, 0, 0], [1e30, 0, 0], [-1e30, 1e30, -1e30]])
    got = outlier_ref.radius_outlier(pts, 0.1, 1)
    assert points(got)[:, 0].tolist() == [0.0, np.float32(0.09), np.float32(1e30), np.float32(1e30)]
    assert got == outlier_ref.radius_outlier(pts, 0.1, 1, "brute") == np_ror(pts, 0.1, 1)


def test_tiny_and_huge_radii():
    pts = cloud_of([[0, 0, 0], [1e-30, 0, 0], [3e38, 0, 0], [-3e38, 0, 0]])
    for r in (1e-40, 1e-20, 1e20, 1e200):
        for mn in (1, 2, 3):
            assert outlier_ref.radius_outlier(pts, r, mn) == outlier_ref.radius_outlier(pts, r, mn, "brute"), (r, mn)


@pytest.mark.parametrize("seed", range(12))
def test_pcl_knn_branch_equals_the_rule_on_dense_clouds(seed):
    rng = np.random.default_rng(9300 + seed)
    pts = draw_cloud(rng, int(rng.integers(2, 1500)), ["random", "clustered", "duplicated", "stereo"][seed % 4])
    pts = pts[np.isfinite(pts[:, :3]).all(axis=1)]  # an is_dense cloud
    for _ in range(3):
        radius = pair_distance(pts, rng)
        mn = int(rng.choice([0, 1, 2, 5, 50]))
        assert outlier_ref.pcl_knn(pts, radius, mn) == outlier_ref.radius_outlier(pts, radius, mn), (seed, mn)


def test_pcl_radius_branch_differs_only_on_the_boundary():
    rng = np.random.default_rng(9400)
    same = 0
    for case in range(12):
        pts = draw_cloud(rng, int(rng.integers(50, 1500)), ["random", "clustered", "stereo"][case % 3])
        radius = float(rng.choice([0.03, 0.1, 0.3]))  # no pair sits exactly on these
        mn = int(rng.choice([0, 1, 2, 5]))
        ours = outlier_ref.radius_outlier(pts, radius, mn)
        if outlier_ref.pcl_radius(pts, radius, mn) == ours:
            same += 1
    assert same == 12
    # a pair exactly r apart: the rule keeps both points, PCL's radiusSearch (dist < r^2) finds only the point itself
    pair = cloud_of([[0, 0, 0], [0.5, 0, 0], [np.nan, 0, 0]])
    assert len(outlier_ref.radius_outlier(pair, 0.5, 1)) == 32
    assert outlier_ref.pcl_radius(pair, 0.5, 1) == b""
    assert outlier_ref.pcl_knn(pair[:2], 0.5, 1) == pair[:2].tobytes()


def test_binding_radius_outlier_matches_the_header_layout(tmp_path):
    import disparity_to_point_cloud_b200 as d2pc
    hdr = open(os.path.join(ROOT, "include", "d2pc_b200.h")).read()
    body = re.search(r"typedef struct d2pc_radius_outlier \{(.*?)\} d2pc_radius_outlier;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"([a-z_]+)(?=[,;])", body)
    assert names == [f[0] for f in d2pc.RadiusOutlier._fields_]
    src = tmp_path / "layout.c"
    fields = ", ".join(f'(unsigned)offsetof(d2pc_radius_outlier, {n})' for n in names)
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "d2pc_b200.h"\n'
                   f'int main(void) {{ unsigned o[] = {{{fields}}}; printf("%u", (unsigned)sizeof(d2pc_radius_outlier));'
                   ' for (unsigned i = 0; i < sizeof o / sizeof o[0]; ++i) printf(" %u", o[i]); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(d2pc.RadiusOutlier)] + [getattr(d2pc.RadiusOutlier, n).offset for n in names]
    assert got == want
