"""CPU: the occupancy map recipe of include/d2pc_b200.h (tests/map_ref/occupancy.c, on the library's csrc/map_math.h)
against the literal restatement of octomap's computeRayKeys / insertScan / updateNode (tests/map_ref/
octomap_literal.cpp): identical cells on 10^6 seeded rays and on the edges, known answers of the map, the log-odds
conversion and the export's Morton order."""
import math

import numpy as np
import pytest

import map_ref as M

RES = 0.05


def same_rays(origins, points, res=RES, max_range=-1.0):
    a = M.rays_digest(origins, points, res, max_range)
    b = M.literal_rays_digest(origins, points, res, max_range)
    bad = np.nonzero((a != b).any(axis=1))[0]
    assert bad.size == 0, (res, max_range, bad[:5], a[bad[:5]], b[bad[:5]])
    return a


@pytest.mark.parametrize("res,max_range,n,seed", [(0.05, -1.0, 400_000, 1), (0.1, 10.0, 300_000, 2),
                                                  (0.05, 3.0, 200_000, 3), (0.37, -1.0, 100_000, 4)])
def test_recipe_and_literal_give_identical_rays_on_seeded_rays(res, max_range, n, seed):
    # S2-like rays: an origin near the vehicle, points 3-32 m away in every direction (10^6 rays over the four cases)
    rng = np.random.default_rng(seed)
    o = rng.uniform(-3, 3, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    p = (o + d * rng.uniform(3, 32, (n, 1))).astype(np.float32)
    a = same_rays(o, p, res, max_range)
    assert a[:, 0].mean() > 10


def test_edges():
    rng = np.random.default_rng(5)
    g = np.arange(-40, 41, dtype=np.float32) * np.float32(RES)  # voxel faces, zero and negative coordinates
    o, p = [], []
    for _ in range(20000):
        oo = rng.choice(g, 3)
        pp = rng.choice(g, 3)
        pp[rng.integers(0, 3, rng.integers(0, 3))] = oo[0]  # axis-aligned and planar rays
        o.append(oo), p.append(pp)
    # across key 32768 with tiny coordinates, origin and end in one voxel, corners
    o += [[0, 0, 0], [-1e-7, 0, 0], [0.01, 0.01, 0.01], [0.05, 0.05, 0.05], [-0.05, -0.05, -0.05], [1e-30, -1e-30, 0]]
    p += [[1, 0, 0], [1e-7, 1e-7, -1e-7], [0.02, 0.03, 0.04], [-0.05, 0.05, -0.05], [0.05, 0.05, 0.05], [-1, 1, -1]]
    # invalid keys: the origin or the point beyond 32768 voxels; non-finite points
    o += [[0, 0, 0], [2000, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0]]
    p += [[2000, 0, 0], [0, 0, 0], [np.inf, 0, 0], [np.nan, 1, 1], [1638.3, -1638.4, 1]]
    for mr in (-1.0, 0.0, 0.5, 10.0):
        same_rays(np.float32(o), np.float32(p), RES, mr)


def test_one_metre_along_x_at_a_tenth():
    keys, hit = M.ray((0, 0, 0), (1.0, 0, 0), 0.1)
    # nine free cells 0.0-0.9; 1.0 lies on the face of cells 9 and 10: floor puts it in 10, and the DDA stops at
    # tMax = 1.05 > 1.0 before cell 9 is added
    assert [tuple(k) for k in keys] == [(32768 + i, 32768, 32768) for i in range(9)]
    assert hit == (32778, 32768, 32768)
    t = M.Octree(resolution=0.1)
    t.insert(np.float32([[1.0, 0, 0, 1]]))
    k, lo = t.voxels()
    assert len(k) == 10 and lo[-1] == np.float32(M.logodds(0.7)) and (lo[:-1] == np.float32(M.logodds(0.4))).all()


def test_max_range_truncates_and_marks_no_hit():
    keys, hit = M.ray((0, 0, 0), (1.0, 0, 0), 0.1, max_range=0.5)
    # e = 0.5 lies on a face: its key is cell 5, and the DDA stops at tMax = 0.55 > 0.5 before cell 4
    assert hit is None and [k[0] for k in keys] == [32768 + i for i in range(4)]


def test_a_hit_beats_a_miss_in_one_frame():
    t = M.Octree(resolution=0.1)
    # the second point's ray crosses the first point's cell
    t.insert(np.float32([[0.55, 0.05, 0.05, 1], [1.05, 0.05, 0.05, 1]]))
    k, lo = t.voxels()
    d = {int(a): float(v) for a, v in zip(k[:, 0], lo)}
    assert d[32773] == np.float32(M.logodds(0.7)) and d[32772] == np.float32(M.logodds(0.4))


def test_clamp_sequence_and_the_early_abort():
    hit, cmax = np.float32(M.logodds(0.7)), np.float32(M.logodds(0.97))
    t = M.Octree(resolution=0.1)
    cloud = np.float32([[0.55, 0.05, 0.05, 1]])
    v = np.float32(0)
    for i in range(8):
        t.insert(cloud)
        v = min(np.float32(v + hit), cmax)
        assert t.voxels()[1][-1] == v, i
    assert v == cmax
    # lower clamp_max below the value: a hit now aborts early and leaves the value above the new bound
    t.set_params(clamp_max=0.9)
    t.insert(cloud)
    assert t.voxels()[1][-1] == cmax
    # raise it again: the value moves on from where it is
    t.set_params(clamp_max=0.999)
    t.insert(cloud)
    assert t.voxels()[1][-1] == min(np.float32(cmax + hit), np.float32(M.logodds(0.999)))


def test_the_threshold_is_inclusive():
    t = M.Octree(resolution=0.1, prob_hit=0.7, occupancy_thres=0.7)
    t.insert(np.float32([[0.55, 0.05, 0.05, 1]]))
    c = t.centers()
    assert len(c) == 1 and c[0].tolist() == [np.float32(0.55), np.float32(0.05), np.float32(0.05), 1.0]


def test_log_odds_conversion():
    for p in (0.12, 0.4, 0.5, 0.7, 0.97, 1e-6, 1 - 1e-6):
        assert M.logodds(p) == float(np.float32(math.log(p / (1 - p))))


def test_morton_order_is_the_leaf_iterators():
    rng = np.random.default_rng(7)
    ks = rng.integers(0, 65536, (3000, 3))
    py = [sum((((int(z) >> b) & 1) << (3 * b + 2)) | (((int(y) >> b) & 1) << (3 * b + 1)) | (((int(x) >> b) & 1) << (3 * b))
              for b in range(16)) for x, y, z in ks]
    assert [M.morton(*map(int, k)) for k in ks] == py
    # the literal's leaf order over a random cloud equals the Morton order of its keys
    t = M.Octree(resolution=0.2)
    pts = np.concatenate([rng.uniform(-20, 20, (2000, 3)), np.ones((2000, 1))], 1).astype(np.float32)
    t.insert(pts, (0.3, -0.2, 0.1))
    k, _ = t.voxels()
    m = [M.morton(*map(int, kk)) for kk in k]
    assert m == sorted(m) and len(set(m)) == len(m)


MAP_PARAMS = ["map_enable", "map_resolution", "map_sensor_model_hit", "map_sensor_model_miss", "map_sensor_model_min",
              "map_sensor_model_max", "map_occupancy_thres", "map_max_range", "map_max_bricks", "map_keep_cloud"]


def test_node_map_params():
    """The launch-file values of the node's map params reach it as numbers (tests/test_node_params.py checks that each
    lands in its settings field), both bindings advertise the centres, and no launch file of the package turns the map
    on."""
    import os
    import subprocess
    import tempfile

    from disparity_to_point_cloud_b200 import build
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    build.build()
    harness = build.build_harness()
    values = ["1", "0.1", "0.75", "0.35", "0.15", "0.95", "0.6", "9.5", "5000", "0"]
    with tempfile.TemporaryDirectory() as d:
        launch = os.path.join(d, "m.launch")
        with open(launch, "w") as f:
            f.write('<launch>\n  <node name="n" pkg="p" type="t">\n' +
                    "".join(f'    <param name="{k}" value="{v}"/>\n' for k, v in zip(MAP_PARAMS, values)) +
                    "  </node>\n</launch>\n")
        out = subprocess.run([harness, "params", launch] + MAP_PARAMS, check=True, capture_output=True,
                             text=True).stdout
    got = dict((ln.split(" ")[0], ln.split(" ")[2]) for ln in out.splitlines())
    assert all(float(got[k]) == float(v) for k, v in zip(MAP_PARAMS, values))
    for path in (os.path.join(root, "include", "d2pc_b200", "nodes.hpp"),
                 os.path.join(root, "ros1_shim", "disparity_to_point_cloud_node.cpp")):
        assert '"/octomap_point_cloud_centers"' in open(path).read(), path
    for name in os.listdir(os.path.join(root, "launch")):
        assert 'name="map_' not in open(os.path.join(root, "launch", name)).read()
