"""CPU: the projected 2-D map recipe of include/d2pc_b200.h.  The per-voxel recipe in C (tests/map_ref/projected_map.c,
fed the flat voxels of octomap_literal.cpp) against octomap_server's projection restated literally over octomap's
pointer tree (tests/map_ref/projected_map.cpp), byte for byte in cells, width, height, resolution and origin bits:
sequences that really prune, known answers, z limits, padding, float rounding at the min face, the key range; the
OccupancyGrid message on the ROS1 wire."""
import struct
import subprocess

import numpy as np
import pytest

import map_ref as M
from map_ref import projected as P
from test_oracle_octomap_msg import octant, sequence

RES = 0.1
C0 = 32768


def same_grid(a, b, what):
    assert not isinstance(a, str) and not isinstance(b, str) and a is not None and b is not None, (what, a, b)
    (ca, ra, oa), (cb, rb, ob) = a, b
    assert ca.shape == cb.shape, (what, ca.shape, cb.shape)
    assert ca.tobytes() == cb.tobytes(), (what, int((ca != cb).sum()))
    assert np.float32(ra).tobytes() == np.float32(rb).tobytes(), what
    assert np.float64(oa).tobytes() == np.float64(ob).tobytes(), (what, oa, ob)


def both(tree, thres=0.5, **kw):
    """the pointer tree's projection and the recipe's on the tree's voxels; they must agree, the tree's is returned"""
    k, lo = tree.voxels()
    want = tree.projected_map(**kw)
    got = P.projected_map(k, lo, tree.resolution, thres, **kw)
    if want is None or isinstance(want, str):
        assert got == want
    else:
        same_grid(want, got, kw)
    return want


LIMITS = [dict(), dict(occupancy_min_z=-0.3, occupancy_max_z=0.25), dict(occupancy_min_z=0.05),
          dict(occupancy_max_z=-0.1), dict(occupancy_min_z=-np.inf, occupancy_max_z=np.inf),
          dict(min_x_size=1.0, min_y_size=0.3), dict(min_x_size=20.0, min_y_size=12.5),
          dict(occupancy_min_z=0.0, occupancy_max_z=0.4, min_x_size=6.0)]


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_recipe_equals_the_pointer_tree_on_pruning_sequences(seed):
    flat, tree = M.Octree(resolution=RES, max_range=6.0), P.ProjTree(resolution=RES, max_range=6.0)
    for i, (cloud, o) in enumerate(sequence(seed)):
        flat.insert(cloud, o)
        tree.insert(cloud, o)
        for kw in LIMITS if i in (0, 7) else LIMITS[:2]:
            g = both(tree, **kw)
            assert g is not None and not isinstance(g, str)
    depths = [0] * 17
    tree.voxels(depths)
    assert sum(depths[:16]) > 0, depths  # coarse leaves: the projection really sees pruned nodes
    cells = both(tree)[0]
    assert (cells == 100).any() and (cells == 0).any() and (cells == -1).any()
    # the tree the recipe is fed is the flat map's
    k, lo = flat.voxels()
    tk, tlo = tree.voxels()
    assert k.tobytes() == tk.tobytes() and lo.tobytes() == tlo.tobytes()


def test_changing_thresholds_between_frames():
    tree = P.ProjTree(resolution=RES)
    for i, (cloud, o) in enumerate(sequence(5, frames=6)):
        p = dict(clamp_min=0.12 + 0.02 * (i % 3), clamp_max=0.97 - 0.03 * (i % 2), occupancy_thres=0.4 + 0.05 * i)
        tree.set_params(**p)
        tree.insert(cloud, o)
        both(tree, p["occupancy_thres"], occupancy_min_z=-0.2)


def test_set_values_builds_the_inserted_tree():
    tree = P.ProjTree(resolution=RES)
    for cloud, o in sequence(6):
        tree.insert(cloud, o)
    k, lo = tree.voxels()
    built = P.ProjTree(resolution=RES)
    built.set_values(k, lo)
    assert built.data() == tree.data() and built.tree_size() == tree.tree_size()
    same_grid(built.projected_map(), tree.projected_map(), "set_values")


def test_empty_map_publishes_nothing():
    tree = P.ProjTree(resolution=RES)
    assert tree.projected_map() is None
    assert P.projected_map(np.zeros((0, 3), np.uint16), np.zeros(0, np.float32), RES) is None


def test_one_voxel():
    tree = P.ProjTree(resolution=RES)
    tree.update((C0, C0, C0), True)
    cells, res, origin = both(tree)
    # lo = 0 gives key 32768; hi = 0.1 as a float is just above 0.1, key 32769: a 2 x 2 grid
    assert cells.tolist() == [[100, -1], [-1, -1]]
    assert res == np.float32(RES) and origin[0] == float(np.float32(0.05)) - 0.05 == origin[1]


def test_pruned_octant_covers_its_square_and_the_origin_column():
    tree = P.ProjTree(resolution=RES)
    base = (C0 + 20, C0 + 8, C0 - 4)  # x > 0 only: the grid still starts at key 32768
    for k in octant(base, 4):
        tree.update(k, False)
    depths = [0] * 17
    tree.voxels(depths)
    assert depths[14] == 1 and sum(depths) == 1
    cells, _, origin = both(tree)
    assert origin[0] == float(np.float32(0.05)) - 0.05  # paddedMin.x is the world origin's key
    assert cells.shape == (8 + 4 + 1, 20 + 4 + 1)  # up to the max face's key, one past the octant
    want = np.full(cells.shape, -1, np.int8)
    want[8:12, 20:24] = 0
    assert cells.tobytes() == want.tobytes()
    tree.update((base[0] + 1, base[1] + 2, base[2] + 3), True)  # one hit expands the leaf and marks its column
    cells = both(tree)[0]
    want[8 + 2, 20 + 1] = 100
    assert cells.tobytes() == want.tobytes()


def test_coarse_leaf_passes_the_height_test_by_its_extent():
    tree = P.ProjTree(resolution=RES)
    for k in octant((C0, C0, C0), 4):  # one depth-14 leaf: z in [0, 0.4], centre 0.2
        tree.update(k, True)
    cells = both(tree, occupancy_min_z=0.3, occupancy_max_z=0.35)[0]  # the centre is outside, the extent overlaps
    assert (cells[:4, :4] == 100).all()
    cells = both(tree, occupancy_min_z=0.41)[0]
    assert (cells == -1).all()
    cells = both(tree, occupancy_max_z=0.0)[0]  # strict: c - h < max_z fails at 0
    assert (cells == -1).all()


def test_padding_smaller_and_larger_than_the_map():
    tree = P.ProjTree(resolution=RES)
    for cloud, o in sequence(9, frames=3):
        tree.insert(cloud, o)
    plain = both(tree)
    small = both(tree, min_x_size=0.2, min_y_size=0.2)
    same_grid(plain, small, "smaller padding changes nothing")
    large = both(tree, min_x_size=30.0, min_y_size=10.0)
    assert large[0].shape[1] >= 300 and large[0].shape[0] >= 100
    assert large[2][0] < plain[2][0] and large[2][1] < plain[2][1]
    assert (large[0] == 100).sum() == (plain[0] == 100).sum() and (large[0] == 0).sum() == (plain[0] == 0).sum()


def test_min_face_on_a_float_rounding_boundary():
    # at 0.1 m the min face of key 29771 is stored as a float just below its boundary: its key is 29770
    tree = P.ProjTree(resolution=RES)
    tree.update((29771, C0 + 2, C0), True)
    cells, _, origin = both(tree)
    assert cells.shape[1] == C0 + 1 - 29770 and cells[2, 1] == 100 and cells[2, 0] == -1
    tree = P.ProjTree(resolution=RES)
    tree.update((29773, C0 + 2, C0), True)
    cells = both(tree)[0]
    assert cells.shape[1] == C0 + 1 - 29773 and cells[2, 0] == 100


@pytest.mark.parametrize("key", [(65535, C0, C0), (C0, 65535, C0), (C0, C0, 65535), (0, C0, C0), (C0, C0, 0)])
def test_key_range_edge_has_no_padded_key(key):
    tree = P.ProjTree(resolution=RES)
    tree.update(key, False)
    assert both(tree) == "BAD_DIMS"
    # at 0.02 m the same faces still have keys
    tree = P.ProjTree(resolution=0.02)
    tree.update(key, False)
    g = both(tree)
    assert g is not None and not isinstance(g, str)


def test_occupancy_grid_on_the_ros1_wire(tmp_path):
    """ros_lite's nav_msgs/OccupancyGrid: header, MapMetaData (time, float32 resolution, uint32 width and height,
    geometry_msgs/Pose of 7 float64), int8[] data, and back."""
    from disparity_to_point_cloud_b200 import build
    build.build()
    harness = build.build_harness()
    out = tmp_path / "grid.bin"
    subprocess.run([harness, "wire-grid", str(out)], check=True)
    frame = b"/map"
    want = struct.pack("<IIII", 7, 11, 13, len(frame)) + frame
    want += struct.pack("<IIfII", 17, 19, 0.05, 3, 2) + struct.pack("<7d", -1.25, 2.5, 0.125, 0, 0, 0, 1.0)
    want += struct.pack("<I", 6) + bytes([0xFF, 0, 100, 100, 0, 0xFF])
    assert out.read_bytes() == want
