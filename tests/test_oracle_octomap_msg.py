"""CPU: the octomap_msgs/Octomap recipe of include/d2pc_b200.h.  The pointer OcTree of tests/map_ref/octree_pointer.cpp
(octomap's updateNode with pruning, restated literally) against the flat map of octomap_literal.cpp -- the recipe's
claim that the pruned tree is a function of the known full-depth voxels alone -- and its writeData / writeBinaryData
bytes against the C recipe of tests/map_ref/octomap_msg.c fed the flat voxels; known answers; the Octomap message on
the ROS1 wire."""
import struct
import subprocess

import numpy as np
import pytest

import map_ref as M
from map_ref import octree as O

RES = 0.1
C0 = 32768


def wall(rng, x=2.0, half=0.8, step=0.03):
    """a dense wall of points at distance x in front of the sensor, with a little depth noise"""
    g = np.arange(-half, half, step, dtype=np.float32)
    yy, zz = np.meshgrid(g, g)
    n = yy.size
    pts = np.stack([x + rng.uniform(-0.05, 0.05, n), yy.ravel(), zz.ravel(), np.ones(n)], 1)
    return pts.astype(np.float32)


def sequence(seed, frames=8):
    """repeated frames of one wall from nearby origins: free space clamps, so octants become uniform and prune"""
    rng = np.random.default_rng(seed)
    out = []
    for f in range(frames):
        o = rng.uniform(-0.15, 0.15, 3).astype(np.float32)
        out.append((wall(rng, x=2.0 + 0.3 * (seed % 3)), o))
    return out


def both(**params):
    return M.Octree(resolution=RES, **params), O.PointerTree(resolution=RES, **params)


def same_voxels(ptr, flat, what):
    depths = [0] * 17
    pk, plo = ptr.voxels(depths)
    fk, flo = flat.voxels()
    assert pk.tobytes() == fk.tobytes(), (what, len(pk), len(fk))
    assert plo.view(np.uint32).tobytes() == flo.view(np.uint32).tobytes(), what
    return fk, flo, depths


def same_bytes(ptr, keys, lo, thres, what):
    for binary in (False, True):
        want = O.octomap_data(keys, lo, binary, thres)
        got = ptr.data(binary)
        assert got == want, (what, binary, len(got), len(want))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_pointer_tree_is_a_function_of_the_flat_voxels(seed):
    flat, ptr = both(max_range=6.0)
    pruned = False
    for i, (cloud, o) in enumerate(sequence(seed)):
        flat.insert(cloud, o)
        ptr.insert(cloud, o)
        k, lo, depths = same_voxels(ptr, flat, (seed, i))
        same_bytes(ptr, k, lo, 0.5, (seed, i))
        pruned = pruned or sum(depths[:16]) > 0
    assert sum(depths[:16]) > 0 and pruned, depths  # leaves above depth 16: the sequence really prunes
    assert len(k) > 2000


def test_clamp_and_threshold_changes_between_frames():
    flat, ptr = both()
    seq = sequence(5, frames=10)
    for i, (cloud, o) in enumerate(seq):
        p = dict(clamp_min=0.12 + 0.02 * (i % 3), clamp_max=0.97 - 0.03 * (i % 2), occupancy_thres=0.4 + 0.05 * i)
        flat.set_params(**p)
        ptr.set_params(**p)
        flat.insert(cloud, o)
        ptr.insert(cloud, o)
        k, lo, _ = same_voxels(ptr, flat, i)
        same_bytes(ptr, k, lo, p["occupancy_thres"], i)


def test_full_stream_reads_back_to_the_flat_voxels():
    flat, ptr = both()
    for cloud, o in sequence(6):
        flat.insert(cloud, o)
        ptr.insert(cloud, o)
    k, lo = flat.voxels()
    data = O.octomap_data(k, lo)
    rk, rlo = O.read_full(data)
    assert rk.tobytes() == k.tobytes() and rlo.view(np.uint32).tobytes() == lo.view(np.uint32).tobytes()


def records(data):
    """the full stream as (value, mask) records"""
    assert len(data) % 5 == 0
    return [(struct.unpack_from("<f", data, 5 * i)[0], data[5 * i + 4]) for i in range(len(data) // 5)]


def test_one_voxel():
    t = O.PointerTree(resolution=RES)
    t.update((C0, C0, C0), True)
    full, binary = t.data(), t.data(True)
    assert len(full) == 85 and len(binary) == 32 and t.tree_size() == 17
    hit = np.float32(M.logodds(0.7))
    recs = records(full)
    # key (32768, ...) has bit 15 set on every axis: child 7 below the root, child 0 below every other node
    assert [m for _, m in recs] == [0x80] + [0x01] * 15 + [0]
    assert all(np.float32(v) == hit for v, _ in recs)
    assert binary == bytes([0, 0xC0]) + bytes([3, 0]) * 14 + bytes([2, 0])
    k = np.uint16([[C0, C0, C0]])
    assert O.octomap_data(k, np.float32([hit])) == full and O.octomap_data(k, np.float32([hit]), True) == binary


def octant(base, level_span):
    """the keys of the aligned cube of level_span^3 voxels at base, in Morton order"""
    ks = [(base[0] + x, base[1] + y, base[2] + z) for z in range(level_span) for y in range(level_span)
          for x in range(level_span)]
    return sorted(ks, key=lambda k: M.morton(*k))


def test_equal_siblings_collapse():
    for span, depth in ((2, 15), (4, 14)):
        t = O.PointerTree(resolution=RES)
        for k in octant((C0, C0, C0), span):
            t.update(k, False)
        depths = [0] * 17
        k, lo = t.voxels(depths)
        assert len(k) == span ** 3 and depths[depth] == 1 and sum(depths) == 1, depths
        recs = records(t.data())
        assert len(recs) == depth + 1 and recs[-1][1] == 0  # the path to one leaf at `depth`
        assert t.data() == O.octomap_data(k, lo) and t.data(True) == O.octomap_data(k, lo, True)


def test_one_differing_sibling_blocks_the_collapse():
    t = O.PointerTree(resolution=RES)
    ks = octant((C0, C0, C0), 2)
    for k in ks:
        t.update(k, False)
    t.update(ks[5], False)  # one more miss: different log-odds
    depths = [0] * 17
    k, lo = t.voxels(depths)
    assert depths[16] == 8 and sum(depths) == 8
    assert t.data() == O.octomap_data(k, lo) and t.data(True) == O.octomap_data(k, lo, True)
    recs = records(t.data())
    assert recs[15] == (np.float32(lo).max(), 0xFF)  # the level-15 node: all eight children, the max of them


def test_a_hit_inside_a_collapsed_free_octant_expands_it():
    t = O.PointerTree(resolution=RES)
    ks = octant((C0, C0, C0), 4)
    for k in ks:
        t.update(k, False)
    before = [0] * 17
    t.voxels(before)
    assert before[14] == 1
    t.update(ks[9], True)
    depths = [0] * 17
    k, lo = t.voxels(depths)
    assert depths[14] == 0 and depths[15] == 7 and depths[16] == 8, depths
    miss, hit = np.float32(M.logodds(0.4)), np.float32(M.logodds(0.7))
    assert lo[9] == np.float32(miss + hit) and (np.delete(lo, 9) == miss).all()
    assert t.data() == O.octomap_data(k, lo) and t.data(True) == O.octomap_data(k, lo, True)


def test_inner_values_are_the_max_of_their_children():
    flat, ptr = both()
    for cloud, o in sequence(7, frames=3):
        flat.insert(cloud, o)
        ptr.insert(cloud, o)
    recs = records(ptr.data())
    k, lo = flat.voxels()
    assert np.float32(recs[0][0]) == lo.max()  # the root
    # every inner record's value is the max of its children's, read back from the stream
    pos = 0

    def walk():
        nonlocal pos
        v, mask = recs[pos]
        pos += 1
        if mask == 0:
            return v
        kids = [walk() for i in range(8) if (mask >> i) & 1]
        assert v == max(kids)
        return v
    walk()
    assert pos == len(recs)


def test_the_occupancy_threshold_moves_binary_bytes_only():
    flat, ptr = both()
    for cloud, o in sequence(8, frames=4):
        flat.insert(cloud, o)
        ptr.insert(cloud, o)
    k, lo = flat.voxels()
    full, binary = ptr.data(), ptr.data(True)
    ptr.set_params(occupancy_thres=0.9)
    assert ptr.data() == full and ptr.data(True) != binary
    assert ptr.data(True) == O.octomap_data(k, lo, True, 0.9) and len(ptr.data(True)) == len(binary)


def test_an_empty_map_writes_nothing():
    t = O.PointerTree(resolution=RES)
    assert t.data() == b"" and t.data(True) == b""
    k = np.zeros((0, 3), np.uint16)
    assert O.octomap_data(k, np.zeros(0, np.float32)) == b"" and O.octomap_data(k, np.zeros(0, np.float32), True) == b""


def test_octomap_message_on_the_ros1_wire(tmp_path):
    """ros_lite's octomap_msgs/Octomap: header, bool binary, string id, float64 resolution, int8[] data, and back."""
    from disparity_to_point_cloud_b200 import build
    build.build()
    harness = build.build_harness()
    out = tmp_path / "octomap.bin"
    subprocess.run([harness, "wire-octomap", str(out)], check=True)
    b = out.read_bytes()
    frame = b"/map"
    want = struct.pack("<IIII", 7, 11, 13, len(frame)) + frame
    want += struct.pack("<B", 1) + struct.pack("<I", 6) + b"OcTree" + struct.pack("<d", 0.05)
    want += struct.pack("<I", 5) + bytes([0, 0x80, 0x3F, 0xFF, 0x01])
    assert b == want
